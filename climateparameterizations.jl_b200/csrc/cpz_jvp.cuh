// Pushforwards (forward-mode derivatives) of the right-hand side (cpz_rhs_jvp) and of the fixed-step solve (cpz_solve_jvp).
//
// One tangent stage at the stage input X with tangent Xd computes k = f(X) and
//   kd = (df/dX) Xd + (df/dtheta) theta_dot + (df/dp) p_dot,   p = (nu0, nu_m, dRi, Ric, Pr),
// the forward-mode restatement of one reverse stage of adjoint_body (cpz_adjoint.cuh): the primal forward keeps z of every
// layer, the tangent runs layer by layer (zd_l = W_l ad_{l-1} + Wdot_l a_{l-1} + bdot_l, ad_l = act'(z_l) zd_l), then the face
// fluxes (faces_jvp, the tangent of the statements faces_vjp transposes) and the cell differences (centres_jvp). The solve
// kernel runs the Runge–Kutta recursion on state and tangent with the same tableau,
//   Xd_i = xd + h sum_j a_ij kd_j,   xd <- xd + h sum_i b_i kd_i,
// and, with implicit diffusion, the tangent of the backward-Euler step before every sub-step (implicit_jvp_tile).
// FP32 SIMT on the adjoint plan's shared-memory layout (adjoint_smem_layout): xs = x, xbar = xd, xin = X_i (and the transpose
// staging of the bulk copies), xb = Xd_i, arena = a and the face-flux rows, zarena = z, overwritten in place by ad once
// act'(z) has been read. Boundary fluxes, diurnal forcing and t enter f additively, so their tangent is 0. Columns are
// independent: nothing is summed over the batch.
#pragma once
#include "cpz_adjoint.cuh"

namespace cpz {

struct JvpArgs {
  const float* theta;
  const float* theta_dot;  // [P] in destructure order, or null (= 0)
  const float* pdot;       // [5] tangent of (nu0, nu_m, dRi, Ric, Pr), or null (= 0)
  const float* x;          // [ncol][S]: x (rhs) or x0 (solve)
  const float* xdot;       // [ncol][S] or null (= 0)
  const float* bcs;        // [ncol][nbc]
  const float* Q;          // [ncol] diurnal amplitudes or null
  float* y;                // rhs: dxdt [ncol][S]; solve: traj [ncol][n_saved][S]; or null
  float* ydot;             // the tangent of y, same layout
  float* kslots;           // solve: [grid][2 n_stages][S][CT]: k_j at slot j, kd_j at slot n_stages + j
  float t;                 // rhs: evaluation time
  int ncol, n_tiles, n_saved;
};

// Richardson number at an interior face (the shear clamped as in faces_vjp) and, returned, its tangent
__device__ __forceinline__ float ri_tangent(const ModelD& M, float Gu, float Gv, float GT, float Gud, float Gvd, float GTd, float eps,
                                            float* Ri) {
  const float su = M.rc.sig_u * (Gu + eps), sv = M.rc.sig_v * (Gv + eps);
  const float iS2 = __fdividef(1.f, fmaxf(su * su + sv * sv, 1e-18f));
  *Ri = M.rc.BzC * (GT + eps) * iS2;
  return M.rc.BzC * GTd * iS2 - *Ri * iS2 * 2.f * (su * M.rc.sig_u * Gud + sv * M.rc.sig_v * Gvd);
}

// nu = nu0 + nu_m s(Ri) and, returned, its tangent from Rid and the mPP-parameter tangent pd (the factors faces_vjp
// accumulates into pg); *s receives s.
__device__ __forceinline__ float nu_tangent(const ModelD& M, float Ri, float Rid, const float* __restrict__ pd, float* nu, float* s_out) {
  const float y2 = 2.f * (Ri - M.rc.Ric) * M.rc.inv_dRi;
  const float s = __fdividef(1.f, 1.f + __expf(y2));
  const float ss = s * (1.f - s);
  *nu = M.rc.nu0 + M.rc.nu_m * s;
  *s_out = s;
  float nud = -2.f * M.rc.inv_dRi * M.rc.nu_m * ss * Rid;
  if (pd != nullptr) {
    nud += __ldg(pd) + s * __ldg(pd + 1);
    nud += M.rc.nu_m * ss * M.rc.inv_dRi * (y2 * __ldg(pd + 2) + 2.f * __ldg(pd + 3));
  }
  return nud;
}

// tangent of nu_T = nu / Pr (or kappa where the inference variant's convective adjustment applies, tangent 0)
__device__ __forceinline__ float nuT_tangent(const ModelD& M, float nu, float nud, float Gu, float GT, const float* __restrict__ pd,
                                             float* nuT) {
  if (M.variant == RHS_INFER && (M.flags & F_CA)) {
    const float test = (M.flags & F_CA_LITERAL_U) ? Gu : GT;
    if (!(test > 0.f)) { *nuT = M.rc.kappa; return 0.f; }
  }
  *nuT = nu * M.rc.inv_Pr;
  float d = nud * M.rc.inv_Pr;
  if (pd != nullptr) d -= nu * M.rc.inv_Pr * M.rc.inv_Pr * __ldg(pd + 4);
  return d;
}

// Tangent of face_diffusivity (the D_q of the implicit-diffusion step) at interior face k
__device__ __forceinline__ float face_diffusivity_dot(const ModelD& M, const float* __restrict__ X, const float* __restrict__ Xd, int q,
                                                      int k, int c, int CT_, const float* __restrict__ pd) {
  const int N = M.Nz;
  const float Nf = M.rc.Nf;
  if (M.variant == RHS_FC) {
    if (!(M.flags & F_MPP)) return 0.f;  // the convective-adjustment part is piecewise constant
    const float G = Nf * (X[k * CT_ + c] - X[(k - 1) * CT_ + c]);
    float dcnu;
    fc_mpp_cnu(M, G, &dcnu);
    return dcnu * Nf * (Xd[k * CT_ + c] - Xd[(k - 1) * CT_ + c]);
  }
  if (!((M.flags & F_MPP) || M.variant == RHS_INFER)) return 0.f;
  const float eps = M.variant == RHS_TRAIN ? M.rc.eps : 0.f;
  float G[3], Gd[3];
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    G[f] = Nf * (X[(f * N + k) * CT_ + c] - X[(f * N + k - 1) * CT_ + c]);
    Gd[f] = Nf * (Xd[(f * N + k) * CT_ + c] - Xd[(f * N + k - 1) * CT_ + c]);
  }
  float Ri, nu, s, nuT;
  const float Rid = ri_tangent(M, G[0], G[1], G[2], Gd[0], Gd[1], Gd[2], eps, &Ri);
  const float nud = nu_tangent(M, Ri, Rid, pd, &nu, &s);
  if (q < 2) return M.rc.c[q] * nud;
  return M.rc.c[2] * nuT_tangent(M, nu, nud, G[0], G[2], pd, &nuT);
}

// Tangent of layer l of every net that has it: zd = W ad_{l-1} + Wdot a_{l-1} + bdot (ad_{-1} = Xd, a_{-1} = X), then
// ad_l = act'(z_l) zd in place over z_l in zarena. Tiles of 4 outputs x 4 columns over the flattened tile space of the
// layer's gemms. One block barrier must follow.
template <bool WS, int CT, int NT>
__device__ __noinline__ void mlp_tangent_layer(const ModelD& M, int l, const float* __restrict__ X, const float* __restrict__ Xd,
                                               const float* __restrict__ arena, float* __restrict__ zarena,
                                               const float* __restrict__ wsm, const float* __restrict__ theta,
                                               const float* __restrict__ theta_dot) {
  constexpr int NCG = CT / 4;
  int gl[3] = {0, 0, 0}, end[4] = {0, 0, 0, 0}, ng = 0;
  for (int gi = 0; gi < M.n_gemm && ng < 3; ++gi) {
    if (M.gemm[gi].layer != l) continue;
    gl[ng] = gi;
    end[ng + 1] = end[ng] + ((M.gemm[gi].N + 3) / 4) * NCG;
    ++ng;
  }
  for (int q = ng + 1; q < 4; ++q) end[q] = end[ng];
  for (int t = threadIdx.x; t < end[ng]; t += NT) {
    const int q = (t >= end[1]) + (t >= end[2]);
    const GemmD& g = M.gemm[q == 0 ? gl[0] : (q == 1 ? gl[1] : gl[2])];
    const int tile = t - (q == 0 ? 0 : (q == 1 ? end[1] : end[2]));
    const int cg = tile % NCG, j0 = (tile / NCG) * 4;
    const int K = g.K, N = g.N;
    const float* a = (g.in_off < 0 ? X : arena + g.in_off * CT) + 4 * cg;
    const float* ad = (g.in_off < 0 ? Xd : zarena + g.in_off * CT) + 4 * cg;
    int jr[4];
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) jr[jj] = min(j0 + jj, N - 1);
    float acc[4][4];
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) acc[jj][cc] = 0.f;
    auto fma_row = [&](const float (&w)[4], const float4 v) {
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        acc[jj][0] = fmaf(w[jj], v.x, acc[jj][0]);
        acc[jj][1] = fmaf(w[jj], v.y, acc[jj][1]);
        acc[jj][2] = fmaf(w[jj], v.z, acc[jj][2]);
        acc[jj][3] = fmaf(w[jj], v.w, acc[jj][3]);
      }
    };
    if (WS) {
      // the plan pads every shared weight row to Npad (a multiple of 4, zero filled): rows past N read zeros
      const float* W = wsm + g.sw_off + j0;
#pragma unroll 4
      for (int k = 0; k < K; ++k) {
        const float4 wv = *reinterpret_cast<const float4*>(W + k * g.Npad);
        const float w[4] = {wv.x, wv.y, wv.z, wv.w};
        fma_row(w, *reinterpret_cast<const float4*>(ad + k * CT));
      }
    } else {
      const float* W = theta + g.w_off;
#pragma unroll 2
      for (int k = 0; k < K; ++k) {
        const float w[4] = {__ldg(W + k * N + jr[0]), __ldg(W + k * N + jr[1]), __ldg(W + k * N + jr[2]), __ldg(W + k * N + jr[3])};
        fma_row(w, *reinterpret_cast<const float4*>(ad + k * CT));
      }
    }
    if (theta_dot != nullptr) {
      const float* Wd = theta_dot + g.w_off;
#pragma unroll 2
      for (int k = 0; k < K; ++k) {
        const float w[4] = {__ldg(Wd + k * N + jr[0]), __ldg(Wd + k * N + jr[1]), __ldg(Wd + k * N + jr[2]), __ldg(Wd + k * N + jr[3])};
        fma_row(w, *reinterpret_cast<const float4*>(a + k * CT));
      }
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const float bd = __ldg(theta_dot + g.b_off + jr[jj]);
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) acc[jj][cc] += bd;
      }
    }
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      if (j0 + jj < N) {
        float4* p = reinterpret_cast<float4*>(zarena + (g.out_off + j0 + jj) * CT + 4 * cg);
        const float4 z = *p;
        *p = make_float4(acc[jj][0] * act_grad(g.act, z.x), acc[jj][1] * act_grad(g.act, z.y), acc[jj][2] * act_grad(g.act, z.z),
                         acc[jj][3] * act_grad(g.act, z.w));
      }
    }
  }
}

// ---- tangent of the face fluxes ------------------------------------------------------------------------------------
// Fd_q at every face into fd [nf][Nz+1][CT] (0 at the boundary faces: their fluxes are data), from the stage input X, its
// tangent Xd and the NN-output tangents in zarena (nn_off rows): Fd_q = nnd_q - c_q (nud G_q + nu Gd_q), with the
// convective-adjustment switch and both smoothing filters (linear) as in faces_phase.
template <int CT, int NT>
__device__ __noinline__ void faces_jvp(const ModelD& M, const float* __restrict__ X, const float* __restrict__ Xd,
                                       const float* __restrict__ zarena, float* __restrict__ fd, const float* __restrict__ pd) {
  const int N = M.Nz, nfaces = N + 1;
  const float Nf = M.rc.Nf;
  const bool has_nn = M.n_nets > 0;
  const bool expl = !(M.flags & F_IMPLICIT);  // implicit diffusion: the diffusivities act in the backward-Euler step
  if (M.variant == RHS_FC) {
    const float* nd = has_nn ? zarena + M.nn_off[0] * CT : nullptr;
    for (int i = threadIdx.x; i < nfaces * CT; i += NT) {
      const int f = i / CT, c = i - f * CT;
      float e = 0.f;
      if (f > 0 && f < N) {
        if (has_nn) e = nd[(f - 1) * CT + c];
        const float G = Nf * (X[f * CT + c] - X[(f - 1) * CT + c]);
        const float Gd = Nf * (Xd[f * CT + c] - Xd[(f - 1) * CT + c]);
        if (expl && (M.flags & F_MPP)) {  // F -= c nu(G) G
          float dcnu;
          const float cnu = fc_mpp_cnu(M, G, &dcnu);
          e -= fmaf(dcnu, G, cnu) * Gd;
        }
        if (expl && (M.flags & F_CA) && M.rc.K_ca * G < 0.f) e -= M.rc.K_ca * Gd;
      }
      fd[i] = e;
    }
    return;
  }
  const bool mpp = ((M.flags & F_MPP) || M.variant == RHS_INFER) && expl;
  const float eps = M.variant == RHS_TRAIN ? M.rc.eps : 0.f;
  const bool smooth_nn = M.variant == RHS_TRAIN && (M.flags & F_SMOOTH_NN) && has_nn;
  const bool smooth_ri = M.variant == RHS_TRAIN && (M.flags & F_SMOOTH_RI) && mpp;
  constexpr float third = 1.f / 3.f;
  for (int i = threadIdx.x; i < nfaces * CT; i += NT) {
    const int f = i / CT, c = i - f * CT;
    auto grads = [&](int k, float (&G)[3], float (&Gd)[3]) {
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        G[q] = Nf * (X[(q * N + k) * CT + c] - X[(q * N + k - 1) * CT + c]);
        Gd[q] = Nf * (Xd[(q * N + k) * CT + c] - Xd[(q * N + k - 1) * CT + c]);
      }
    };
    auto rid_at = [&](int k) -> float {  // tangent of ri_face at face k (0 at the boundary faces, whose gradients are 0)
      if (k < 1 || k > N - 1) return 0.f;
      float G[3], Gd[3], Ri;
      grads(k, G, Gd);
      return ri_tangent(M, G[0], G[1], G[2], Gd[0], Gd[1], Gd[2], eps, &Ri);
    };
    float e[3] = {0.f, 0.f, 0.f};
    if (f > 0 && f < N) {
      if (has_nn) {
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          const float* r = zarena + M.nn_off[q] * CT + c;
          e[q] = smooth_nn ? filt3(r, f - 1, N - 1, CT) : r[(f - 1) * CT];
        }
      }
      float G[3], Gd[3];
      grads(f, G, Gd);
      if (mpp) {
        float Ri, Rid = ri_tangent(M, G[0], G[1], G[2], Gd[0], Gd[1], Gd[2], eps, &Ri);
        if (smooth_ri) {
          Ri = (ri_face(M, X, f - 1, c, CT, eps) + ri_face(M, X, f, c, CT, eps) + ri_face(M, X, f + 1, c, CT, eps)) * third;
          Rid = (rid_at(f - 1) + Rid + rid_at(f + 1)) * third;
        }
        float nu, s, nuT;
        const float nud = nu_tangent(M, Ri, Rid, pd, &nu, &s);
        const float nuTd = nuT_tangent(M, nu, nud, G[0], G[2], pd, &nuT);
        e[0] -= M.rc.c[0] * fmaf(nud, G[0], nu * Gd[0]);
        e[1] -= M.rc.c[1] * fmaf(nud, G[1], nu * Gd[1]);
        e[2] -= M.rc.c[2] * fmaf(nuTd, G[2], nuT * Gd[2]);
      } else if (expl && (M.flags & F_CA)) {
        if (G[2] < 0.f) e[2] -= M.rc.c[2] * M.rc.kappa * Gd[2];
      }
    }
#pragma unroll
    for (int q = 0; q < 3; ++q) fd[(q * nfaces + f) * CT + c] = e[q];
  }
}

// kd = -A Nf (Fd_{k+1} - Fd_k) plus the Coriolis tangent. kd may alias Xd: a thread reads the two Xd values it needs
// before it writes its own (k, c) of every field.
template <int CT, int NT>
__device__ __noinline__ void centres_jvp(const ModelD& M, const float* Xd, const float* __restrict__ fd, float* kd) {
  const int N = M.Nz, nfaces = N + 1;
  for (int it = threadIdx.x; it < N * CT; it += NT) {
    const int k = it / CT, c = it - k * CT;
    if (M.variant == RHS_FC) {
      kd[k * CT + c] = -M.rc.A[2] * M.rc.Nf * (fd[(k + 1) * CT + c] - fd[k * CT + c]);
      continue;
    }
    const float ud = Xd[k * CT + c], vd = Xd[(N + k) * CT + c];
    float r[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) r[q] = -M.rc.A[q] * M.rc.Nf * (fd[(q * nfaces + k + 1) * CT + c] - fd[(q * nfaces + k) * CT + c]);
    r[0] += M.rc.cor_u_s * vd;  // du/dt = ... + cor_u_s*v
    r[1] -= M.rc.cor_v_s * ud;  // dv/dt = ... - cor_v_s*u
#pragma unroll
    for (int q = 0; q < 3; ++q) kd[(q * N + k) * CT + c] = r[q];
  }
}

// One tangent stage at (X, Xd): the tendencies k go to sink (rhs_tendencies), their tangent to kd ([S][CT], may alias Xd).
// The primal forward runs every phase keeping z (the last layer's z too: act' of the output layer scales its tangent).
// Block barriers inside; ends with one.
template <int CT, int NT, bool WS, int NF, class Sink>
__device__ __forceinline__ void jvp_stage(const ModelD& M, const ModelD& Mp, int Lmax, const PhaseCache& pc, const JvpArgs& a,
                                          const float* X, float* Xd, float* arena, float* zarena, const float* wsm, float* bcf,
                                          const float* qs, float t, Sink sink, float* kd) {
  if (M.flags & F_DIURNAL) {
    if (threadIdx.x < CT) bcf[(M.nbc - 1) * CT + threadIdx.x] = diurnal_top_eff(M, qs[threadIdx.x], t);
  }
  for (int p = 0; p < M.n_phase; ++p) {
    run_phase_cached<CT, NT, WS, true>(M, p, pc, X, arena, zarena, wsm, a.theta);
    __syncthreads();
  }
  if (M.n_phase == 0 && (M.flags & F_DIURNAL)) __syncthreads();
  rhs_tendencies<CT, NT, NF>(Mp, X, arena, bcf, sink);
  __syncthreads();
  for (int l = 0; l <= Lmax; ++l) {
    mlp_tangent_layer<WS, CT, NT>(M, l, X, Xd, arena, zarena, wsm, a.theta, a.theta_dot);
    __syncthreads();
  }
  float* fd = arena + M.flux_off * CT;
  faces_jvp<CT, NT>(M, X, Xd, zarena, fd, a.pdot);
  __syncthreads();
  centres_jvp<CT, NT>(M, Xd, fd, kd);
  __syncthreads();
}

// Tangent of the implicit-diffusion step y = L(D(x)) \ x (implicit_diffusion_tile), which it also runs: on entry x, xd hold
// the incoming state and its tangent, on exit y and yd = L^{-1}(xd - Ldot y), Ldot from Ddot, the diffusivity tangent at x
// (with the mPP-parameter tangent). In the incremental form of implicit_diffusion_tile, with yd = xd + delta:
//   L delta = phi_k - phi_{k+1},   phi_k = r_k (xd_{k-1} - xd_k) + rdot_k (y_{k-1} - y_k)   (phi = 0 on the boundary faces),
// one more Thomas sweep with the coefficients of the forward, recomputed from x as implicit_vjp_tile does.
// xcopy, rd: S CT floats each (a copy of x; rdot, then the sweep's values); scr: 2 S CT floats. Block barriers inside; the
// caller syncs afterwards.
template <int CT, int NT>
__device__ __noinline__ void implicit_jvp_tile(const ModelD& M, float* x, float* xd, float* xcopy, float* rd, float* scr, float h,
                                               const float* pd) {
  const int N = M.Nz, nf = M.nf;
  for (int i = threadIdx.x; i < nf * N * CT; i += NT) {
    const int c = i % CT, k = (i / CT) % N, q = i / (CT * N);
    xcopy[i] = x[i];
    rd[i] = k == 0 ? 0.f : h * M.rc.A[nf == 1 ? 2 : q] * M.rc.Nf * M.rc.Nf * face_diffusivity_dot(M, x, xd, q, k, c, CT, pd);
  }
  __syncthreads();
  implicit_diffusion_tile<CT, NT>(M, x, scr, h);  // x -> y
  __syncthreads();
  float* r = scr;
  for (int i = threadIdx.x; i < nf * N * CT; i += NT) {
    const int c = i % CT, k = (i / CT) % N, q = i / (CT * N);
    r[i] = k == 0 ? 0.f : h * M.rc.A[nf == 1 ? 2 : q] * M.rc.Nf * M.rc.Nf * face_diffusivity(M, xcopy, q, k, c, CT);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < nf * CT; t += NT) {
    const int c = t % CT, q = t / CT;
    float* xdq = xd + q * N * CT + c;
    const float* yq = x + q * N * CT + c;
    float* rq = r + q * N * CT + c;
    float* rdq = rd + q * N * CT + c;
    // row k reads r, rdot of faces k and k+1; face k's slots take the sweep's cp_k and d_k once row k is done
    float cprev = 0.f, dprev = 0.f, phi_lo = 0.f;
    for (int k = 0; k < N; ++k) {
      const float rlo = rq[k * CT], rhi = k + 1 < N ? rq[(k + 1) * CT] : 0.f;
      const float phi_hi = k + 1 < N ? rhi * (xdq[k * CT] - xdq[(k + 1) * CT]) + rdq[(k + 1) * CT] * (yq[k * CT] - yq[(k + 1) * CT]) : 0.f;
      const float inv = 1.f / (1.f + rlo + rhi + rlo * cprev);
      cprev = -rhi * inv;
      dprev = (phi_lo - phi_hi + rlo * dprev) * inv;
      rq[k * CT] = cprev;
      rdq[k * CT] = dprev;
      phi_lo = phi_hi;
    }
    float v = rdq[(N - 1) * CT];
    xdq[(N - 1) * CT] += v;
    for (int k = N - 2; k >= 0; --k) {
      v = rdq[k * CT] - rq[k * CT] * v;
      xdq[k * CT] += v;
    }
  }
}

// bcf / qs of the tile's columns (columns past ncol replicate the last valid one)
template <int CT>
__device__ __forceinline__ void load_column_data(const ModelD& M, const JvpArgs& a, int col0, float* bcf, float* qs) {
  if (threadIdx.x < CT) {
    const int col = min(col0 + (int)threadIdx.x, a.ncol - 1);
    float raw[6], eff[6];
    for (int j = 0; j < M.nbc; ++j) raw[j] = __ldg(a.bcs + (size_t)col * M.nbc + j);
    bc_effective(M, raw, eff);
    for (int j = 0; j < M.nbc; ++j) bcf[j * CT + threadIdx.x] = eff[j];
    qs[threadIdx.x] = (a.Q != nullptr) ? __ldg(a.Q + col) : 0.f;
  }
}

// state and tangent of the tile: x into xs, xdot (or 0) into xd, through the staging buffer xin
template <int CT, int NT>
__device__ __forceinline__ void load_state_pair(const ModelD& M, const JvpArgs& a, int col0, float* xs, float* xd, float* xin,
                                                uint64_t* bar, uint32_t& parity) {
  const int S = M.S;
  load_tile<CT, NT>(xs, xin, bar, parity, a.x, (size_t)S, S, col0, a.ncol);
  __syncthreads();
  if (a.xdot != nullptr) load_tile<CT, NT>(xd, xin, bar, parity, a.xdot, (size_t)S, S, col0, a.ncol);
  else
    for (int i = threadIdx.x; i < S * CT; i += NT) xd[i] = 0.f;
  __syncthreads();
}

// ---- cpz_rhs_jvp: one tangent stage per tile ------------------------------------------------------------------------
template <int CT, int NT, bool WS, int NF>
__device__ __forceinline__ void rhs_jvp_body(const ModelD& M, const ModelD& Mp, const JvpArgs& a, float* smem) {
  const AdjSmem L = adjoint_smem_layout(M, CT);
  float* wsm = smem + L.w;
  float* xs = smem + L.xs;      // x
  float* xd = smem + L.xbar;    // xdot, then the tangent of f (in place)
  float* xin = smem + L.xin;    // transpose staging of the bulk copies
  float* kt = smem + L.xb;      // f
  float* arena = smem + L.arena;
  float* zarena = smem + L.zarena;
  float* bcf = smem + L.bcf;
  float* qs = smem + L.qs;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + ((L.total_floats - 4 + 1) & ~1));
  const int S = M.S, N = M.Nz;
  uint32_t parity = 0;
  const int Lmax = M.n_gemm > 0 ? last_layer_of<CT, NT>(M) : -1;
  PhaseCache pc;
  build_phase_cache<WS, CT, NT>(M, pc);
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  if (WS) load_weights_smem<NT>(M, wsm, a.theta);
  __syncthreads();
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int col0 = tile * CT;
    __syncthreads();
    load_column_data<CT>(M, a, col0, bcf, qs);
    load_state_pair<CT, NT>(M, a, col0, xs, xd, xin, bar, parity);
    jvp_stage<CT, NT, WS, NF>(M, Mp, Lmax, pc, a, xs, xd, arena, zarena, wsm, bcf, qs, a.t,
                              [=](int k0, int c, const float (&dx)[NF][4]) {
#pragma unroll
                                for (int q = 0; q < NF; ++q)
#pragma unroll
                                  for (int kk = 0; kk < 4; ++kk) kt[(q * N + k0 + kk) * CT + c] = dx[q][kk];
                              },
                              xd);
    if (a.y != nullptr) {
      store_tile<CT, NT>(kt, xin, a.y, (size_t)S, S, col0, a.ncol);
      if (threadIdx.x < CT) bulk_wait_read0();
      __syncthreads();
    }
    store_tile<CT, NT>(xd, xin, a.ydot, (size_t)S, S, col0, a.ncol);
    if (threadIdx.x < CT) bulk_wait_read0();  // xin is the next tile's staging buffer
  }
  if (threadIdx.x < CT) bulk_wait0();
}

template <int CT, int NT, bool WS>
__global__ void __launch_bounds__(NT, 1) rhs_jvp_kernel(const __grid_constant__ ModelD Mp, const __grid_constant__ JvpArgs a) {
  extern __shared__ __align__(16) float smem[];
  const AdjSmem L = adjoint_smem_layout(Mp, CT);
  const ModelD& M = model_to_smem<NT>(Mp, smem + L.model);
  if (Mp.nf == 3) rhs_jvp_body<CT, NT, WS, 3>(M, Mp, a, smem);
  else rhs_jvp_body<CT, NT, WS, 1>(M, Mp, a, smem);
}

// ---- cpz_solve_jvp: the tangent-linear model of the fixed-step solve -------------------------------------------------
template <int CT, int NT, bool WS, int NF>
__device__ __forceinline__ void solve_jvp_body(const ModelD& M, const ModelD& Mp, const TableauD& tab, const TimeD& tm, const JvpArgs& a,
                                               float* smem) {
  const AdjSmem L = adjoint_smem_layout(M, CT);
  float* wsm = smem + L.w;
  float* xs = smem + L.xs;    // x
  float* xd = smem + L.xbar;  // xdot
  float* xin = smem + L.xin;  // stage input X_i; transpose staging
  float* xb = smem + L.xb;    // stage tangent Xd_i
  float* arena = smem + L.arena;
  float* zarena = smem + L.zarena;
  float* bcf = smem + L.bcf;
  float* qs = smem + L.qs;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + ((L.total_floats - 4 + 1) & ~1));
  const int S = M.S, N = M.Nz, SC = S * CT, ns = tab.n_stages;
  const float h = tm.dt / (float)tm.n_substeps;
  float* slots = a.kslots + (size_t)blockIdx.x * 2 * ns * SC;
  const KSrc kown{slots, CT, (size_t)SC}, kdown{slots + (size_t)ns * SC, CT, (size_t)SC};
  const bool implicit = (M.flags & F_IMPLICIT) != 0;
  float* imp = adjoint_imp_in_arena(M) ? arena : smem + L.imp;  // scratch of the implicit-diffusion step (2 S CT floats)
  const size_t traj_stride = (size_t)a.n_saved * S;
  uint32_t parity = 0;
  const int Lmax = M.n_gemm > 0 ? last_layer_of<CT, NT>(M) : -1;
  PhaseCache pc;
  build_phase_cache<WS, CT, NT>(M, pc);
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  if (WS) load_weights_smem<NT>(M, wsm, a.theta);
  __syncthreads();

  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int col0 = tile * CT;
    __syncthreads();
    load_column_data<CT>(M, a, col0, bcf, qs);
    load_state_pair<CT, NT>(M, a, col0, xs, xd, xin, bar, parity);
    int frame = 0;
    auto save = [&]() {  // frame `frame` of x (optional) and xdot, in the trajectory's column-contiguous layout
      if (a.y != nullptr) {
        store_tile<CT, NT>(xs, xin, a.y + (size_t)frame * S, traj_stride, S, col0, a.ncol);
        if (threadIdx.x < CT) bulk_wait_read0();
        __syncthreads();
      }
      store_tile<CT, NT>(xd, xin, a.ydot + (size_t)frame * S, traj_stride, S, col0, a.ncol);
      if (threadIdx.x < CT) bulk_wait_read0();  // xin is the next stage input
      __syncthreads();
      ++frame;
    };
    if (tm.save_stride > 0) save();
    for (int n = 0; n < tm.n_steps; ++n) {
      for (int sub = 0; sub < tm.n_substeps; ++sub) {
        const float tb = tm.t0 + (float)(tm.step0 + n) * tm.dt + (float)sub * h;
        if (implicit) {
          implicit_jvp_tile<CT, NT>(M, xs, xd, xin, xb, imp, h, a.pdot);
          __syncthreads();
        }
        for (int i = 0; i < ns; ++i) {
          const float* in = xs;
          float* ind = xd;
          if (i > 0) {
            stage_input<CT, NT>(tab, i, h, xs, kown, SC, xin);
            stage_input<CT, NT>(tab, i, h, xd, kdown, SC, xb);
            __syncthreads();
            in = xin;
            ind = xb;
          }
          float* slot_i = slots + (size_t)i * SC;
          jvp_stage<CT, NT, WS, NF>(M, Mp, Lmax, pc, a, in, ind, arena, zarena, wsm, bcf, qs, tb + tab.c[i] * h,
                                    [=](int k0, int c, const float (&dx)[NF][4]) {
#pragma unroll
                                      for (int q = 0; q < NF; ++q)
#pragma unroll
                                        for (int kk = 0; kk < 4; ++kk) __stcg(slot_i + (q * N + k0 + kk) * CT + c, dx[q][kk]);
                                    },
                                    slots + (size_t)(ns + i) * SC);
        }
        // x += h sum b_i k_i, xdot += h sum b_i kd_i
        for (int e4 = threadIdx.x; e4 < 2 * (SC / 4); e4 += NT) {
          const bool tan = e4 >= SC / 4;
          const int f4 = tan ? e4 - SC / 4 : e4;
          const float* kp = tan ? kdown.p : kown.p;
          float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
          for (int i = 0; i < ns; ++i) {
            const float bi = tab.b[i];
            const float4 kv = __ldcg(reinterpret_cast<const float4*>(kp + (size_t)i * SC) + f4);
            acc.x = fmaf(bi, kv.x, acc.x); acc.y = fmaf(bi, kv.y, acc.y); acc.z = fmaf(bi, kv.z, acc.z); acc.w = fmaf(bi, kv.w, acc.w);
          }
          float4* xp = reinterpret_cast<float4*>(tan ? xd : xs) + f4;
          float4 xv = *xp;
          xv.x = fmaf(h, acc.x, xv.x); xv.y = fmaf(h, acc.y, xv.y); xv.z = fmaf(h, acc.z, xv.z); xv.w = fmaf(h, acc.w, xv.w);
          *xp = xv;
        }
        __syncthreads();
      }
      const int step = n + 1;
      if ((tm.save_stride > 0 && step % tm.save_stride == 0) || (tm.save_stride <= 0 && step == tm.n_steps)) save();
    }
  }
  if (threadIdx.x < CT) bulk_wait0();
}

template <int CT, int NT, bool WS>
__global__ void __launch_bounds__(NT, 1) solve_jvp_kernel(const __grid_constant__ ModelD Mp, const __grid_constant__ TableauD tab,
                                                          const TimeD tm, const __grid_constant__ JvpArgs a) {
  extern __shared__ __align__(16) float smem[];
  const AdjSmem L = adjoint_smem_layout(Mp, CT);
  const ModelD& M = model_to_smem<NT>(Mp, smem + L.model);
  if (Mp.nf == 3) solve_jvp_body<CT, NT, WS, 3>(M, Mp, tab, tm, a, smem);
  else solve_jvp_body<CT, NT, WS, 1>(M, Mp, tab, tm, a, smem);
}

}  // namespace cpz
