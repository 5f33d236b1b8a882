// Discrete-adjoint kernel: reverse sweep of the fixed-step Runge–Kutta solve with step checkpoints.
//
// For x_{n+1} = x_n + h sum_i b_i k_i, k_i = f(X_i, theta), X_i = x_n + h sum_{j<i} a_ij k_j the exact reverse is
//   kbar_i = h (b_i xbar_{n+1} + sum_{j>i} a_ji Xbar_j),   Xbar_i = (df/dX)^T(X_i) kbar_i,
//   thetabar += (df/dtheta)^T(X_i) kbar_i,                  xbar_n = xbar_{n+1} + sum_i Xbar_i.
// One CTA owns CT columns: weights, activations (a and z), x, xbar, the stage input and the stage cotangent live in
// shared memory; the six stage slots (k_j while needed, then Xbar_j) live in an L2-resident global scratch slab.
// Replaces Zygote/DiffEqSensitivity's InterpolatingAdjoint(autojacvec=ZygoteVJP()) used at
// wind_mixing/src/NDE_training.jl:291,304 and free_convection/src/solve.jl:4-5 (continuous adjoint there, exact
// discrete adjoint here; see DESIGN.md).
#pragma once
#include "cpz_device.cuh"
#include "cpz_solve.cuh"

namespace cpz {

struct AdjArgs {
  const float* theta;
  const float* bcs;
  const float* Q;
  const float* targets;  // [ncol][n_saved][S]
  const float* ckpt;     // [n_tiles32][n_ckpt][S][32]: global layout in 32-column tiles whatever the kernel's tile width CT
  const float* kstore;   // [n_tiles32][n_rk_steps][n_stages][S][32] stage tendencies of the forward pass, or null (recompute)
  float* kslots;         // [grid][n_stages][S][CT]
  float* segx;           // [grid][seg_len][S][CT]
  float* gpart;          // [grid][M.slab] gradient slabs in tile layout (zeroed by the host)
  float* lpart;          // [grid][LP]: six squared-error sums, then (from LP/2) the five mPP-parameter gradient sums (zeroed by the host)
  int want_pgrad;        // accumulate d(loss)/d(nu0, nu_m, dRi, Ric, Pr)  (diffusivity_parameter_optimisation.jl:1-33)
  int ncol, n_saved, n_ckpt, n_tiles, seg_len;
  float w[6];
  float inv_prof, inv_grad;  // 1/(Nz*n_saved*ncol_global), 1/((Nz+1)*n_saved*ncol_global)
  unsigned long long* prof;  // optional [8] cycle counters of CTA 0 (CPZ_PROF=1)
  const float* cot;      // [ncol][n_saved][S] cotangent of the trajectory (cpz_solve_vjp): selects adjoint_kernel<..., true>
  float* x0bar;          // [ncol][S] cotangent of x0 (cot mode), or null
};
#define CPZ_APROF_T() ((a.prof && blockIdx.x == 0 && threadIdx.x == 0) ? clock64() : 0)
#define CPZ_APROF_ADD(slot, t0) do { if (a.prof && blockIdx.x == 0 && threadIdx.x == 0) a.prof[slot] += (unsigned long long)(clock64() - (t0)); } while (0)

constexpr int LP = 16;  // floats per CTA in lpart

struct AdjSmem {
  int w, xs, xbar, xin, xb, arena, zarena, imp, bcf, qs, red, model, total_floats;
};
// Scratch of the implicit-diffusion step and its VJP (2 S CT floats: r and the Thomas forward-sweep coefficients): the layer-
// output rows of the activation arena are dead at the step boundaries where these run, so they are used when there are
// enough of them; models with no or very small nets get a dedicated region.
__host__ __device__ inline bool adjoint_imp_in_arena(const ModelD& M) { return M.flux_off >= 2 * M.S; }
__host__ __device__ inline AdjSmem adjoint_smem_layout(const ModelD& M, int CT) {
  AdjSmem L;
  int o = 0;
  L.w = o; o += M.w_in_smem ? M.smem_w_floats : 0;
  L.xs = o; o += M.S * CT;
  L.xbar = o; o += M.S * CT;
  L.xin = o; o += CT * (M.S + 4);  // stage input; doubles as transpose staging
  L.xb = o; o += M.S * CT;         // kbar_i, then Xbar_i; target frame at step boundaries
  L.arena = o; o += M.arena_floats * CT;
  L.zarena = o; o += M.flux_off * CT;  // pre-activations / deltas of every layer output row
  L.imp = o; o += ((M.flags & F_IMPLICIT) && !adjoint_imp_in_arena(M)) ? 2 * M.S * CT : 0;
  L.bcf = o; o += M.nbc * CT;
  L.qs = o; o += CT;
  L.red = o; o += 64;
  L.model = o; o += (int)((sizeof(ModelD) + 15) / 16) * 4;
  L.total_floats = o + 4;
  return L;
}
inline size_t adjoint_other_smem(int S, int nbc, int CT) {
  return ((size_t)3 * S * CT + (size_t)CT * (S + 4) + (size_t)nbc * CT + CT + 64 + 4) * sizeof(float) + ((sizeof(ModelD) + 15) / 16) * 16;
}

// ---- VJP of the face fluxes ------------------------------------------------------------------------------------------
// Reads kbar [S][CT] and the stage input X; writes the cotangent of the last-layer NN outputs into `nnbar` rows
// (zarena at M.nn_off) and the cotangent of the face gradients Gbar_q[face][c] into `gbar` (arena flux rows).
template <int CT, int NT>
__device__ __noinline__ void faces_vjp(const ModelD& M, const float* __restrict__ X, const float* __restrict__ kbar,
                                          float* __restrict__ zarena, float* __restrict__ gbar, double* __restrict__ pg /*[5] or null*/) {
  const int N = M.Nz, nfaces = N + 1;
  const bool has_nn = M.n_nets > 0;
  // implicit diffusion: the stages' RHS carries the NN and boundary fluxes only (the diffusivities act in the backward-Euler
  // solve, whose VJP is implicit_vjp_tile)
  const bool expl = !(M.flags & F_IMPLICIT);
  if (M.variant == RHS_FC) {
    const float AN = M.rc.A[2] * M.rc.Nf;
    float* nb = has_nn ? zarena + M.nn_off[0] * CT : nullptr;
    for (int i = threadIdx.x; i < nfaces * CT; i += NT) {
      const int f = i / CT, c = i - f * CT;
      float g = 0.f;
      if (f > 0 && f < N) {
        const float eb = AN * (kbar[f * CT + c] - kbar[(f - 1) * CT + c]);
        if (has_nn) nb[(f - 1) * CT + c] = eb;
        const float G = M.rc.Nf * (X[f * CT + c] - X[(f - 1) * CT + c]);
        if (expl && (M.flags & F_CA) && M.rc.K_ca * G < 0.f) g = -M.rc.K_ca * eb;
        if (expl && (M.flags & F_MPP)) {  // F -= c nu(G) G
          float dcnu;
          const float cnu = fc_mpp_cnu(M, G, &dcnu);
          g -= eb * fmaf(dcnu, G, cnu);
        }
      }
      gbar[i] = g;
    }
    return;
  }
  const bool mpp = ((M.flags & F_MPP) || M.variant == RHS_INFER) && expl;
  const float eps = M.variant == RHS_TRAIN ? M.rc.eps : 0.f;
  // smoothing filters of the training RHS (NDE_training.jl:98-102,121-123; filtering_operators.jl:1-15): both are linear
  // width-3 running means, so their VJP is the same stencil transposed. These variants are rare, so the neighbouring
  // faces' quantities are simply recomputed per thread instead of staged.
  const bool smooth_nn = M.variant == RHS_TRAIN && (M.flags & F_SMOOTH_NN) && has_nn;
  const bool smooth_ri = M.variant == RHS_TRAIN && (M.flags & F_SMOOTH_RI) && mpp;
  constexpr float third = 1.f / 3.f;
  for (int i = threadIdx.x; i < nfaces * CT; i += NT) {
    const int f = i / CT, c = i - f * CT;
    // cotangent of the total flux of field q at interior face k (0 at the boundary faces: their fluxes are data)
    auto ebq = [&](int q, int k) -> float {
      return (k > 0 && k < N) ? M.rc.A[q] * M.rc.Nf * (kbar[(q * N + k) * CT + c] - kbar[(q * N + k - 1) * CT + c]) : 0.f;
    };
    auto ri_used = [&](int k) -> float {  // the Richardson number the diffusivity at interior face k is evaluated at
      if (!smooth_ri) return ri_face(M, X, k, c, CT, eps);
      return (ri_face(M, X, k - 1, c, CT, eps) + ri_face(M, X, k, c, CT, eps) + ri_face(M, X, k + 1, c, CT, eps)) * third;
    };
    auto rib_used = [&](int k) -> float {  // cotangent of ri_used(k)
      if (k < 1 || k > N - 1) return 0.f;
      const float Gu = M.rc.Nf * (X[k * CT + c] - X[(k - 1) * CT + c]);
      const float Gv = M.rc.Nf * (X[(N + k) * CT + c] - X[(N + k - 1) * CT + c]);
      const float GT = M.rc.Nf * (X[(2 * N + k) * CT + c] - X[(2 * N + k - 1) * CT + c]);
      const float y2 = 2.f * (ri_used(k) - M.rc.Ric) * M.rc.inv_dRi;
      const float s = __fdividef(1.f, 1.f + __expf(y2));
      const float nub = -(M.rc.c[0] * Gu * ebq(0, k) + M.rc.c[1] * Gv * ebq(1, k) + M.rc.inv_Pr * M.rc.c[2] * GT * ebq(2, k));
      return nub * (-2.f * M.rc.inv_dRi * M.rc.nu_m * s * (1.f - s));
    };
    float gb[3] = {0.f, 0.f, 0.f};
    if (f > 0 && f < N) {
      float eb[3];
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        eb[q] = ebq(q, f);
        if (has_nn) {
          float nb = eb[q];
          if (smooth_nn) {  // transposed filter: output j = f-1 of the N-1 NN outputs collects rows j-1, j, j+1
            const int j = f - 1, n = N - 1;
            nb = 0.f;
            for (int r = max(j - 1, 0); r <= min(j + 1, n - 1); ++r) nb += ((r == 0 || r == n - 1) ? 0.5f : third) * ebq(q, r + 1);
          }
          zarena[(M.nn_off[q] + f - 1) * CT + c] = nb;
        }
      }
      const float Gu = M.rc.Nf * (X[f * CT + c] - X[(f - 1) * CT + c]);
      const float Gv = M.rc.Nf * (X[(N + f) * CT + c] - X[(N + f - 1) * CT + c]);
      const float GT = M.rc.Nf * (X[(2 * N + f) * CT + c] - X[(2 * N + f - 1) * CT + c]);
      if (mpp) {
        const float gu = Gu + eps, gv = Gv + eps, gT = GT + eps;
        const float su = M.rc.sig_u * gu, sv = M.rc.sig_v * gv;
        const float S2 = su * su + sv * sv;
        // clamped: where the shear vanishes the step is saturated (s (1-s) = 0) and the cotangents below must be 0, not 0 * inf
        const float iS2 = __fdividef(1.f, fmaxf(S2, 1e-18f));
        const float Ri = M.rc.BzC * gT * iS2;
        const float y2 = 2.f * ((smooth_ri ? ri_used(f) : Ri) - M.rc.Ric) * M.rc.inv_dRi;
        const float s = __fdividef(1.f, 1.f + __expf(y2));
        const float nu = M.rc.nu0 + M.rc.nu_m * s;
        float nuT = nu * M.rc.inv_Pr, dnuT = M.rc.inv_Pr;
        if (M.variant == RHS_INFER && (M.flags & F_CA)) {
          const float test = (M.flags & F_CA_LITERAL_U) ? Gu : GT;
          if (!(test > 0.f)) { nuT = M.rc.kappa; dnuT = 0.f; }
        }
        const float Du = -eb[0], Dv = -eb[1], DT = -eb[2];  // cotangents of the diffusive fluxes
        gb[0] = M.rc.c[0] * nu * Du;
        gb[1] = M.rc.c[1] * nu * Dv;
        gb[2] = M.rc.c[2] * nuT * DT;
        const float nub = M.rc.c[0] * Gu * Du + M.rc.c[1] * Gv * Dv + dnuT * M.rc.c[2] * GT * DT;
        // s(1-s) underflows cleanly to 0 for |y| large; inf*0 cannot occur because s is in [0,1]
        float Rib = nub * (-2.f * M.rc.inv_dRi * M.rc.nu_m * s * (1.f - s));
        if (smooth_ri) Rib = (rib_used(f - 1) + Rib + rib_used(f + 1)) * third;  // transposed face filter (interior rows only)
        if (pg != nullptr && !smooth_ri) {
          // gradient wrt p = (nu0, nu_m, dRi, Ric, Pr) of `DE` (diffusivity_parameter_optimisation.jl:2,20): nu = nu0 + nu_m s(y),
          // s = 1/(1+e^y), y = 2 (Ri - Ric)/dRi; nu_T = nu/Pr. nub is the cotangent of nu at this face and stage.
          const float ss = s * (1.f - s);
          pg[0] += nub;
          pg[1] += nub * s;
          pg[2] += nub * M.rc.nu_m * ss * y2 * M.rc.inv_dRi;
          pg[3] += nub * M.rc.nu_m * ss * 2.f * M.rc.inv_dRi;
          if (dnuT != 0.f) pg[4] += eb[2] * M.rc.c[2] * nu * GT * M.rc.inv_Pr * M.rc.inv_Pr;
        }
        gb[2] += Rib * M.rc.BzC * iS2;
        const float t = -Rib * Ri * iS2 * 2.f;
        gb[0] += t * M.rc.sig_u * su;
        gb[1] += t * M.rc.sig_v * sv;
      } else if (expl && (M.flags & F_CA)) {
        if (GT < 0.f) gb[2] = -M.rc.c[2] * M.rc.kappa * eb[2];
      }
    }
#pragma unroll
    for (int q = 0; q < 3; ++q) gbar[(q * nfaces + f) * CT + c] = gb[q];
  }
}

// Direct (non-MLP) part of Xbar_i = (df/dX)^T kbar_i, written IN PLACE over kbar (each thread owns (k,c) of all fields).
template <int CT, int NT>
__device__ __noinline__ void centres_vjp(const ModelD& M, float* __restrict__ kbar_xb, const float* __restrict__ gbar) {
  const int N = M.Nz, nfaces = N + 1;
  for (int it = threadIdx.x; it < N * CT; it += NT) {
    const int k = it / CT, c = it - k * CT;
    if (M.variant == RHS_FC) {
      const float g0 = (k >= 1) ? gbar[k * CT + c] : 0.f;
      const float g1 = (k + 1 <= N - 1) ? gbar[(k + 1) * CT + c] : 0.f;
      kbar_xb[k * CT + c] = M.rc.Nf * (g0 - g1);
      continue;
    }
    const float kbu = kbar_xb[k * CT + c], kbv = kbar_xb[(N + k) * CT + c];
    float r[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      const float g0 = (k >= 1) ? gbar[(q * nfaces + k) * CT + c] : 0.f;
      const float g1 = (k + 1 <= N - 1) ? gbar[(q * nfaces + k + 1) * CT + c] : 0.f;
      r[q] = M.rc.Nf * (g0 - g1);
    }
    r[0] -= M.rc.cor_v_s * kbv;  // dv/dt = ... - cor_v_s*u
    r[1] += M.rc.cor_u_s * kbu;  // du/dt = ... + cor_u_s*v
#pragma unroll
    for (int q = 0; q < 3; ++q) kbar_xb[(q * N + k) * CT + c] = r[q];
  }
}

// ---- MLP backward tiles ------------------------------------------------------------------------------------------------
// Backward-data for one gemm: abar[k][c] = sum_j W[k][j] delta[j][c] on a 4-row x 4-column tile.
// Returns the tile in acc (pairs over columns); the caller applies act' or accumulates into Xbar.
template <bool WS, int CT>
__device__ __forceinline__ void bwd_data_tile(const GemmD& g, const float* __restrict__ W, const float* __restrict__ delta,
                                              int k0, int cg, float (&acc)[4][4]) {
  const int K = g.K, N = g.N;
  const int ldw = WS ? g.Npad : N;
  int kr[4];
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) kr[kk] = min(k0 + kk, K - 1) * ldw;
  const float* dp = delta + 4 * cg;
  const int N4 = WS ? (N & ~3) : 0;
#pragma unroll 2
  for (int j = 0; j < N4; j += 4) {
    float4 d[4];
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) d[jj] = *reinterpret_cast<const float4*>(dp + (j + jj) * CT);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const float4 wv = *reinterpret_cast<const float4*>(W + kr[kk] + j);
      const float wj[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        acc[kk][0] = fmaf(wj[jj], d[jj].x, acc[kk][0]);
        acc[kk][1] = fmaf(wj[jj], d[jj].y, acc[kk][1]);
        acc[kk][2] = fmaf(wj[jj], d[jj].z, acc[kk][2]);
        acc[kk][3] = fmaf(wj[jj], d[jj].w, acc[kk][3]);
      }
    }
  }
  for (int j = N4; j < N; ++j) {
    const float4 d = *reinterpret_cast<const float4*>(dp + j * CT);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const float wv = WS ? W[kr[kk] + j] : __ldg(W + kr[kk] + j);
      acc[kk][0] = fmaf(wv, d.x, acc[kk][0]);
      acc[kk][1] = fmaf(wv, d.y, acc[kk][1]);
      acc[kk][2] = fmaf(wv, d.z, acc[kk][2]);
      acc[kk][3] = fmaf(wv, d.w, acc[kk][3]);
    }
  }
}

// Weight gradient of one gemm on a 4(k) x 4(j) tile: dW[k][j] += sum_c a[k][c] delta[j][c], accumulated into the
// tile's 16 contiguous floats of the CTA's gradient slab with a plain vectorised read-modify-write (every tile has
// exactly one owner thread per CTA, stages are separated by block barriers, so no atomics are needed; the 16 floats of
// consecutive lanes are contiguous, i.e. fully coalesced).
template <int CT>
__device__ __forceinline__ void bwd_weight_tile(const GemmD& g, const float* __restrict__ a, const float* __restrict__ delta,
                                                int k0, int j0, float* __restrict__ gtile) {
  const int K = g.K, N = g.N;
  float4 old[4];
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) old[kk] = __ldcg(reinterpret_cast<const float4*>(gtile) + kk);  // issued early, used last
  float acc[4][4];
#pragma unroll
  for (int kk = 0; kk < 4; ++kk)
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) acc[kk][jj] = 0.f;
  int kr[4], jr[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) { kr[t] = min(k0 + t, K - 1) * CT; jr[t] = min(j0 + t, N - 1) * CT; }
  // The reduction runs over the tile's columns in chunks of 4. Lanes of a quarter-warp own tiles whose delta rows are
  // 4 rows (= 512 B, the same banks) apart, so every lane starts at a different chunk: at each step the 8 lanes read 8
  // different 16-byte bank groups (conflict-free) instead of colliding 8-way on one.
  const int rot = (threadIdx.x & 7) * 4;
#pragma unroll 2
  for (int c0 = 0; c0 < CT; c0 += 4) {
    const int c = (c0 + rot) & (CT - 1);
    float4 av[4], dv[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      av[t] = *reinterpret_cast<const float4*>(a + kr[t] + c);
      dv[t] = *reinterpret_cast<const float4*>(delta + jr[t] + c);
    }
#pragma unroll
    for (int kk = 0; kk < 4; ++kk)
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        acc[kk][jj] = fmaf(av[kk].x, dv[jj].x, acc[kk][jj]);
        acc[kk][jj] = fmaf(av[kk].y, dv[jj].y, acc[kk][jj]);
        acc[kk][jj] = fmaf(av[kk].z, dv[jj].z, acc[kk][jj]);
        acc[kk][jj] = fmaf(av[kk].w, dv[jj].w, acc[kk][jj]);
      }
  }
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    // rows/columns past the layer edge hold duplicates of the clamped row: zero them so the slab stays clean
    const bool kv = k0 + kk < K;
    float4 o = old[kk];
    o.x += (kv && j0 + 0 < N) ? acc[kk][0] : 0.f;
    o.y += (kv && j0 + 1 < N) ? acc[kk][1] : 0.f;
    o.z += (kv && j0 + 2 < N) ? acc[kk][2] : 0.f;
    o.w += (kv && j0 + 3 < N) ? acc[kk][3] : 0.f;
    __stcg(reinterpret_cast<float4*>(gtile) + kk, o);
  }
}

// Backward through layer index `l` of every net that has it: weight/bias gradients, then delta of the previous layer
// (or the accumulation of W_0 delta_0 into Xbar for l == 0). One block barrier must follow.
template <bool WS, int CT, int NT>
__device__ __noinline__ void mlp_backward_layer(const ModelD& M, int l, const float* __restrict__ Xin,
                                                   const float* __restrict__ arena, float* __restrict__ zarena,
                                                   float* __restrict__ xb, const float* __restrict__ wsm,
                                                   const float* __restrict__ theta, float* __restrict__ gpart) {
  constexpr int NCG = CT / 4;
  // gemms of layer l (at most one per net, three nets) and the prefix sums of their tile counts; unused slots repeat
  // the total so that the slot search below never selects them
  int gl[3] = {0, 0, 0}, end[4] = {0, 0, 0, 0}, wend[4] = {0, 0, 0, 0}, bend[4] = {0, 0, 0, 0}, ng = 0;
  for (int gi = 0; gi < M.n_gemm && ng < 3; ++gi) {
    const GemmD& g = M.gemm[gi];
    if (g.layer != l) continue;
    gl[ng] = gi;
    end[ng + 1] = end[ng] + ((g.K + 3) / 4) * NCG;
    wend[ng + 1] = wend[ng] + ((g.K + 3) / 4) * ((g.N + 3) / 4);
    bend[ng + 1] = bend[ng] + g.N;
    ++ng;
  }
  for (int q = ng + 1; q < 4; ++q) { end[q] = end[ng]; wend[q] = wend[ng]; bend[q] = bend[ng]; }
  // (a) backward-data
  if (l == 0) {
    const int S = M.S;
    const int nkg = (S + 3) / 4;
    for (int tile = threadIdx.x; tile < nkg * NCG; tile += NT) {
      const int cg = tile % NCG, k0 = (tile / NCG) * 4;
      float acc[4][4];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) acc[kk][cc] = 0.f;
      for (int gi = 0; gi < M.n_gemm; ++gi) {
        const GemmD& g = M.gemm[gi];
        if (g.layer != 0) continue;
        const float* W = WS ? wsm + g.sw_off : theta + g.w_off;
        bwd_data_tile<WS, CT>(g, W, zarena + g.out_off * CT, k0, cg, acc);
      }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        if (k0 + kk < S) {
          float4* p = reinterpret_cast<float4*>(xb + (k0 + kk) * CT + 4 * cg);
          float4 v = *p;
          v.x += acc[kk][0]; v.y += acc[kk][1]; v.z += acc[kk][2]; v.w += acc[kk][3];
          *p = v;
        }
      }
    }
  } else {
    // the nets' gemms of layer l share one flattened tile space, so that 3 x 40 tiles fill one pass of the CTA instead of
    // three passes of 40 threads (the nets touch disjoint rows of zarena)
    for (int t = threadIdx.x; t < end[ng]; t += NT) {
      const int q = (t >= end[1]) + (t >= end[2]);
      const GemmD& g = M.gemm[q == 0 ? gl[0] : (q == 1 ? gl[1] : gl[2])];
      const int tile = t - (q == 0 ? 0 : (q == 1 ? end[1] : end[2]));
      // the producer of this gemm's input is the gemm of the same net at layer l-1
      int gp = -1;
      for (int gj = 0; gj < M.n_gemm; ++gj)
        if (M.gemm[gj].net == g.net && M.gemm[gj].layer == l - 1) gp = gj;
      const int actp = M.gemm[gp].act;
      const float* W = WS ? wsm + g.sw_off : theta + g.w_off;
      float* zprev = zarena + g.in_off * CT;
      const int cg = tile % NCG, k0 = (tile / NCG) * 4;
      float acc[4][4];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) acc[kk][cc] = 0.f;
      bwd_data_tile<WS, CT>(g, W, zarena + g.out_off * CT, k0, cg, acc);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        if (k0 + kk < g.K) {
          float4* p = reinterpret_cast<float4*>(zprev + (k0 + kk) * CT + 4 * cg);
          const float4 z = *p;
          float4 d;
          d.x = acc[kk][0] * act_grad(actp, z.x);
          d.y = acc[kk][1] * act_grad(actp, z.y);
          d.z = acc[kk][2] * act_grad(actp, z.z);
          d.w = acc[kk][3] * act_grad(actp, z.w);
          *p = d;
        }
      }
    }
  }
  // (b) weight and bias gradients of layer l (read delta_l and a_{l-1}; neither is written by (a)), again over one
  // flattened tile space. No barrier separates (a) from (b), so (b) is dealt from the top of the CTA downwards: the
  // threads that had no (or one fewer) (a) tile take the first weight tiles. At layer 0 an (a) tile sums over every
  // net and costs about sum(N)/CT weight tiles, so the threads without one take that many extra tiles up front.
  {
    const int u = NT - 1 - (int)threadIdx.x;
    int idle = 0, extra = 0;
    if (l == 0) {
      idle = NT - min(NT, ((M.S + 3) / 4) * NCG);
      extra = idle > 0 ? min(bend[ng] / CT, wend[ng] / idle) : 0;
    }
    const int head = idle * extra, mine = u < idle ? extra : 0;
    for (int i = 0;; ++i) {
      const int t = i < mine ? u + i * idle : head + u + (i - mine) * NT;
      if (t >= wend[ng]) break;
      const int q = (t >= wend[1]) + (t >= wend[2]);
      const GemmD& g = M.gemm[q == 0 ? gl[0] : (q == 1 ? gl[1] : gl[2])];
      const int tile = t - (q == 0 ? 0 : (q == 1 ? wend[1] : wend[2]));
      const float* a = g.in_off < 0 ? Xin : arena + g.in_off * CT;
      const int njg = (g.N + 3) / 4;
      const int jg = tile % njg, kg = tile / njg;
      bwd_weight_tile<CT>(g, a, zarena + g.out_off * CT, kg * 4, jg * 4, gpart + g.gw_off + (size_t)tile * 16);
    }
  }
  for (int t = threadIdx.x; t < bend[ng]; t += NT) {
    const int q = (t >= bend[1]) + (t >= bend[2]);
    const GemmD& g = M.gemm[q == 0 ? gl[0] : (q == 1 ? gl[1] : gl[2])];
    const int j = t - (q == 0 ? 0 : (q == 1 ? bend[1] : bend[2]));
    const float* delta = zarena + g.out_off * CT;
    float s = 0.f;
    for (int c = 0; c < CT; c += 4) {
      const float4 d = *reinterpret_cast<const float4*>(delta + j * CT + c);
      s += (d.x + d.y) + (d.z + d.w);
    }
    gpart[g.gb_off + j] += s;  // exactly one thread per CTA owns this entry
  }
}

// NOTE on (a)/(b) hazards for l > 0: (a) overwrites z_{l-1} (rows of layer l-1) with delta_{l-1}; (b) of layer l reads
// a_{l-1} from the ARENA (post-activation copy), not from zarena, so the two never touch the same rows.

template <int CT, int NT>
__device__ __forceinline__ int last_layer_of(const ModelD& M) {
  int L = 0;
  for (int gi = 0; gi < M.n_gemm; ++gi) L = max(L, M.gemm[gi].layer);
  return L;
}

// MLP forward keeping z and a for mlp_backward_layer. The last layer's outputs are not needed (everything downstream of
// the nets is affine in them), so its phases are skipped. Each phase ends with a block barrier.
template <int CT, int NT, bool WS>
__device__ __forceinline__ void mlp_forward_keep(const ModelD& M, int Lmax, const PhaseCache& pc, const float* in, float* arena,
                                                 float* zarena, const float* wsm, const float* theta) {
  for (int p = 0; p < M.n_phase; ++p) {
    if (M.gemm[M.phase[p].g0].layer == Lmax && M.gemm[M.phase[p].g1 - 1].layer == Lmax) continue;
    run_phase_cached<CT, NT, WS, true>(M, p, pc, in, arena, zarena, wsm, theta);
    __syncthreads();
  }
}

// Reverse of the MLP, last layer first, from the NN-output cotangents in zarena: weight gradients into gpart, the input
// cotangent added to xb. Each layer ends with a block barrier.
template <int CT, int NT, bool WS>
__device__ __forceinline__ void mlp_backward(const ModelD& M, int Lmax, const float* in, const float* arena, float* zarena,
                                             float* xb, const float* wsm, const float* theta, float* gpart) {
  for (int l = Lmax; l >= 0; --l) {
    mlp_backward_layer<WS, CT, NT>(M, l, in, arena, zarena, xb, wsm, theta, gpart);
    __syncthreads();
  }
}

// Block reduction (fixed order) of the five FP64 mPP-parameter sums into this CTA's lpart row at LP/2 .. LP/2+4.
// red: NT/32 floats of shared scratch.
template <int NT>
__device__ __forceinline__ void store_pgrad_sums(const double (&pgs)[5], float* red, float* lpart) {
  for (int q = 0; q < 5; ++q) {
    double vd = pgs[q];
    for (int o = 16; o > 0; o >>= 1) vd += __shfl_xor_sync(0xffffffffu, vd, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = (float)vd;
    __syncthreads();
    if (threadIdx.x == 0) {
      float s = 0.f;
      for (int wdx = 0; wdx < NT / 32; ++wdx) s += red[wdx];
      lpart[(size_t)blockIdx.x * LP + LP / 2 + q] = s;
    }
    __syncthreads();
  }
}

// loss terms at one saved frame: accumulates the 6 squared-error sums and adds d(loss)/dx to xbar.
// x: state tile, tg: target tile (same layout). Invalid columns (c >= nvalid) contribute nothing.
template <int CT, int NT>
__device__ __noinline__ void loss_frame(const ModelD& M, const AdjArgs& a, const float* __restrict__ x,
                                           const float* __restrict__ tg, float* __restrict__ xbar, int nvalid,
                                           float (&lsum)[6]) {
  const int N = M.Nz;
  for (int it = threadIdx.x; it < N * CT; it += NT) {
    const int k = it / CT, c = it - k * CT;
    if (c >= nvalid) continue;
    for (int q = 0; q < M.nf; ++q) {
      const int wq = M.nf == 1 ? 2 : q;
      const int e = (q * N + k) * CT + c;
      const float d = x[e] - tg[e];
      lsum[wq] = fmaf(d, d, lsum[wq]);
      float gx = a.w[wq] * 2.f * a.inv_prof * d;
      if (M.nf == 3 && a.w[3 + q] != 0.f) {
        // gradient loss: g[f] = Nf (d[f]-d[f-1]) on interior faces f=1..N-1; this thread owns face f=k (if k>=1)
        float g0 = 0.f, g1 = 0.f;
        if (k >= 1) {
          g0 = M.rc.Nf * (d - (x[e - CT] - tg[e - CT]));
          lsum[3 + q] = fmaf(g0, g0, lsum[3 + q]);
        }
        if (k + 1 <= N - 1) g1 = M.rc.Nf * ((x[e + CT] - tg[e + CT]) - d);
        gx += a.w[3 + q] * 2.f * a.inv_grad * M.rc.Nf * (g0 - g1);
      }
      xbar[e] += gx;
    }
  }
}

// cot mode (cpz_solve_vjp): the trajectory cotangent of one saved frame, cb (a tile loaded like the targets), goes into
// xbar unchanged. load_tile replicates the last valid column into the padding columns, which must stay at zero.
template <int CT, int NT>
__device__ __noinline__ void cot_frame(const ModelD& M, const float* __restrict__ cb, float* __restrict__ xbar, int nvalid) {
  for (int it = threadIdx.x; it < M.S * CT; it += NT) {
    if (it % CT < nvalid) xbar[it] += cb[it];
  }
}

// Global arrays shared with the forward kernels (checkpoints, stored stage tendencies) are laid out in 32-column tiles
// [tile32][...][S][32] whatever this kernel's tile width CT is (CT divides 32): float4 number e4 of a [S][CT] tile sits at
// row e4 / (CT/4), float4 e4 % (CT/4) of a row of `ld` floats. The CTA's private scratch uses ld = CT (contiguous).
constexpr int LT = 32;
template <int CT>
__device__ __forceinline__ const float4* row4(const float* base, int ld, int e4) {
  constexpr int Q = CT / 4;
  return reinterpret_cast<const float4*>(base + (size_t)(e4 / Q) * ld) + (e4 % Q);
}
struct KSrc {  // where the forward stage tendencies k_j of the current Runge–Kutta step are
  const float* p;
  int ld;          // row stride (CT: private slots, 32: stored by the forward pass)
  size_t stride;   // floats between stages
};

// x_in = xs + h * sum_{j<i} a_ij k_j
template <int CT, int NT>
__device__ __noinline__ void stage_input(const TableauD& tab, int i, float h, const float* __restrict__ xs,
                                            const KSrc ks, int SC, float* __restrict__ xin) {
  for (int e4 = threadIdx.x; e4 < SC / 4; e4 += NT) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int j = 0; j < i; ++j) {
      const float aij = tab.a[i][j];
      if (aij != 0.f) {
        const float4 kv = __ldcg(row4<CT>(ks.p + (size_t)j * ks.stride, ks.ld, e4));
        acc.x = fmaf(aij, kv.x, acc.x); acc.y = fmaf(aij, kv.y, acc.y);
        acc.z = fmaf(aij, kv.z, acc.z); acc.w = fmaf(aij, kv.w, acc.w);
      }
    }
    const float4 xv = reinterpret_cast<const float4*>(xs)[e4];
    reinterpret_cast<float4*>(xin)[e4] = make_float4(fmaf(h, acc.x, xv.x), fmaf(h, acc.y, xv.y), fmaf(h, acc.z, xv.z),
                                                     fmaf(h, acc.w, xv.w));
  }
}

// VJP of y = L(D(x)) \ x (implicit_diffusion_tile): on entry `xbar` holds ybar, on exit xbar_x.
//   lambda = L^{-1} ybar (L is symmetric);  rbar_k = -(lambda_k - lambda_{k-1}) (y_k - y_{k-1});  Dbar = h A Nz^2 rbar;
//   xbar = lambda + (dD/dx)^T Dbar through the same Richardson-number chain as faces_vjp.
// x: the incoming state (diffusivities are evaluated there), y: the outgoing state, scr: 2 S CT floats, gbar: 3 (Nz+1) CT floats.
template <int CT, int NT>
__device__ __noinline__ void implicit_vjp_tile(const ModelD& M, const float* __restrict__ x, const float* __restrict__ y,
                                                 float* __restrict__ xbar, float* __restrict__ scr, float* __restrict__ gbar,
                                                 float h, double* __restrict__ pg) {
  const int N = M.Nz, nf = M.nf, nfaces = N + 1;
  float* r = scr;
  float* cp = scr + nf * N * CT;
  for (int i = threadIdx.x; i < nf * N * CT; i += NT) {
    const int c = i % CT, k = (i / CT) % N, q = i / (CT * N);
    r[i] = k == 0 ? 0.f : h * M.rc.A[nf == 1 ? 2 : q] * M.rc.Nf * M.rc.Nf * face_diffusivity(M, x, q, k, c, CT);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < nf * CT; t += NT) {  // lambda = L \ ybar, in place
    const int c = t % CT, q = t / CT;
    float* xq = xbar + q * N * CT + c;
    const float* rq = r + q * N * CT + c;
    float* cq = cp + q * N * CT + c;
    float cprev = 0.f, dprev = 0.f;
    for (int k = 0; k < N; ++k) {
      const float rlo = rq[k * CT], rhi = k + 1 < N ? rq[(k + 1) * CT] : 0.f;
      const float inv = 1.f / (1.f + rlo + rhi + rlo * cprev);
      cprev = -rhi * inv;
      dprev = (xq[k * CT] + rlo * dprev) * inv;
      cq[k * CT] = cprev;
      xq[k * CT] = dprev;
    }
    float v = xq[(N - 1) * CT];
    for (int k = N - 2; k >= 0; --k) {
      v = xq[k * CT] - cq[k * CT] * v;
      xq[k * CT] = v;
    }
  }
  __syncthreads();
  // cotangents of the face gradients
  for (int i = threadIdx.x; i < nfaces * CT; i += NT) {
    const int f = i / CT, c = i - f * CT;
    float gb[3] = {0.f, 0.f, 0.f};
    if (f > 0 && f < N) {
      float Db[3];  // cotangent of D_q at this face
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        Db[q] = 0.f;
        if (q < nf) {
          const int e = (q * N + f) * CT + c;
          const float rb = -(xbar[e] - xbar[e - CT]) * (y[e] - y[e - CT]);
          Db[q] = h * M.rc.A[nf == 1 ? 2 : q] * M.rc.Nf * M.rc.Nf * rb;
        }
      }
      if (M.variant == RHS_FC) {
        if (M.flags & F_MPP) {
          const float G = M.rc.Nf * (x[f * CT + c] - x[(f - 1) * CT + c]);
          float dcnu;
          fc_mpp_cnu(M, G, &dcnu);
          gb[0] = Db[0] * dcnu;  // the convective-adjustment part K [G < 0] is piecewise constant
        }
      } else {
        const bool mpp = (M.flags & F_MPP) || M.variant == RHS_INFER;
        if (mpp) {
          const float eps = M.variant == RHS_TRAIN ? M.rc.eps : 0.f;
          const float Gu = M.rc.Nf * (x[f * CT + c] - x[(f - 1) * CT + c]);
          const float Gv = M.rc.Nf * (x[(N + f) * CT + c] - x[(N + f - 1) * CT + c]);
          const float GT = M.rc.Nf * (x[(2 * N + f) * CT + c] - x[(2 * N + f - 1) * CT + c]);
          const float su = M.rc.sig_u * (Gu + eps), sv = M.rc.sig_v * (Gv + eps);
          const float iS2 = __fdividef(1.f, fmaxf(su * su + sv * sv, 1e-18f));  // see faces_vjp
          const float Ri = M.rc.BzC * (GT + eps) * iS2;
          const float y2 = 2.f * (Ri - M.rc.Ric) * M.rc.inv_dRi;
          const float s = __fdividef(1.f, 1.f + __expf(y2));
          const float nu = M.rc.nu0 + M.rc.nu_m * s;
          float dnuT = M.rc.inv_Pr;
          if (M.variant == RHS_INFER && (M.flags & F_CA)) {
            const float test = (M.flags & F_CA_LITERAL_U) ? Gu : GT;
            if (!(test > 0.f)) dnuT = 0.f;
          }
          const float nub = M.rc.c[0] * Db[0] + M.rc.c[1] * Db[1] + M.rc.c[2] * dnuT * Db[2];
          const float ss = s * (1.f - s);
          if (pg != nullptr) {
            pg[0] += nub;
            pg[1] += nub * s;
            pg[2] += nub * M.rc.nu_m * ss * y2 * M.rc.inv_dRi;
            pg[3] += nub * M.rc.nu_m * ss * 2.f * M.rc.inv_dRi;
            if (dnuT != 0.f) pg[4] -= Db[2] * M.rc.c[2] * nu * M.rc.inv_Pr * M.rc.inv_Pr;
          }
          const float Rib = nub * (-2.f * M.rc.inv_dRi * M.rc.nu_m * ss);
          gb[2] = Rib * M.rc.BzC * iS2;
          const float t = -Rib * Ri * iS2 * 2.f;
          gb[0] = t * M.rc.sig_u * su;
          gb[1] = t * M.rc.sig_v * sv;
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 3; ++q)
      if (q < nf) gbar[(q * nfaces + f) * CT + c] = gb[q];
  }
  __syncthreads();
  for (int it = threadIdx.x; it < nf * N * CT; it += NT) {
    const int c = it % CT, k = (it / CT) % N, q = it / (CT * N);
    const float g0 = (k >= 1) ? gbar[(q * nfaces + k) * CT + c] : 0.f;
    const float g1 = (k + 1 <= N - 1) ? gbar[(q * nfaces + k + 1) * CT + c] : 0.f;
    xbar[it] += M.rc.Nf * (g0 - g1);
  }
}

// COT: cot mode (cpz_solve_vjp) — the trajectory cotangent a.cot replaces the loss terms at the saved frames and the
// cotangent of x0 is stored to a.x0bar. A template parameter so that the loss-mode kernels are compiled as before.
template <int CT, int NT, bool WS, int NF, bool COT>
__device__ __forceinline__ void adjoint_body(const ModelD& M, const ModelD& Mp, const TableauD& tab, const TimeD& tm,
                                             const AdjArgs& a, float* smem) {
  const AdjSmem L = adjoint_smem_layout(M, CT);
  float* wsm = smem + L.w;
  float* xs = smem + L.xs;
  float* xbar = smem + L.xbar;
  float* xin = smem + L.xin;
  float* xb = smem + L.xb;
  float* arena = smem + L.arena;
  float* zarena = smem + L.zarena;
  float* bcf = smem + L.bcf;
  float* qs = smem + L.qs;
  float* red = smem + L.red;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + ((L.total_floats - 4 + 1) & ~1));
  const int S = M.S, N = M.Nz, SC = S * CT, ns = tab.n_stages;
  const float h = tm.dt / (float)tm.n_substeps;
  float* slots = a.kslots + (size_t)blockIdx.x * ns * SC;
  float* segx = a.segx + (size_t)blockIdx.x * a.seg_len * SC;
  float* gpart = a.gpart + (size_t)blockIdx.x * M.slab;
  float* gflux = arena + M.flux_off * CT;
  const bool implicit = (M.flags & F_IMPLICIT) != 0;
  float* imp = adjoint_imp_in_arena(M) ? arena : smem + L.imp;  // scratch of the implicit-diffusion step (2 S CT floats)
  uint32_t parity = 0;
  float lsum[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  double pgs[5] = {0., 0., 0., 0., 0.};  // FP64 accumulators: sums of ~1e8 small terms of both signs (rare path, 5 adds per face)
  const int Lmax = M.n_gemm > 0 ? last_layer_of<CT, NT>(M) : -1;
  PhaseCache pc;
  build_phase_cache<WS, CT, NT>(M, pc);

  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  if (WS) load_weights_smem<NT>(M, wsm, a.theta);
  __syncthreads();

  auto load_state = [&](float* dst, const float* src, int ld) {  // [S][CT] tile from global (rows of ld floats)
    for (int i = threadIdx.x; i < SC / 4; i += NT) reinterpret_cast<float4*>(dst)[i] = __ldcg(row4<CT>(src, ld, i));
  };
  auto store_state = [&](float* dst, const float* src) {
    for (int i = threadIdx.x; i < SC / 4; i += NT) __stcg(reinterpret_cast<float4*>(dst) + i, reinterpret_cast<const float4*>(src)[i]);
  };
  auto frame_of = [&](int step) -> int {  // saved-frame index of a step, or -1
    if (tm.save_stride <= 0) return step == tm.n_steps ? 0 : -1;
    return (step % tm.save_stride == 0) ? step / tm.save_stride : -1;
  };

  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int col0 = tile * CT;
    const int nvalid = min(CT, a.ncol - col0);
    __syncthreads();
    if (threadIdx.x < CT) {
      const int col = min(col0 + (int)threadIdx.x, a.ncol - 1);
      float raw[6], eff[6];
      for (int j = 0; j < M.nbc; ++j) raw[j] = __ldg(a.bcs + (size_t)col * M.nbc + j);
      bc_effective(M, raw, eff);
      for (int j = 0; j < M.nbc; ++j) bcf[j * CT + threadIdx.x] = eff[j];
      qs[threadIdx.x] = (a.Q != nullptr) ? __ldg(a.Q + col) : 0.f;
    }
    for (int i = threadIdx.x; i < SC; i += NT) xbar[i] = 0.f;
    const int tile32 = col0 / LT, coff = col0 % LT;
    const size_t SL = (size_t)S * LT;  // floats of one state in the global 32-column-tile layout
    const float* ck = a.ckpt + (size_t)tile32 * a.n_ckpt * SL + coff;
    load_state(xs, ck + (size_t)(a.n_ckpt - 1) * SL, LT);  // x_N
    __syncthreads();
    {
      const int fr = frame_of(tm.n_steps);
      if (fr >= 0) {
        load_tile<CT, NT>(xb, xin, bar, parity, (COT ? a.cot : a.targets) + (size_t)fr * S, (size_t)a.n_saved * S, S, col0, a.ncol);
        __syncthreads();
        if constexpr (COT) cot_frame<CT, NT>(M, xb, xbar, nvalid);
        else loss_frame<CT, NT>(M, a, xs, xb, xbar, nvalid, lsum);
        __syncthreads();
      }
    }
    const int cs = tm.ckpt_stride;
    const int nseg = (tm.n_steps + cs - 1) / cs;
    for (int seg = nseg - 1; seg >= 0; --seg) {
      const int n0 = seg * cs, n1 = min(n0 + cs, tm.n_steps);
      const int R = (n1 - n0) * tm.n_substeps;
      load_state(xs, ck + (size_t)seg * SL, LT);
      __syncthreads();
      // ---- forward recompute of the segment's Runge–Kutta step starts (all but the last need a forward step)
      store_state(segx, xs);
      const size_t nrk = (size_t)tm.n_steps * tm.n_substeps;
      const float* kst = a.kstore != nullptr ? a.kstore + ((size_t)tile32 * nrk + (size_t)n0 * tm.n_substeps) * ns * SL + coff : nullptr;
      const KSrc own{slots, CT, (size_t)SC};
      for (int r = 0; r + 1 < R; ++r) {
        const float tb = tm.t0 + (float)(n0 + r / tm.n_substeps) * tm.dt + (float)(r % tm.n_substeps) * h;
        const KSrc kfw = kst != nullptr ? KSrc{kst + (size_t)r * ns * SL, LT, SL} : own;  // stored k_i, or recomputed below
        if (implicit) { implicit_diffusion_tile<CT, NT>(M, xs, imp, h); __syncthreads(); }  // xs: x_r -> y_r
        for (int i = 0; i < ns && kst == nullptr; ++i) {
          const float* in = xs;
          if (i > 0) { stage_input<CT, NT>(tab, i, h, xs, own, SC, xin); __syncthreads(); in = xin; }
          rhs_mlp<CT, NT, WS>(M, pc, in, arena, wsm, a.theta, bcf, qs, tb + tab.c[i] * h);
          float* slot_i = slots + (size_t)i * SC;
          rhs_tendencies<CT, NT, NF>(Mp, in, arena, bcf, [=](int k0, int c, const float (&dx)[NF][4]) {
#pragma unroll
            for (int q = 0; q < NF; ++q)
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) __stcg(slot_i + (q * N + k0 + kk) * CT + c, dx[q][kk]);
          });
          __syncthreads();
        }
        for (int e4 = threadIdx.x; e4 < SC / 4; e4 += NT) {  // x += h sum b_i k_i
          float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
          for (int i = 0; i < ns; ++i) {
            const float bi = tab.b[i];
            const float4 kv = __ldcg(row4<CT>(kfw.p + (size_t)i * kfw.stride, kfw.ld, e4));
            acc.x = fmaf(bi, kv.x, acc.x); acc.y = fmaf(bi, kv.y, acc.y); acc.z = fmaf(bi, kv.z, acc.z); acc.w = fmaf(bi, kv.w, acc.w);
          }
          float4 xv = reinterpret_cast<float4*>(xs)[e4];
          xv.x = fmaf(h, acc.x, xv.x); xv.y = fmaf(h, acc.y, xv.y); xv.z = fmaf(h, acc.z, xv.z); xv.w = fmaf(h, acc.w, xv.w);
          reinterpret_cast<float4*>(xs)[e4] = xv;
          __stcg(reinterpret_cast<float4*>(segx + (size_t)(r + 1) * SC) + e4, xv);
        }
        __syncthreads();
      }
      // ---- reverse sweep over the segment
      for (int r = R - 1; r >= 0; --r) {
        if (R > 1 || implicit) { load_state(xs, segx + (size_t)r * SC, CT); __syncthreads(); }
        if (implicit) { implicit_diffusion_tile<CT, NT>(M, xs, imp, h); __syncthreads(); }  // the explicit stages start from y_r
        const int nstep = n0 + r / tm.n_substeps, sub = r % tm.n_substeps;
        const float tb = tm.t0 + (float)nstep * tm.dt + (float)sub * h;
        // (a) forward stages 0..ns-2 -> k_i into the slots
        const long long pa0 = CPZ_APROF_T();
        const KSrc kfw = kst != nullptr ? KSrc{kst + (size_t)r * ns * SL, LT, SL} : own;
        for (int i = 0; i + 1 < ns && kst == nullptr; ++i) {
          const float* in = xs;
          if (i > 0) { stage_input<CT, NT>(tab, i, h, xs, own, SC, xin); __syncthreads(); in = xin; }
          rhs_mlp<CT, NT, WS>(M, pc, in, arena, wsm, a.theta, bcf, qs, tb + tab.c[i] * h);
          float* slot_i = slots + (size_t)i * SC;
          rhs_tendencies<CT, NT, NF>(Mp, in, arena, bcf, [=](int k0, int c, const float (&dx)[NF][4]) {
#pragma unroll
            for (int q = 0; q < NF; ++q)
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) __stcg(slot_i + (q * N + k0 + kk) * CT + c, dx[q][kk]);
          });
          __syncthreads();
        }
        CPZ_APROF_ADD(0, pa0);
        // (b) reverse stages
        for (int i = ns - 1; i >= 0; --i) {
          const long long pb0 = CPZ_APROF_T();
          const float* in = xs;
          if (i > 0) { stage_input<CT, NT>(tab, i, h, xs, kfw, SC, xin); in = xin; }
          // kbar_i = h (b_i xbar + sum_{j>i} a_ji Xbar_j)   (slots j>i hold Xbar_j)
          for (int e4 = threadIdx.x; e4 < SC / 4; e4 += NT) {
            const float bi = tab.b[i];
            const float4 xv = reinterpret_cast<const float4*>(xbar)[e4];
            float4 acc = make_float4(bi * xv.x, bi * xv.y, bi * xv.z, bi * xv.w);
            for (int j = i + 1; j < ns; ++j) {
              const float aji = tab.a[j][i];
              if (aji != 0.f) {
                const float4 kv = __ldcg(reinterpret_cast<const float4*>(slots + (size_t)j * SC) + e4);
                acc.x = fmaf(aji, kv.x, acc.x); acc.y = fmaf(aji, kv.y, acc.y); acc.z = fmaf(aji, kv.z, acc.z); acc.w = fmaf(aji, kv.w, acc.w);
              }
            }
            reinterpret_cast<float4*>(xb)[e4] = make_float4(h * acc.x, h * acc.y, h * acc.z, h * acc.w);
          }
          if (M.flags & F_DIURNAL) {
            if (threadIdx.x < CT) bcf[(M.nbc - 1) * CT + threadIdx.x] = diurnal_top_eff(M, qs[threadIdx.x], tb + tab.c[i] * h);
          }
          __syncthreads();
          CPZ_APROF_ADD(1, pb0);
          const long long pb1 = CPZ_APROF_T();
          mlp_forward_keep<CT, NT, WS>(M, Lmax, pc, in, arena, zarena, wsm, a.theta);
          CPZ_APROF_ADD(2, pb1);
          const long long pb2 = CPZ_APROF_T();
          faces_vjp<CT, NT>(M, in, xb, zarena, gflux, a.want_pgrad ? pgs : nullptr);
          __syncthreads();
          centres_vjp<CT, NT>(M, xb, gflux);
          __syncthreads();
          CPZ_APROF_ADD(3, pb2);
          for (int l = Lmax; l >= 0; --l) {
            const long long pb3 = CPZ_APROF_T();
            mlp_backward_layer<WS, CT, NT>(M, l, in, arena, zarena, xb, wsm, a.theta, gpart);
            __syncthreads();
            CPZ_APROF_ADD(4 + (l < 2 ? l : 2), pb3);
          }
          const long long pb4 = CPZ_APROF_T();
          store_state(slots + (size_t)i * SC, xb);  // slot i now holds Xbar_i
          __syncthreads();
          CPZ_APROF_ADD(1, pb4);
        }
        // xbar_n = xbar_{n+1} + sum_i Xbar_i
        for (int e4 = threadIdx.x; e4 < SC / 4; e4 += NT) {
          float4 acc = reinterpret_cast<float4*>(xbar)[e4];
          for (int i = 0; i < ns; ++i) {
            const float4 kv = __ldcg(reinterpret_cast<const float4*>(slots + (size_t)i * SC) + e4);
            acc.x += kv.x; acc.y += kv.y; acc.z += kv.z; acc.w += kv.w;
          }
          reinterpret_cast<float4*>(xbar)[e4] = acc;
        }
        __syncthreads();
        if (implicit) {
          // xbar is the cotangent of y_r; pull it back through y_r = L(D(x_r)) \ x_r. x_r is re-read from the segment scratch.
          load_state(xin, segx + (size_t)r * SC, CT);
          __syncthreads();
          implicit_vjp_tile<CT, NT>(M, xin, xs, xbar, imp, gflux, h, a.want_pgrad ? pgs : nullptr);
          __syncthreads();
          if (sub == 0 && frame_of(nstep) >= 0) {  // the saved frame is x_r, not y_r
            load_state(xs, segx + (size_t)r * SC, CT);
            __syncthreads();
          }
        }
        if (sub == 0) {
          const int fr = frame_of(nstep);
          if (fr >= 0) {
            load_tile<CT, NT>(xb, xin, bar, parity, (COT ? a.cot : a.targets) + (size_t)fr * S, (size_t)a.n_saved * S, S, col0, a.ncol);
            __syncthreads();
            if constexpr (COT) cot_frame<CT, NT>(M, xb, xbar, nvalid);
            else loss_frame<CT, NT>(M, a, xs, xb, xbar, nvalid, lsum);
            __syncthreads();
          }
        }
      }
    }
    if (COT && a.x0bar != nullptr) {  // xbar is now the cotangent of x0
      __syncthreads();
      store_tile<CT, NT>(xbar, xin, a.x0bar, (size_t)S, S, col0, a.ncol);
      if (threadIdx.x < CT) bulk_wait_read0();  // xin is the next tile's staging buffer
    }
  }
  if (COT && a.x0bar != nullptr && threadIdx.x < CT) bulk_wait0();
  // block reduction of the six loss sums and the five mPP-parameter gradient sums
  for (int q = 0; q < 11; ++q) {
    double vd = q < 6 ? (double)lsum[q] : pgs[q - 6];
    for (int o = 16; o > 0; o >>= 1) vd += __shfl_xor_sync(0xffffffffu, vd, o);
    float v = (float)vd;
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      float s = 0.f;
      for (int wdx = 0; wdx < NT / 32; ++wdx) s += red[wdx];
      a.lpart[(size_t)blockIdx.x * LP + (q < 6 ? q : LP / 2 + q - 6)] = s;
    }
    __syncthreads();
  }
}

template <int CT, int NT, bool WS, bool COT>
__global__ void __launch_bounds__(NT, 1) adjoint_kernel(const __grid_constant__ ModelD Mp, const __grid_constant__ TableauD tab,
                                                        const TimeD tm, const __grid_constant__ AdjArgs a) {
  extern __shared__ __align__(16) float smem[];
  const AdjSmem L = adjoint_smem_layout(Mp, CT);
  const ModelD& M = model_to_smem<NT>(Mp, smem + L.model);
  if (Mp.nf == 3) adjoint_body<CT, NT, WS, 3, COT>(M, Mp, tab, tm, a, smem);
  else adjoint_body<CT, NT, WS, 1, COT>(M, Mp, tab, tm, a, smem);
}

struct W6 { float w[6]; };

}  // namespace cpz
