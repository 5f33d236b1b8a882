// Pullback of the embedded u/v/T closure step (cpz_closure_step_uvt_vjp): for the cotangents Dbar of dz_flux and Ybar of
// (u', v', T') of closure_uvt_kernel, per column
//   (u, v, T)_bar = L^-T Ybar + (dL/dx)^T ... (mPP step)  +  (dNN/dx)^T (forcing),   theta_bar += (dNN/dtheta)^T (forcing),
//   p_bar += (dL/dp)^T ... (mPP step),   p = (nu0, nu_m, dRi, Ric, Pr).
// The step's two outputs depend on the incoming state through separate paths (oracle/nde.py: closure_step_uvt): dz_flux is
// the transposed face difference of the NN forcing chains, (u', v', T') = L(nu(x))^-1 x is the backward-Euler mPP step of the
// incoming state (the host applies the forcing itself), with T'[bottom] = T[bottom] and nu = 0 on the two boundary faces.
// Reverse of the step, with L symmetric:
//   lambda = L^-1 Ybar (T: Ybar[bottom] goes straight to T_bar[bottom], the solve sees 0 there),
//   nubar_f = -r (lambda_f - lambda_{f-1}) (y_f - y_{f-1})   (y: the solve's output, before the T'[bottom] override),
//   then the diffusivity chain nu(Ri), nu_T = Ri > 0 ? nu/Pr : kappa_ca, Ri = g alpha T_z / (u_z^2 + v_z^2) back to the state.
// Everything is dimensional, with the closure's own dz and dt, as in closure_uvt_kernel; the MLP runs on the adjoint plan with
// the device functions of the discrete adjoint (mlp_forward_keep, mlp_backward).
// At relu kinks and at the convective-adjustment switch the derivative is that of the branch the forward evaluated.
#pragma once
#include "cpz_adjoint.cuh"
#include "cpz_closure_uvt.cuh"

namespace cpz {

struct ClosureUvtVjpArgs {
  const float* theta;
  const float* f[3];     // u, v, T: [Nz][ncol]
  const float* dzf_bar;  // [3][Nz][ncol] cotangent of dz_flux, or null (zero)
  const float* out_bar;  // [3][Nz][ncol] cotangent of (u', v', T'), or null (zero)
  float* fbar[3];        // u_bar, v_bar, T_bar: [Nz][ncol], each may be null
  float* gpart;          // [grid][M.slab] weight-gradient slabs in tile layout (zeroed by the host)
  float* lpart;          // [grid][LP]: the five mPP-parameter sums at LP/2 .. LP/2+4 (zeroed by the host)
  int want_mlp;          // dzf_bar given and a state or theta cotangent requested: run the MLP forward and backward
  int want_imp;          // out_bar given and a state or mPP cotangent requested: reverse the mPP step
  int want_pgrad;        // accumulate the five mPP-parameter sums
  int ncol, n_tiles;
};

// Rows of the mPP-step scratch, which lives in the activation arena and zarena (contiguous, dead until the MLP forward):
// nu, nu_T (2 Nz), Thomas c' then the face-gradient cotangents (3 Nz), the solve's increments y - x (3 Nz).
__host__ __device__ inline int closure_uvt_vjp_scratch_rows(int Nz) { return 8 * Nz; }

template <int CT, int NT, bool WS>
__global__ void __launch_bounds__(NT, 1) closure_uvt_vjp_kernel(const __grid_constant__ ModelD Mp, const __grid_constant__ ClosureUvtD cd,
                                                                const __grid_constant__ ClosureUvtVjpArgs a) {
  extern __shared__ __align__(16) float smem[];
  const AdjSmem L = adjoint_smem_layout(Mp, CT);
  const ModelD& M = model_to_smem<NT>(Mp, smem + L.model);
  const int N = M.Nz;
  float* wsm = smem + L.w;
  float* xs = smem + L.xs;     // scaled NN input
  float* st = smem + L.xbar;   // incoming u, v, T (dimensional)
  float* lam = smem + L.xin;   // Ybar -> lambda -> cotangent of the state through the mPP step
  float* xb = smem + L.xb;     // Dbar; then the cotangent of the scaled NN input
  float* arena = smem + L.arena;
  float* zarena = smem + L.zarena;
  float* nus = arena;          // [2][N][CT]: nu, nu_T of face f at row f (face 0 unused)
  float* cps = arena + 2 * N * CT;  // [3][N][CT]: Thomas c'; then the face-gradient cotangents (row q N + f)
  float* incs = arena + 5 * N * CT; // [3][N][CT]: y - x
  float* yb0 = smem + L.qs;    // [CT]: cotangent of T'[bottom]
  float* red = smem + L.red;
  float* gpart = a.gpart + (size_t)blockIdx.x * M.slab;
  double pgs[5] = {0., 0., 0., 0., 0.};
  const int Lmax = M.n_gemm > 0 ? last_layer_of<CT, NT>(M) : -1;
  PhaseCache pc;
  build_phase_cache<WS, CT, NT>(M, pc);
  if (WS && a.want_mlp) load_weights_smem<NT>(M, wsm, a.theta);
  __syncthreads();

  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int col0 = tile * CT;
    __syncthreads();
    // coalesced loads: row (q, k) of the tile = CT consecutive floats of field q at level k. Columns past ncol replicate the
    // last valid one with zero cotangents, which keeps them out of theta_bar and p_bar.
    for (int i = threadIdx.x; i < 3 * N * CT; i += NT) {
      const int row = i / CT, c = i - row * CT;
      const int q = row / N;
      const bool live = col0 + c < a.ncol;
      const size_t g = (size_t)row * a.ncol + min(col0 + c, a.ncol - 1);
      const float v = __ldg(a.f[q] + (g - (size_t)q * N * a.ncol));
      st[i] = v;
      xs[i] = (v - cd.mu[q]) * cd.inv_sig[q];
      lam[i] = (a.out_bar != nullptr && live) ? __ldg(a.out_bar + g) : 0.f;
      xb[i] = (a.dzf_bar != nullptr && live) ? __ldg(a.dzf_bar + g) : 0.f;
    }
    __syncthreads();
    if (a.want_imp) {
      // face diffusivities of the incoming state (closure_uvt_kernel's statements)
      for (int i = threadIdx.x; i < (N - 1) * CT; i += NT) {
        const int f = 1 + i / CT, c = i - (f - 1) * CT;
        const float du = (st[f * CT + c] - st[(f - 1) * CT + c]) * cd.inv_dz;
        const float dv = (st[(N + f) * CT + c] - st[(N + f - 1) * CT + c]) * cd.inv_dz;
        const float dT = (st[(2 * N + f) * CT + c] - st[(2 * N + f - 1) * CT + c]) * cd.inv_dz;
        const float Ri = cd.g_alpha * dT * uvt_rcp(du * du + dv * dv);
        const float nu = cd.nu0 + cd.nu_m * (0.5f * (1.f - tanhf((Ri - cd.Ric) * cd.inv_dRi)));
        nus[f * CT + c] = nu;
        nus[(N + f) * CT + c] = (cd.ca && !(Ri > 0.f)) ? cd.kappa_ca : nu * cd.inv_Pr;
      }
      __syncthreads();
      // one thread per (field, column): the forward sweep of the step (increment form, as closure_uvt_kernel) and of
      // lambda = L^-1 Ybar share the coefficients; then both back substitutions
      if (threadIdx.x < 3 * CT) {
        const int q = threadIdx.x / CT, c = threadIdx.x - q * CT;
        const float* sq = st + q * N * CT + c;
        const float* nv = nus + (q == 2 ? N * CT : 0) + c;
        float* cpv = cps + q * N * CT + c;
        float* inv = incs + q * N * CT + c;
        float* lv = lam + q * N * CT + c;
        if (q == 2) {  // T'[bottom] = T[bottom] (:93): its cotangent bypasses the solve
          yb0[c] = lv[0];
          lv[0] = 0.f;
        }
        auto nuq = [&](int f) -> float { return (f <= 0 || f >= N) ? 0.f : nv[f * CT]; };
        float nk = nuq(0), nn1 = nuq(1);
        float diag = 1.f + cd.r * (nk + nn1);
        float cprev = uvt_div(-cd.r * nn1, diag);
        float xk = sq[0], xup = sq[CT];
        float dprev = uvt_div(cd.r * nn1 * (xup - xk), diag);
        float lprev = uvt_div(lv[0], diag);
        cpv[0] = cprev;
        inv[0] = dprev;
        lv[0] = lprev;
        for (int k = 1; k < N; ++k) {
          nk = nn1;
          nn1 = nuq(k + 1);
          const float xdn = xk;
          xk = xup;
          xup = k + 1 < N ? sq[(k + 1) * CT] : xk;
          const float lo = -cd.r * nk;
          diag = 1.f + cd.r * (nk + nn1);
          const float den = diag - lo * cprev;
          cprev = uvt_div(-cd.r * nn1, den);
          dprev = uvt_div(cd.r * (nk * (xdn - xk) + nn1 * (xup - xk)) - lo * dprev, den);
          lprev = uvt_div(lv[k * CT] - lo * lprev, den);
          cpv[k * CT] = cprev;
          inv[k * CT] = dprev;
          lv[k * CT] = lprev;
        }
        float dn = dprev, ln = lprev;
        for (int k = N - 2; k >= 0; --k) {
          dn = inv[k * CT] - cpv[k * CT] * dn;
          ln = lv[k * CT] - cpv[k * CT] * ln;
          inv[k * CT] = dn;
          lv[k * CT] = ln;
        }
      }
      __syncthreads();
      // cotangents of the face diffusivities, then through nu(Ri) and Ri(u_z, v_z, T_z) to the face gradients
      for (int i = threadIdx.x; i < (N - 1) * CT; i += NT) {
        const int f = 1 + i / CT, c = i - (f - 1) * CT;
        float nb[3], G[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          const int e = (q * N + f) * CT + c;
          G[q] = (st[e] - st[e - CT]) * cd.inv_dz;
          // y_f - y_{f-1} from the state and the increments: the rounding stays relative to the increment
          const float dy = (st[e] - st[e - CT]) + (incs[e] - incs[e - CT]);
          nb[q] = -cd.r * (lam[e] - lam[e - CT]) * dy;
        }
        const float S2 = G[0] * G[0] + G[1] * G[1];
        const float iS2 = uvt_rcp(S2);
        const float Ri = cd.g_alpha * G[2] * iS2;
        const float yv = (Ri - cd.Ric) * cd.inv_dRi;
        const float th = tanhf(yv);
        const float s = 0.5f * (1.f - th);
        const float nu = cd.nu0 + cd.nu_m * s;
        const bool kap = cd.ca && !(Ri > 0.f);  // nu_T = kappa_ca: no dependence on nu or Pr
        const float nub = nb[0] + nb[1] + (kap ? 0.f : nb[2] * cd.inv_Pr);
        const float sech2 = (1.f - th) * (1.f + th);  // 0 where the step is saturated (zero shear: Ri = +-inf)
        const float dnu = -0.5f * cd.nu_m * sech2 * cd.inv_dRi;  // d nu / d Ri
        if (a.want_pgrad) {
          // d nu/d(nu0, nu_m, dRi, Ric) and d nu_T/d Pr = -nu/Pr^2 (the same parameters as cpz_loss_grad_mpp)
          pgs[0] += nub;
          pgs[1] += nub * s;
          if (sech2 != 0.f) {
            pgs[2] += -nub * dnu * yv;
            pgs[3] += -nub * dnu;
          }
          if (!kap) pgs[4] -= nb[2] * nu * cd.inv_Pr * cd.inv_Pr;
        }
        const float Rib = nub * dnu;
        float gb[3] = {0.f, 0.f, 0.f};
        if (Rib != 0.f) {
          gb[2] = Rib * cd.g_alpha * iS2;
          const float t = -2.f * Rib * Ri * iS2;
          gb[0] = t * G[0];
          gb[1] = t * G[1];
        }
#pragma unroll
        for (int q = 0; q < 3; ++q) cps[(q * N + f) * CT + c] = gb[q] * cd.inv_dz;
      }
      __syncthreads();
      // transpose of the face gradient at the centres, plus the bypass of T'[bottom]
      for (int i = threadIdx.x; i < 3 * N * CT; i += NT) {
        const int row = i / CT, c = i - row * CT;
        const int q = row / N, k = row - q * N;
        const float g0 = k >= 1 ? cps[(q * N + k) * CT + c] : 0.f;
        const float g1 = k + 1 <= N - 1 ? cps[(q * N + k + 1) * CT + c] : 0.f;
        lam[i] += (g0 - g1) + ((q == 2 && k == 0) ? yb0[c] : 0.f);
      }
      __syncthreads();
    }
    if (a.want_mlp) {
      mlp_forward_keep<CT, NT, WS>(M, Lmax, pc, xs, arena, zarena, wsm, a.theta);
      // cotangent of the NN outputs: F = [0; sig (nn_j) + mu - shift; top], dz_flux = D_c F / dz, shift = the first unscaled
      // output, unscaled once more for momentum (:292,301, literal) and as is for temperature (:324)
      for (int i = threadIdx.x; i < 3 * (N - 1) * CT; i += NT) {
        const int row = i / CT, c = i - row * CT;
        const int q = row / (N - 1), j = row - q * (N - 1);
        const float* Db = xb + q * N * CT + c;
        const float sg = cd.sig[3 + q];
        float fb = (Db[j * CT] - Db[(j + 1) * CT]) * cd.inv_dz;  // cotangent of F at face j + 1
        if (j == 0) fb -= (q < 2 ? sg : 1.f) * (Db[0] - Db[(N - 1) * CT]) * cd.inv_dz;  // shift: minus the sum over faces 1..N-1
        zarena[(M.nn_off[q] + j) * CT + c] = sg * fb;
      }
      __syncthreads();
      for (int i = threadIdx.x; i < 3 * N * CT; i += NT) xb[i] = 0.f;
      __syncthreads();
      mlp_backward<CT, NT, WS>(M, Lmax, xs, arena, zarena, xb, wsm, a.theta, gpart);
    }
    // row stores of u_bar, v_bar, T_bar: the mPP-step part plus the NN-input part unscaled
    for (int i = threadIdx.x; i < 3 * N * CT; i += NT) {
      const int row = i / CT, c = i - row * CT;
      const int q = row / N, k = row - q * N;
      if (a.fbar[q] == nullptr || col0 + c >= a.ncol) continue;
      a.fbar[q][(size_t)k * a.ncol + col0 + c] = lam[i] + (a.want_mlp ? xb[i] * cd.inv_sig[q] : 0.f);
    }
  }
  if (a.want_pgrad) store_pgrad_sums<NT>(pgs, red, a.lpart);
}

}  // namespace cpz
