// Pullback of the gyre closure step (cpz_closure_step_vjp): for the cotangents Fbar of the forcing and Ybar of T' of
// closure_kernel, per column
//   T_bar = A^-T (Ybar + (dNN/dx)^T nbar / (T_div sig_T) - mu_relax Fbar[N-1] / dz e_{N-1}),   theta_bar += (dNN/dtheta)^T nbar,
//   nbar_j = sig_wT (Fbar_j - Fbar_{j+1}) / dz   (NN output j sits at face j + 1),
// where T' = A^-1 T is the implicit convective adjustment (oracle/nde.py: closure_step). A is symmetric (lower[k+1] =
// upper[k] = -r kappa_{k+1}), so A^-T = A^-1: one more Thomas solve with the forward's coefficients. kappa is piecewise
// constant in T: at the switch the derivative is that of the branch the forward evaluated, as at relu kinks. y, T_mid, dT
// and Ly enter the forcing additively and drop out.
// The MLP runs in FP32 SIMT on the adjoint plan with the device functions of the discrete adjoint (mlp_forward_keep,
// mlp_backward); the last layer's forward is skipped, because the forcing is affine in the NN outputs.
#pragma once
#include "cpz_adjoint.cuh"
#include "cpz_closure.cuh"

namespace cpz {

struct ClosureVjpArgs {
  const float* theta;
  const float* T;      // [Nz][ncol] incoming temperature
  const float* f_bar;  // [Nz][ncol] cotangent of the forcing, or null (zero)
  const float* y_bar;  // [Nz][ncol] cotangent of T', or null (zero)
  float* T_bar;        // [Nz][ncol] or null
  float* gpart;        // [grid][M.slab] weight-gradient slabs in tile layout (zeroed by the host)
  int want_mlp;        // f_bar given and T_bar or theta_bar requested: run the adjustment, the MLP forward and backward
  int ncol, n_tiles;
};

// Rows of the Thomas c' scratch, which lives in the activation arena and zarena (contiguous, dead outside the MLP).
__host__ __device__ inline int closure_vjp_scratch_rows(int Nz) { return Nz; }

// Thomas forward sweep of the adjustment matrix A(T) of column c (closure_kernel's statements, so that the coefficients are
// bitwise the forward's) for the right-hand side rhs: c' into cp, d' into d (d may alias rhs). tt: incoming T.
template <int CT>
__device__ __forceinline__ void adjustment_sweep(const ClosureD& cd, int N, int c, const float* tt, const float* rhs, float* cp,
                                                 float* d) {
  auto G = [&](int f) -> float { return (f <= 0 || f >= N) ? 0.f : (tt[f * CT + c] - tt[(f - 1) * CT + c]) * cd.inv_dz; };
  auto kap = [&](int k) -> float { return (0.5f * (G(k) + G(k + 1)) < 0.f) ? cd.K : 0.f; };
  float kk = kap(0), kn = kap(1);
  float diag = 1.f + cd.r * (kk + kn);
  float up = -cd.r * kn;
  float cprev = up / diag;
  float dprev = rhs[c] / diag;
  cp[c] = cprev;
  d[c] = dprev;
  for (int k = 1; k < N; ++k) {
    kk = kn;
    kn = (k + 1 < N) ? kap(k + 1) : 0.f;
    const float lo = -cd.r * kk;
    diag = (k < N - 1) ? 1.f + cd.r * (kk + kn) : 1.f + cd.r * kk;
    up = (k < N - 1) ? -cd.r * kn : 0.f;
    const float den = diag - lo * cprev;
    cprev = up / den;
    dprev = (rhs[k * CT + c] - lo * dprev) / den;
    cp[k * CT + c] = cprev;
    d[k * CT + c] = dprev;
  }
}

template <int CT, int NT, bool WS>
__global__ void __launch_bounds__(NT, 1) closure_vjp_kernel(const __grid_constant__ ModelD Mp, const __grid_constant__ ClosureD cd,
                                                            const __grid_constant__ ClosureVjpArgs a) {
  extern __shared__ __align__(16) float smem[];
  const AdjSmem L = adjoint_smem_layout(Mp, CT);
  const ModelD& M = model_to_smem<NT>(Mp, smem + L.model);
  const int N = M.Nz;
  float* wsm = smem + L.w;
  float* xs = smem + L.xs;      // adjustment d', then the scaled NN input x
  float* tt = smem + L.xbar;    // incoming T (the adjustment's coefficients are recomputed from it)
  float* lam = smem + L.xin;    // Ybar and the surface-flux term -> T'bar -> lambda = A^-1 T'bar
  float* xb = smem + L.xb;      // Fbar; then the cotangent of x
  float* arena = smem + L.arena;
  float* zarena = smem + L.zarena;
  float* cps = arena;           // [N][CT] Thomas c' (dead rows of the arena outside the MLP)
  float* gpart = a.gpart + (size_t)blockIdx.x * M.slab;
  const int Lmax = last_layer_of<CT, NT>(M);
  const float dxdT = cd.inv_T_div * cd.inv_sig_T;  // d x / d T'
  PhaseCache pc;
  build_phase_cache<WS, CT, NT>(M, pc);
  if (WS && a.want_mlp) load_weights_smem<NT>(M, wsm, a.theta);
  __syncthreads();

  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int col0 = tile * CT;
    __syncthreads();
    // coalesced loads: row k of the tile = CT consecutive floats of level k. Columns past ncol replicate the last valid one
    // with zero cotangents, which keeps them out of theta_bar.
    for (int i = threadIdx.x; i < N * CT; i += NT) {
      const int k = i / CT, c = i - k * CT;
      const bool live = col0 + c < a.ncol;
      const size_t g = (size_t)k * a.ncol + min(col0 + c, a.ncol - 1);
      tt[i] = __ldg(a.T + g);
      const float fb = (a.f_bar != nullptr && live) ? __ldg(a.f_bar + g) : 0.f;
      const float yb = (a.y_bar != nullptr && live) ? __ldg(a.y_bar + g) : 0.f;
      xb[i] = fb;
      // wT[N] = -mu_relax (T'[N-1] - T_ref): forcing[N-1] = (wT[N] - wT[N-1]) / dz
      lam[i] = k == N - 1 ? yb - cd.mu_relax * (fb * cd.inv_dz) : yb;
    }
    __syncthreads();
    if (a.want_mlp) {
      // the adjustment, one thread per column; the back substitution writes the NN input straight from T'
      if (threadIdx.x < CT) {
        const int c = threadIdx.x;
        adjustment_sweep<CT>(cd, N, c, tt, tt, cps, xs);
        float tn = 0.f;
        for (int k = N - 1; k >= 0; --k) {
          tn = k == N - 1 ? xs[k * CT + c] : xs[k * CT + c] - cps[k * CT + c] * tn;
          xs[k * CT + c] = ((cd.T_shift + tn * cd.inv_T_div) - cd.mu_T) * cd.inv_sig_T;
        }
      }
      __syncthreads();
      mlp_forward_keep<CT, NT, WS>(M, Lmax, pc, xs, arena, zarena, wsm, a.theta);
      // cotangent of the NN outputs: wT[j + 1] = sig_wT nn_j + mu_wT, forcing_k = (wT[k + 1] - wT[k]) / dz
      for (int i = threadIdx.x; i < (N - 1) * CT; i += NT) {
        const int j = i / CT, c = i - j * CT;
        zarena[(M.nn_off[0] + j) * CT + c] = cd.sig_wT * ((xb[j * CT + c] - xb[(j + 1) * CT + c]) * cd.inv_dz);
      }
      __syncthreads();
      for (int i = threadIdx.x; i < N * CT; i += NT) xb[i] = 0.f;
      __syncthreads();
      mlp_backward<CT, NT, WS>(M, Lmax, xs, arena, zarena, xb, wsm, a.theta, gpart);
    }
    if (a.T_bar == nullptr) continue;
    // T'bar, then lambda = A^-1 T'bar with the adjustment's coefficients (one thread per column), in place
    if (a.want_mlp)
      for (int i = threadIdx.x; i < N * CT; i += NT) lam[i] += xb[i] * dxdT;
    __syncthreads();
    if (threadIdx.x < CT) {
      const int c = threadIdx.x;
      adjustment_sweep<CT>(cd, N, c, tt, lam, cps, lam);
      float ln = lam[(N - 1) * CT + c];
      for (int k = N - 2; k >= 0; --k) {
        ln = lam[k * CT + c] - cps[k * CT + c] * ln;
        lam[k * CT + c] = ln;
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < N * CT; i += NT) {
      const int k = i / CT, c = i - k * CT;
      if (col0 + c < a.ncol) a.T_bar[(size_t)k * a.ncol + col0 + c] = lam[i];
    }
  }
}

}  // namespace cpz
