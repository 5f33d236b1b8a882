// Pullback of the right-hand side (cpz_rhs_vjp): for every column c of a batch
//   x_bar[c] = (df/dx)^T(x_c) ybar_c,   theta_bar += (df/dtheta)^T(x_c) ybar_c,   p_bar += (df/dp)^T(x_c) ybar_c,
// p = (nu0, nu_m, dRi, Ric, Pr). This is one reverse stage of adjoint_body (cpz_adjoint.cuh) without the Runge–Kutta
// bookkeeping, built from the same device functions: MLP forward keeping a and z, faces_vjp, centres_vjp,
// mlp_backward_layer. It lets a host that runs its own time stepper (adaptive Tsit5 / ROCK4 with InterpolatingAdjoint,
// a continuous adjoint) differentiate through cpz_rhs.
//
// The boundary fluxes, the diurnal amplitudes and t enter f additively (the two boundary faces of every field), so the
// cotangents wrt x, theta and p do not depend on them and the kernel does not read them.
#pragma once
#include "cpz_adjoint.cuh"

namespace cpz {

struct VjpArgs {
  const float* theta;
  const float* x;     // [ncol][S]
  const float* ybar;  // [ncol][S] cotangent of dx/dt
  float* xbar;        // [ncol][S] or null
  float* gpart;       // [grid][M.slab] weight-gradient slabs in tile layout (zeroed by the host)
  float* lpart;       // [grid][LP]: the five mPP-parameter sums at LP/2 .. LP/2+4 (zeroed by the host)
  int want_mlp;       // x_bar or theta_bar requested: run the MLP forward and backward
  int want_pgrad;     // accumulate the five mPP-parameter sums
  int ncol, n_tiles;
};

template <int CT, int NT, bool WS>
__global__ void __launch_bounds__(NT, 1) rhs_vjp_kernel(const __grid_constant__ ModelD Mp, const __grid_constant__ VjpArgs a) {
  extern __shared__ __align__(16) float smem[];
  const AdjSmem L = adjoint_smem_layout(Mp, CT);
  const ModelD& M = model_to_smem<NT>(Mp, smem + L.model);
  float* wsm = smem + L.w;
  float* xs = smem + L.xs;     // x
  float* xin = smem + L.xin;   // transpose staging of the bulk copies
  float* xb = smem + L.xb;     // ybar, then x_bar
  float* arena = smem + L.arena;
  float* zarena = smem + L.zarena;
  float* red = smem + L.red;
  float* gflux = arena + M.flux_off * CT;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + ((L.total_floats - 4 + 1) & ~1));
  const int S = M.S, N = M.Nz;
  float* gpart = a.gpart + (size_t)blockIdx.x * M.slab;
  uint32_t parity = 0;
  double pgs[5] = {0., 0., 0., 0., 0.};  // FP64 accumulators, as in adjoint_body
  const int Lmax = M.n_gemm > 0 ? last_layer_of<CT, NT>(M) : -1;
  PhaseCache pc;
  build_phase_cache<WS, CT, NT>(M, pc);

  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  if (WS && a.want_mlp) load_weights_smem<NT>(M, wsm, a.theta);
  __syncthreads();

  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int col0 = tile * CT;
    const int nvalid = min(CT, a.ncol - col0);
    __syncthreads();
    load_tile<CT, NT>(xs, xin, bar, parity, a.x, (size_t)S, S, col0, a.ncol);
    __syncthreads();
    load_tile<CT, NT>(xb, xin, bar, parity, a.ybar, (size_t)S, S, col0, a.ncol);
    __syncthreads();
    // columns past ncol replicate the last valid one: a zero cotangent keeps them out of theta_bar and p_bar
    for (int i = threadIdx.x; i < N * CT; i += NT) {
      const int c = i % CT;
      if (c >= nvalid)
        for (int q = 0; q < M.nf; ++q) xb[q * N * CT + i] = 0.f;
    }
    __syncthreads();
    // MLP forward keeping z and a (the last layer's outputs are not needed: f is linear in them)
    if (a.want_mlp) {
      for (int p = 0; p < M.n_phase; ++p) {
        if (M.gemm[M.phase[p].g0].layer == Lmax && M.gemm[M.phase[p].g1 - 1].layer == Lmax) continue;
        run_phase_cached<CT, NT, WS, true>(M, p, pc, xs, arena, zarena, wsm, a.theta);
        __syncthreads();
      }
    }
    faces_vjp<CT, NT>(M, xs, xb, zarena, gflux, a.want_pgrad ? pgs : nullptr);
    __syncthreads();
    centres_vjp<CT, NT>(M, xb, gflux);
    __syncthreads();
    if (a.want_mlp) {
      for (int l = Lmax; l >= 0; --l) {
        mlp_backward_layer<WS, CT, NT>(M, l, xs, arena, zarena, xb, wsm, a.theta, gpart);
        __syncthreads();
      }
    }
    if (a.xbar != nullptr) {
      store_tile<CT, NT>(xb, xin, a.xbar, (size_t)S, S, col0, a.ncol);
      if (threadIdx.x < CT) bulk_wait_read0();  // xin is the next tile's staging buffer
    }
  }
  if (a.xbar != nullptr && threadIdx.x < CT) bulk_wait0();
  if (!a.want_pgrad) return;
  // block reduction of the five mPP-parameter sums (fixed order)
  for (int q = 0; q < 5; ++q) {
    double vd = pgs[q];
    for (int o = 16; o > 0; o >>= 1) vd += __shfl_xor_sync(0xffffffffu, vd, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = (float)vd;
    __syncthreads();
    if (threadIdx.x == 0) {
      float s = 0.f;
      for (int wdx = 0; wdx < NT / 32; ++wdx) s += red[wdx];
      a.lpart[(size_t)blockIdx.x * LP + LP / 2 + q] = s;
    }
    __syncthreads();
  }
}

}  // namespace cpz
