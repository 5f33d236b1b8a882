// Tensor-core discrete adjoint of the u/v/T NDE solve (tcgen05 / UTCHMMA, 3xTF32), sm_100a.
//
// Replaces Zygote/DiffEqSensitivity's InterpolatingAdjoint(autojacvec=ZygoteVJP()) at wind_mixing/src/NDE_training.jl:291,304
// for the models the tcgen05 forward solve covers (cpz_k_tc.cu: three Dense(96,h1) -> Dense(h1,h2) -> Dense(h2,31) chains).
// The reverse sweep of one checkpoint segment runs as three kernels that exchange per-stage records through HBM (AuxD,
// cpz_solve.cuh) because forward weights, transposed weights and weight-gradient accumulators do not fit 512 TMEM columns
// together:
//   1. solve_tc_kernel<..., AUX>  (cpz_tc.cuh)   re-integrates the segment from its checkpoint with the FORWARD weight image
//      in tensor memory and stores, per stage evaluation, the stage input X_i and the pre-activations z1, z2.
//   2. adjoint_tc_kernel          (this file)    walks the segment backwards with the TRANSPOSED weight images in tensor
//      memory: kbar_i = h (b_i xbar + sum_{j>i} a_ji Xbar_j); VJP of the stencil / Richardson-number diffusivities in
//      registers + shuffles (lane <-> level); delta3 -> delta2 in FP32 (620 MACs per net and column); delta2 -> delta1 and
//      delta1 -> Xbar on tcgen05 (D = W delta, weights = M side from TMEM, 16 columns = N side); stores delta1..3.
//   3. wgrad_tc_kernel            (this file)    the weight gradient is one long contraction over (column, stage):
//      dW1 += [X;1] delta1^T, dW2 += [a1;1] delta2^T, dW3 += [a2;1] delta3^T with K = 32 columns per record, operands read
//      straight from the records (they are stored as K-major operand images), accumulators resident in tensor memory for the
//      whole launch; the appended row of ones yields the bias gradients.
// Thread <-> data mapping of kernel 2 is the forward kernel's: 2 column groups x 8 warps, warp quadrant <-> field / TMEM lane
// quadrant, lane <-> level, 8 columns per thread.
#pragma once
#include "cpz_tc.cuh"

namespace cpz {

struct TcB {
  int K1;          // K extent of the Xbar chain: layer-1 outputs rounded up to a K step (8)
  int K2w;         // K window of one net in the delta1 chains: h2 rounded up to a K step
  int c_a2;        // TMEM column of the layer-2 images: block 0 (nets 0, 1 in lanes 0.. and 64..) hi, lo; block 1 (net 2) hi, lo
  int c_acc;       // first accumulator column; column group g uses [c_acc + 48 g, +48)
  int n_wcols;     // weight columns = c_acc
  int N1, N2;      // MMA N of the layer-1 / layer-2 weight-gradient accumulators (multiples of 16)
};

inline bool tc_bwd_plan(const TcD& T, TcB& B) {
  B.K1 = (3 * T.h1 + 7) & ~7;
  B.K2w = (T.h2 + 7) & ~7;
  B.c_a2 = 2 * B.K1;
  B.c_acc = 2 * B.K1 + 4 * B.K2w;
  B.n_wcols = B.c_acc;
  B.N1 = (3 * T.h1 + 15) & ~15;
  B.N2 = (3 * T.h2 + 15) & ~15;
  return B.c_acc + 96 <= 512 && T.h1 <= 64 && B.N1 + 2 * B.N2 + 96 <= 512;
}
// rows of the records (multiples of 8; one spare row for the ones that produce the bias gradients)
inline void tc_aux_rows(const TcD& T, AuxD& A) {
  A.rx = 104;
  A.r1 = (3 * T.h1 + 1 + 7) & ~7;
  A.r2 = (3 * T.h2 + 1 + 7) & ~7;
  A.r3 = 96;
}

// ---- transposed weight image --------------------------------------------------------------------------------------
// wimg[c][l] = TMEM column c, lane l:
//   [0,K1) hi, [K1,2K1) lo:   lane k < 96 (input row 32*field+level), column f = net*h1+o:  W1_net[o][k]
//   block 0 at c_a2 (+K2w: lo): lane 64*n+o (n = 0, 1), column j < h2:                     W2_n[j][o]   (out j, in o)
//   block 1 at c_a2 + 2 K2w:     lane o (net 2)
// Flux stores W (out x in) column-major: element (out, in) at theta[w_off + in*out_dim + out].
static __global__ void tc_bwd_image_kernel(const __grid_constant__ TcD T, const __grid_constant__ TcB B, const float* __restrict__ theta,
                                           float* __restrict__ wimg) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B.n_wcols * 128) return;
  const int c = idx >> 7, l = idx & 127;
  float w = 0.f;
  bool lo = false;
  if (c < 2 * B.K1) {
    lo = c >= B.K1;
    const int f = lo ? c - B.K1 : c;
    if (l < 96 && f < 3 * T.h1) { const int q = f / T.h1, o = f - q * T.h1; w = theta[T.w_off[q][0] + l * T.h1 + o]; }
  } else {
    int cc = c - B.c_a2;
    const int blk = cc / (2 * B.K2w);
    cc -= blk * 2 * B.K2w;
    lo = cc >= B.K2w;
    const int j = lo ? cc - B.K2w : cc;
    const int q = blk == 0 ? (l >> 6) : 2, o = blk == 0 ? (l & 63) : l;
    if (o < T.h1 && j < T.h2 && (blk == 0 || l < 64)) w = theta[T.w_off[q][1] + o * T.h2 + j];
  }
  const float hi = tf32_hi(w);
  wimg[idx] = lo ? (w - hi) : hi;
}

struct AdjTcArgs {
  const float* wimg;     // transposed weight image [n_wcols][128]
  const float* theta;
  const float* targets;  // [ncol][n_saved][96]
  const float* xN;       // state at the end of the segment in checkpoint layout (tile t at xN + t*xN_stride), read when first != 0
  size_t xN_stride;
  float* xbar;           // [n_tiles][96][32] cotangent of the state, carried from segment to segment
  float* lpart;          // [n_tiles][8] squared-error sums (u, v, T profiles; u, v, T gradients), accumulated over the launches
  AuxD aux;
  int ncol, n_saved;
  int first;             // last segment of the solve: xbar starts from the loss cotangent of the final frame
  int split;             // two CTAs per tile: CTA b sweeps column group b & 1 of tile b >> 1 (lpart is then indexed by CTA)
  int seg_step0, seg_steps;
  float w[6];
  float inv_prof, inv_grad;
  const float* cot;      // [ncol][n_saved][96] cotangent of the trajectory (cpz_solve_vjp): selects adjoint_tc_kernel<..., true>
  float* x0bar;          // [ncol][96] cotangent of x0, written by the launch that ends at step 0 (cot mode), or null
};

constexpr int TCB_SIDE_ARRAYS = 11;  // X_u X_v X_T | e_u e_v e_T (face-flux cotangents) | g_u g_v g_T (cotangents of the level differences) | kbar_u kbar_v

struct TcBSmem {
  int d1h, d1l, d2h, d2l, side, grp_bytes;
  int ks, w3, misc, total;
};
__host__ __device__ inline TcBSmem tc_bwd_smem_layout(const TcB& B, int n_stages) {
  TcBSmem L;
  int o = 0;
  auto take = [&](int bytes) { int r = o; o += (bytes + 127) & ~127; return r; };
  L.d1h = take((B.K1 / 4) * TC_LBO); L.d1l = take((B.K1 / 4) * TC_LBO);
  L.d2h = take((3 * B.K2w / 4) * TC_LBO); L.d2l = take((3 * B.K2w / 4) * TC_LBO);
  L.side = take(TCB_SIDE_ARRAYS * (4 * 32 * 16 + 16));  // 16-byte pad per array: the broadcast reads of two nets' arrays in one warp (S1) hit different banks
  L.grp_bytes = o;
  o = TC_NG * L.grp_bytes;
  L.ks = take(n_stages * (TC_NG * 2 * 3 * 32) * 8 * 4);
  L.w3 = take(31 * 64 * 4);
  L.misc = take(256);
  L.total = o;
  return L;
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// derivative of the hidden activation at the pre-activation z (same fast MUFU forms as tc_act)
template <int ACT>
__device__ __forceinline__ float tc_act_grad(int act_rt, float z) {
  constexpr float L2E = 1.4426950408889634f;
  if constexpr (ACT == ACT_MISH) {  // t + z t', t = n/(n+2), n = e(e+2): t' = 4 e (e+1) / (n+2)^2
    const float e = ex2_fast(fminf(z, 20.f) * L2E);
    const float n = e * (e + 2.f);
    const float r = rcp_fast(n + 2.f);
    return fmaf(z * 4.f * e * (e + 1.f), r * r, n * r);
  } else if constexpr (ACT == ACT_RELU) {
    return z > 0.f ? 1.f : 0.f;
  } else {
    return act_grad(act_rt, z);
  }
}

// VJP of side_column: cotangents (bu, bv, bT) of the three face diffusivities -> cotangents of the level differences.
template <int MODE>
__device__ __forceinline__ void side_column_vjp(const SideC& C, float du, float dv, float dT, float bu, float bv, float bT,
                                                float& Du, float& Dv, float& DT, float& gu, float& gv, float& gT) {
  gu = 0.f; gv = 0.f; gT = 0.f;
  if constexpr (MODE == SIDE_NONE) {
    Du = 0.f; Dv = 0.f; DT = 0.f;
  } else if constexpr (MODE == SIDE_CA_ONLY) {
    Du = 0.f; Dv = 0.f; DT = dT < 0.f ? C.kap : 0.f;  // piecewise constant
  } else {
    constexpr float LN2 = 0.6931471805599453f;
    const float a = du + C.e, b = dv + C.e, c = dT + C.e;
    const float den = fmaf(C.sv2 * b, b, C.su2 * a * a);
    const float rden = rcp_fast(fmaxf(den, 1e-20f));  // finite, and its square too: a saturated step (w (1-w) = 0) must give 0, not 0 * inf
    const float y = fmaf(C.k1 * c, rden, -C.k2);
    const float w = rcp_fast(1.f + ex2_fast(fminf(y, 126.f)));
    Du = fmaf(C.a1, w, C.a0); Dv = fmaf(C.b1, w, C.b0); DT = fmaf(C.t1, w, C.t0);
    bool t_live = true;
    if constexpr (MODE == SIDE_MPP_CA_T) { if (!(dT > 0.f)) { DT = C.kap; t_live = false; } }
    if constexpr (MODE == SIDE_MPP_CA_U) { if (!(du > 0.f)) { DT = C.kap; t_live = false; } }
    const float wb = fmaf(C.a1, bu, fmaf(C.b1, bv, t_live ? C.t1 * bT : 0.f));
    const float yb = -LN2 * w * (1.f - w) * wb;
    gT = yb * C.k1 * rden;
    const float denb = -gT * c * rden;
    gu = 2.f * C.su2 * a * denb;
    gv = 2.f * C.sv2 * b * denb;
  }
}

// ---- reverse sweep over one checkpoint segment -----------------------------------------------------------------------
// IMPL: CPZ_FLAG_IMPLICIT_DIFFUSION models (the VJP of the implicit step is compiled only into this instantiation)
// COT: cot mode (cpz_solve_vjp): a.cot replaces the loss terms; a template parameter because the kernel has no register headroom
template <int ACT, bool IMPL = false, bool COT = false>
__global__ void __launch_bounds__(TC_NT, 1) adjoint_tc_kernel(const __grid_constant__ ModelD M, const __grid_constant__ TcD T,
                                                              const __grid_constant__ TcB B, const __grid_constant__ TableauD tab,
                                                              const TimeD tm, const __grid_constant__ AdjTcArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_tcb[];
  const TcBSmem L = tc_bwd_smem_layout(B, tab.n_stages);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = warp >> 3, wg = warp & 7, qd = wg & 3, h = wg >> 2;
  const uint32_t sbase = smem_u32(smem_tcb);
  const uint32_t gbase = sbase + g * L.grp_bytes;
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem_tcb + L.misc) + g;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_tcb + L.misc + 64);
  float* red = reinterpret_cast<float*>(smem_tcb + L.misc + 128);  // [16 warps][2]
  float* w3s = reinterpret_cast<float*>(smem_tcb + L.w3);          // [j][64]: W3_net[j][o] at row net*h2 + o (the S1 thread's own row: conflict-free)
  const bool active = !a.split || g == (int)(blockIdx.x & 1);
  const int tile = a.split ? (int)(blockIdx.x >> 1) : (int)blockIdx.x, col0 = tile * TC_CT;
  const int cg0 = 16 * g + 8 * h;

  for (int i = tid; i < L.total / 16; i += TC_NT) reinterpret_cast<float4*>(smem_tcb)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  if (tid == 0) {
    mbar_init(mbar, 1);
    mbar_init(mbar + 1, 1);
    fence_mbar_init();
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  for (int i = tid; i < 31 * 64; i += TC_NT) {
    const int r = i & 63, j = i >> 6, q = min(r / T.h2, 2), o = r - q * T.h2;
    w3s[i] = (r < 3 * T.h2 && j < T.nout) ? __ldg(a.theta + T.w_off[q][2] + o * T.nout + j) : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tb = *tmem_slot;
  const uint32_t tlane = tb + ((uint32_t)(32 * qd) << 16);
  for (int c0 = 8 * (warp >> 2); c0 < B.n_wcols; c0 += 32) {  // the four warps of a lane quadrant interleave 8-column chunks
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __ldg(a.wimg + (size_t)(c0 + i) * 128 + 32 * qd + lane);
    tmem_st8(tlane + c0, v);
  }
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");

  const int ns = tab.n_stages, nsub = tm.n_substeps;
  const float hstep = tm.dt / (float)nsub;
  auto frame_of = [&](int step) -> int {
    if (tm.save_stride <= 0) return step == tm.n_steps ? 0 : -1;
    return (step % tm.save_stride == 0) ? step / tm.save_stride : -1;
  };
  float lp = 0.f, lg = 0.f;  // squared-error sums of this thread's field: profile, gradient
  float xbar[8], X[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) { xbar[r] = 0.f; X[r] = 0.f; }
  const float wq = qd < 3 ? a.w[qd] : 0.f, wgq = qd < 3 ? a.w[3 + qd] : 0.f;
  const float Nf = M.rc.Nf;
  // loss terms of one saved frame at state xs (loss.jl:1-42): squared-error sums and d(loss)/dx into xbar
  auto loss_frame = [&](const float* xs, int fr) {
    if constexpr (COT) {  // the trajectory cotangent of the frame, 0 on padding columns
      if (qd < 3) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          const int col = col0 + cg0 + r;
          if (col < a.ncol) xbar[r] += __ldg(a.cot + ((size_t)col * a.n_saved + fr) * 96 + 32 * qd + lane);
        }
      }
      return;
    }
    if (qd < 3) {
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const int col = col0 + cg0 + r;
        const float tg = col < a.ncol ? __ldg(a.targets + ((size_t)col * a.n_saved + fr) * 96 + 32 * qd + lane) : xs[r];
        const float d = xs[r] - tg;
        lp = fmaf(d, d, lp);
        float gx = wq * 2.f * a.inv_prof * d;
        const float dn = __shfl_up_sync(0xffffffffu, d, 1), up = __shfl_down_sync(0xffffffffu, d, 1);
        if (wgq != 0.f) {
          const float g0 = lane >= 1 ? Nf * (d - dn) : 0.f;
          const float g1 = lane <= 30 ? Nf * (up - d) : 0.f;
          lg = fmaf(g0, g0, lg);
          gx = fmaf(wgq * 2.f * a.inv_grad * Nf, g0 - g1, gx);
        }
        xbar[r] += gx;
      }
    }
  };
  float* xb_g = a.xbar + ((size_t)tile * 96 + 32 * qd + lane) * TC_CT + cg0;
  if (qd < 3 && active) {
    if (a.first) {
      const float* src = a.xN + (size_t)tile * a.xN_stride + (size_t)(32 * qd + lane) * TC_CT + cg0;
      const float4 p0 = __ldcg(reinterpret_cast<const float4*>(src)), p1 = __ldcg(reinterpret_cast<const float4*>(src) + 1);
      X[0] = p0.x; X[1] = p0.y; X[2] = p0.z; X[3] = p0.w; X[4] = p1.x; X[5] = p1.y; X[6] = p1.z; X[7] = p1.w;
    } else {
      const float4 p0 = __ldcg(reinterpret_cast<const float4*>(xb_g)), p1 = __ldcg(reinterpret_cast<const float4*>(xb_g) + 1);
      xbar[0] = p0.x; xbar[1] = p0.y; xbar[2] = p0.z; xbar[3] = p0.w; xbar[4] = p1.x; xbar[5] = p1.y; xbar[6] = p1.z; xbar[7] = p1.w;
    }
  }
  if (a.first && active) {
    const int fr = frame_of(tm.n_steps);
    if (fr >= 0) loss_frame(X, fr);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  const uint32_t side = gbase + L.side;
  auto side_addr = [&](int arr, int blk) { return side + (uint32_t)(((arr * 4 + blk) * 32 + lane) * 16 + arr * 16); };
  const int tq = ((g * 2 + h) * 3 + qd) * 32 + lane;
  const uint32_t ks_base = sbase + L.ks + (uint32_t)tq * 16;  // stage slots: [stage][column half][thread] float4 (16-byte thread stride: conflict-free 128-bit accesses)
  const uint32_t ks_stride = (uint32_t)(TC_NG * 2 * 3 * 32) * 32, ks_half = ks_stride / 2;
  const uint32_t dg = tb + B.c_acc + 48 * g;
  const uint32_t id16 = tc_idesc(128, TC_GN);
  uint32_t parity = 0;
  const int bar_id = 1 + g;
  const float Aq = qd < 3 ? M.rc.A[qd] * M.rc.Nf : 0.f;
  const float cso = qd == 0 ? -M.rc.cor_v_s : (qd == 1 ? M.rc.cor_u_s : 0.f);  // Xbar_u += -cor_v_s kbar_v, Xbar_v += cor_u_s kbar_u
  // CPZ_FLAG_IMPLICIT_DIFFUSION: the Runge–Kutta stages carry no diffusive flux; the diffusivities act in the backward-Euler
  // solve at the start of every sub-step, reversed below after the stages of the sub-step
  const int side_mode = IMPL ? (int)SIDE_NONE : T.side_mode;
  const int K1S = B.K1 / 8, K2S = B.K2w / 8;
  const int h1 = T.h1, h2 = T.h2;

  auto chain = [&](uint32_t d, uint32_t ahi, uint32_t alo, uint64_t bh, uint64_t bl, int steps) {
    constexpr uint64_t kstep = (2 * TC_LBO) >> 4;
    for (int s = 0; s < steps; ++s) tc_mma_ts(d, ahi + 8 * s, bl + s * kstep, id16, s > 0);
    for (int s = 0; s < steps; ++s) tc_mma_ts(d, alo + 8 * s, bh + s * kstep, id16, 1);
    for (int s = 0; s < steps; ++s) tc_mma_ts(d, ahi + 8 * s, bh + s * kstep, id16, 1);
  };
  auto rec4 = [&](float* base, int rows, int ev) -> float4* {  // this thread's first column quad of an x / z record (row 0)
    return reinterpret_cast<float4*>(base + ((size_t)tile * a.aux.n_eval + a.aux.ev0 + ev) * (size_t)(32 * rows)) + (size_t)(cg0 >> 2) * rows;
  };
  auto rec4d = [&](float* base, int rows, int ev) -> float4* {  // ... of a d record
    return reinterpret_cast<float4*>(base + ((size_t)tile * a.aux.n_eval_d + ev) * (size_t)(32 * rows)) + (size_t)(cg0 >> 2) * rows;
  };
  auto ld8g = [&](const float4* p, int rows, float* v) {
    const float4 p0 = __ldcs(p), p1 = __ldcs(p + rows);
    v[0] = p0.x; v[1] = p0.y; v[2] = p0.z; v[3] = p0.w; v[4] = p1.x; v[5] = p1.y; v[6] = p1.z; v[7] = p1.w;
  };
  auto st8g = [&](float4* p, int rows, const float* v) {
    p[0] = make_float4(v[0], v[1], v[2], v[3]);
    p[rows] = make_float4(v[4], v[5], v[6], v[7]);
  };

  const int R = a.seg_steps * nsub;
  // delta2 phase mapping: thread (packed row = net*h2 + o, column quad) — 4 outputs per thread, every warp of the group works
  const int gt = tid & 255, d2row = gt & 63, d2quad = gt >> 6;
  const bool d2valid = d2row < 3 * h2;
  const int d2q = d2valid ? d2row / h2 : 0, d2o = d2row - d2q * h2;
  bool have_X = false;  // X already holds the next stage's input (fetched while the previous stage's last MMAs ran)
  for (int rr = active ? R - 1 : -1; rr >= 0; --rr) {
    const int nstep = a.seg_step0 + rr / nsub, sub = rr % nsub;
#pragma unroll 1
    for (int i = ns - 1; i >= 0; --i) {
      const int ev = rr * ns + i;
      // ---- S0: stage input, kbar_i, cotangent of the face fluxes -------------------------------------------------
      if (ev > 0) {  // pull the records of the next stage (evaluation ev - 1) into L2: one 128-byte line per thread
        const int nx = a.aux.rx >> 1, n1 = a.aux.r1 >> 1, n2 = a.aux.r2 >> 1;
        const size_t r = (size_t)tile * a.aux.n_eval + a.aux.ev0 + ev - 1;
        const float* pl = nullptr;  // the group's 4 column quads of a record are contiguous: rows * 64 bytes
        if (gt < nx) pl = a.aux.x + r * (size_t)(32 * a.aux.rx) + (size_t)g * (16 * a.aux.rx) + 32 * gt;
        else if (gt < nx + n1) pl = a.aux.z1 + r * (size_t)(32 * a.aux.r1) + (size_t)g * (16 * a.aux.r1) + 32 * (gt - nx);
        else if (gt < nx + n1 + n2) pl = a.aux.z2 + r * (size_t)(32 * a.aux.r2) + (size_t)g * (16 * a.aux.r2) + 32 * (gt - nx - n1);
        if (pl != nullptr) prefetch_l2(pl);
      }
      float4 z2v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (d2valid) z2v = __ldcs(reinterpret_cast<const float4*>(a.aux.z2 + ((size_t)tile * a.aux.n_eval + a.aux.ev0 + ev) * (size_t)(32 * a.aux.r2)) +
                                (size_t)(4 * g + d2quad) * a.aux.r2 + d2row);
      if (qd < 3) {
        if (!have_X) ld8g(rec4(a.aux.x, a.aux.rx, ev) + 32 * qd + lane, a.aux.rx, X);
        float kb[8];
        const float bi = tab.b[i];
#pragma unroll
        for (int r = 0; r < 8; ++r) kb[r] = bi * xbar[r];
#pragma unroll 1
        for (int j = i + 1; j < ns; ++j) {
          const float aji = tab.a[j][i];
          const float4 p0 = lds_v4(ks_base + j * ks_stride), p1 = lds_v4(ks_base + j * ks_stride + ks_half);
          kb[0] = fmaf(aji, p0.x, kb[0]); kb[1] = fmaf(aji, p0.y, kb[1]); kb[2] = fmaf(aji, p0.z, kb[2]); kb[3] = fmaf(aji, p0.w, kb[3]);
          kb[4] = fmaf(aji, p1.x, kb[4]); kb[5] = fmaf(aji, p1.y, kb[5]); kb[6] = fmaf(aji, p1.z, kb[6]); kb[7] = fmaf(aji, p1.w, kb[7]);
        }
        float eb[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          kb[r] *= hstep;
          const float up = __shfl_down_sync(0xffffffffu, kb[r], 1);
          eb[r] = lane < 31 ? Aq * (up - kb[r]) : 0.f;  // cotangent of the flux at face lane+1 (boundary fluxes are data)
        }
        sts_v4(side_addr(qd, 2 * h), X[0], X[1], X[2], X[3]);
        sts_v4(side_addr(qd, 2 * h + 1), X[4], X[5], X[6], X[7]);
        // e arrays = delta3 (row 32*net + j, j = lane < 31; lane 31 is zero): read by the delta2 phase and the side VJP
        sts_v4(side_addr(3 + qd, 2 * h), eb[0], eb[1], eb[2], eb[3]);
        sts_v4(side_addr(3 + qd, 2 * h + 1), eb[4], eb[5], eb[6], eb[7]);
        if (qd < 2) {
          sts_v4(side_addr(9 + qd, 2 * h), kb[0], kb[1], kb[2], kb[3]);
          sts_v4(side_addr(9 + qd, 2 * h + 1), kb[4], kb[5], kb[6], kb[7]);
        }
        st8g(rec4d(a.aux.d3, a.aux.r3, ev) + 32 * qd + lane, a.aux.r3, eb);
      }
      bar_sync_named(bar_id, 256);  // B1
      // ---- S1: delta2 = (W3 delta3) .* act2'(z2) in FP32 ------------------------------------------------------------
      if (d2valid) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        const float* wp = w3s + d2row;
        const uint32_t dp = side + (uint32_t)((((3 + d2q) * 4 + d2quad) * 32) * 16 + (3 + d2q) * 16);
#pragma unroll 8
        for (int j = 0; j < 31; ++j) {
          const float w = wp[j * 64];
          const float4 p0 = lds_v4(dp + j * 16);
          acc[0] = fmaf(w, p0.x, acc[0]); acc[1] = fmaf(w, p0.y, acc[1]); acc[2] = fmaf(w, p0.z, acc[2]); acc[3] = fmaf(w, p0.w, acc[3]);
        }
        acc[0] *= tc_act_grad<ACT>(T.act2, z2v.x); acc[1] *= tc_act_grad<ACT>(T.act2, z2v.y);
        acc[2] *= tc_act_grad<ACT>(T.act2, z2v.z); acc[3] *= tc_act_grad<ACT>(T.act2, z2v.w);
        // plane row = the net's K window; columns 4*quad .. +3 of the group
        const uint32_t ro = tc_row_off(B.K2w * d2q + d2o, d2quad >> 1) + (uint32_t)(d2quad & 1) * 64;
        store_row_hilo<4>(gbase + L.d2h + ro, gbase + L.d2l + ro, acc);
        reinterpret_cast<float4*>(a.aux.d2 + ((size_t)tile * a.aux.n_eval_d + ev) * (size_t)(32 * a.aux.r2))[(size_t)(4 * g + d2quad) * a.aux.r2 + d2row] =
            make_float4(acc[0], acc[1], acc[2], acc[3]);
      }
      fence_proxy_async();
      tc_fence_before();
      bar_sync_named(bar_id, 256);  // B2
      // ---- S2: delta1 = (W2 delta2) .* act1'(z1); the side VJP runs under the MMAs ------------------------------------
      if (wg == 3) {
        tc_fence_after();
        if (elect_one()) {
#pragma unroll 1
          for (int q = 0; q < 3; ++q) {
            const uint64_t bh = tc_desc(gbase + L.d2h + (uint32_t)(B.K2w * q >> 2) * TC_LBO);
            const uint64_t bl = tc_desc(gbase + L.d2l + (uint32_t)(B.K2w * q >> 2) * TC_LBO);
            const uint32_t ahi = tb + B.c_a2 + (q == 2 ? 2 * B.K2w : 0);
            chain(dg + 16 * q, ahi, ahi + B.K2w, bh, bl, K2S);
          }
          tc_commit(mbar);
        }
        __syncwarp();
      }
      // rows of delta1 this thread owns: net 0 / net 1 rows sit in lanes 0.. / 64.. of the block-0 accumulators (columns
      // +0 / +16), net 2 rows in lanes 0.. of the block-1 accumulator (columns +32): quadrants 0, 1 own two rows
      const int o1 = 32 * (qd & 1) + lane;  // output index inside the net
      const int netA = qd < 2 ? 0 : 1;
      float z1a[8], z1b[8];
      const bool rowA = o1 < h1, rowB = qd < 2 && o1 < h1;
      if (rowA) ld8g(rec4(a.aux.z1, a.aux.r1, ev) + netA * h1 + o1, a.aux.r1, z1a);
      if (rowB) ld8g(rec4(a.aux.z1, a.aux.r1, ev) + 2 * h1 + o1, a.aux.r1, z1b);
      {
        // every thread: face lane+1 of two columns (8h + 2qd, +1): diffusivities and their VJP
        const uint32_t off = (uint32_t)(8 * (qd & 1));
        const int blk = 2 * h + (qd >> 1);
        float2 u, v, Tt, eu, ev2, eT;
        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(u.x), "=f"(u.y) : "r"(side_addr(0, blk) + off) : "memory");
        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(side_addr(1, blk) + off) : "memory");
        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(Tt.x), "=f"(Tt.y) : "r"(side_addr(2, blk) + off) : "memory");
        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(eu.x), "=f"(eu.y) : "r"(side_addr(3, blk) + off) : "memory");
        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(ev2.x), "=f"(ev2.y) : "r"(side_addr(4, blk) + off) : "memory");
        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(eT.x), "=f"(eT.y) : "r"(side_addr(5, blk) + off) : "memory");
        u.x = __shfl_down_sync(0xffffffffu, u.x, 1) - u.x; u.y = __shfl_down_sync(0xffffffffu, u.y, 1) - u.y;
        v.x = __shfl_down_sync(0xffffffffu, v.x, 1) - v.x; v.y = __shfl_down_sync(0xffffffffu, v.y, 1) - v.y;
        Tt.x = __shfl_down_sync(0xffffffffu, Tt.x, 1) - Tt.x; Tt.y = __shfl_down_sync(0xffffffffu, Tt.y, 1) - Tt.y;
        float2 gu, gv, gT;
        auto one = [&](float du, float dv, float dT, float e_u, float e_v, float e_T, float& ou, float& ov, float& oT) {
          float Du, Dv, DT, su, sv, sT;
          // cotangents of the diffusivities: F = -D dq + ...  =>  Dbar = -dq ebar
          switch (side_mode) {
#define CPZ_SIDE_CASE(MODE) \
  case MODE: side_column_vjp<MODE>(T.sc, du, dv, dT, -du * e_u, -dv * e_v, -dT * e_T, Du, Dv, DT, su, sv, sT); break;
            CPZ_SIDE_CASE(SIDE_MPP)
            CPZ_SIDE_CASE(SIDE_MPP_CA_T)
            CPZ_SIDE_CASE(SIDE_MPP_CA_U)
            CPZ_SIDE_CASE(SIDE_CA_ONLY)
            default:
              CPZ_SIDE_CASE(SIDE_NONE)
#undef CPZ_SIDE_CASE
          }
          ou = fmaf(-Du, e_u, su); ov = fmaf(-Dv, e_v, sv); oT = fmaf(-DT, e_T, sT);
          if (lane == 31) { ou = 0.f; ov = 0.f; oT = 0.f; }  // face 32 is the top boundary: its flux is data
        };
        one(u.x, v.x, Tt.x, eu.x, ev2.x, eT.x, gu.x, gv.x, gT.x);
        one(u.y, v.y, Tt.y, eu.y, ev2.y, eT.y, gu.y, gv.y, gT.y);
        asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(side_addr(6, blk) + off), "f"(gu.x), "f"(gu.y) : "memory");
        asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(side_addr(7, blk) + off), "f"(gv.x), "f"(gv.y) : "memory");
        asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(side_addr(8, blk) + off), "f"(gT.x), "f"(gT.y) : "memory");
      }
      mbar_wait(mbar, parity); parity ^= 1u;
      tc_fence_after();
      {
        float v[8];
        tmem_ld8(dg + ((uint32_t)(32 * qd) << 16) + 16 * netA + 8 * h, v);
        if (rowA) {
#pragma unroll
          for (int r = 0; r < 8; ++r) v[r] *= tc_act_grad<ACT>(T.act1, z1a[r]);
          const uint32_t ro = tc_row_off(netA * h1 + o1, h);
          store_row_hilo<8>(gbase + L.d1h + ro, gbase + L.d1l + ro, v);
          st8g(rec4d(a.aux.d1, a.aux.r1, ev) + netA * h1 + o1, a.aux.r1, v);
        }
        if (qd < 2) {
          tmem_ld8(dg + ((uint32_t)(32 * qd) << 16) + 32 + 8 * h, v);
          if (rowB) {
#pragma unroll
            for (int r = 0; r < 8; ++r) v[r] *= tc_act_grad<ACT>(T.act1, z1b[r]);
            const uint32_t ro = tc_row_off(2 * h1 + o1, h);
            store_row_hilo<8>(gbase + L.d1h + ro, gbase + L.d1l + ro, v);
            st8g(rec4d(a.aux.d1, a.aux.r1, ev) + 2 * h1 + o1, a.aux.r1, v);
          }
        }
      }
      fence_proxy_async();
      tc_fence_before();
      bar_sync_named(bar_id, 256);  // B3
      // ---- S3: Xbar_i = W1 delta1 + direct part -------------------------------------------------------------------
      if (wg == 7) {
        tc_fence_after();
        if (elect_one()) {
          chain(dg, tb, tb + B.K1, tc_desc(gbase + L.d1h), tc_desc(gbase + L.d1l), K1S);
          tc_commit(mbar);
        }
        __syncwarp();
      }
      // direct (non-MLP) part of Xbar_i while the MMAs run
      float direct[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) direct[r] = 0.f;
      if (qd < 3) {
        float gq[8];
        lds8(side_addr(6 + qd, 2 * h), side_addr(6 + qd, 2 * h + 1), gq);
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          float dn = __shfl_up_sync(0xffffffffu, gq[r], 1);
          if (lane == 0) dn = 0.f;
          direct[r] = dn - gq[r];  // dq(face lane+1) = X[lane+1] - X[lane]; gq is zero on lane 31
        }
        if (qd < 2) {
          float ko[8];
          lds8(side_addr(9 + (1 - qd), 2 * h), side_addr(9 + (1 - qd), 2 * h + 1), ko);
#pragma unroll
          for (int r = 0; r < 8; ++r) direct[r] = fmaf(cso, ko[r], direct[r]);
        }
        // the next stage's input (stage 0's X must survive until the loss terms of the step start)
        have_X = i > 0;
        if (have_X) ld8g(rec4(a.aux.x, a.aux.rx, ev - 1) + 32 * qd + lane, a.aux.rx, X);
      }
      mbar_wait(mbar, parity); parity ^= 1u;
      tc_fence_after();
      if (qd < 3) {
        float v[8];
        tmem_ld8(dg + ((uint32_t)(32 * qd) << 16) + 8 * h, v);
#pragma unroll
        for (int r = 0; r < 8; ++r) v[r] += direct[r];
        sts_v4(ks_base + i * ks_stride, v[0], v[1], v[2], v[3]);
        sts_v4(ks_base + i * ks_stride + ks_half, v[4], v[5], v[6], v[7]);
      }
      tc_fence_before();
    }
    // xbar_n = xbar_{n+1} + sum_i Xbar_i
    if (qd < 3) {
#pragma unroll 1
      for (int i = 0; i < ns; ++i) {
        const float4 p0 = lds_v4(ks_base + i * ks_stride), p1 = lds_v4(ks_base + i * ks_stride + ks_half);
        xbar[0] += p0.x; xbar[1] += p0.y; xbar[2] += p0.z; xbar[3] += p0.w; xbar[4] += p1.x; xbar[5] += p1.y; xbar[6] += p1.z; xbar[7] += p1.w;
      }
    }
    if constexpr (IMPL) {
      // ---- VJP of x' = L(nu(x))^-1 x (cpz_tc.cuh implicit_step): L is symmetric, so lambda = L^-1 xbar' with the same
      // coefficients; rbar(face) = -(lambda_up - lambda)(x'_up - x'); Dbar = h A_q rbar goes through the VJP of the
      // diffusivities at the INCOMING state x (record xp); xbar = lambda + the face-gradient cotangents scattered to the levels.
      // X holds x' (the input of stage 0), xbar its cotangent.
      float xp[8], Xq[3][8];
#pragma unroll
      for (int r = 0; r < 8; ++r) xp[r] = 0.f;
      if (qd < 3) {
        const size_t rec = (size_t)tile * (a.aux.n_eval / ns) + a.aux.ev0 / ns + rr;
        ld8g(reinterpret_cast<float4*>(a.aux.xp + rec * (size_t)(32 * a.aux.rx)) + (size_t)(cg0 >> 2) * a.aux.rx + 32 * qd + lane, a.aux.rx, xp);
        sts_v4(side_addr(qd, 2 * h), xp[0], xp[1], xp[2], xp[3]);
        sts_v4(side_addr(qd, 2 * h + 1), xp[4], xp[5], xp[6], xp[7]);
      }
      bar_sync_named(bar_id, 256);
      float du[8], dv[8], dT[8], lam[8], rb[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) { du[r] = 0.f; dv[r] = 0.f; dT[r] = 0.f; lam[r] = 0.f; rb[r] = 0.f; }
      if (qd < 3) {
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          if (q == qd) {
#pragma unroll
            for (int r = 0; r < 8; ++r) Xq[q][r] = xp[r];
          } else {
            lds8(side_addr(q, 2 * h), side_addr(q, 2 * h + 1), Xq[q]);
          }
        }
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          du[r] = __shfl_down_sync(0xffffffffu, Xq[0][r], 1) - Xq[0][r];
          dv[r] = __shfl_down_sync(0xffffffffu, Xq[1][r], 1) - Xq[1][r];
          dT[r] = __shfl_down_sync(0xffffffffu, Xq[2][r], 1) - Xq[2][r];
          float Du = 0.f, Dv = 0.f, DT = 0.f;
          switch (T.side_mode) {
            case SIDE_MPP: side_column<SIDE_MPP>(T.sc, du[r], dv[r], dT[r], Du, Dv, DT); break;
            case SIDE_MPP_CA_T: side_column<SIDE_MPP_CA_T>(T.sc, du[r], dv[r], dT[r], Du, Dv, DT); break;
            case SIDE_MPP_CA_U: side_column<SIDE_MPP_CA_U>(T.sc, du[r], dv[r], dT[r], Du, Dv, DT); break;
            case SIDE_CA_ONLY: side_column<SIDE_CA_ONLY>(T.sc, du[r], dv[r], dT[r], Du, Dv, DT); break;
            default: break;
          }
          const float D = qd == 0 ? Du : (qd == 1 ? Dv : DT);
          const float rup = lane == 31 ? 0.f : hstep * Aq * D;
          float rdn = __shfl_up_sync(0xffffffffu, rup, 1);
          if (lane == 0) rdn = 0.f;
          lam[r] = pcr32(-rdn, 1.f + rdn + rup, -rup, xbar[r]);
          const float lup = __shfl_down_sync(0xffffffffu, lam[r], 1), xup = __shfl_down_sync(0xffffffffu, X[r], 1);
          rb[r] = lane == 31 ? 0.f : -hstep * Aq * (lup - lam[r]) * (xup - X[r]);  // cotangent of D_q at face lane+1
        }
        sts_v4(side_addr(3 + qd, 2 * h), rb[0], rb[1], rb[2], rb[3]);
        sts_v4(side_addr(3 + qd, 2 * h + 1), rb[4], rb[5], rb[6], rb[7]);
      }
      bar_sync_named(bar_id, 256);
      if (qd < 3) {
        float Db[3][8];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          if (q == qd) {
#pragma unroll
            for (int r = 0; r < 8; ++r) Db[q][r] = rb[r];
          } else {
            lds8(side_addr(3 + q, 2 * h), side_addr(3 + q, 2 * h + 1), Db[q]);
          }
        }
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          float Du, Dv, DT, gu = 0.f, gv = 0.f, gT = 0.f;
          switch (T.side_mode) {
            case SIDE_MPP: side_column_vjp<SIDE_MPP>(T.sc, du[r], dv[r], dT[r], Db[0][r], Db[1][r], Db[2][r], Du, Dv, DT, gu, gv, gT); break;
            case SIDE_MPP_CA_T: side_column_vjp<SIDE_MPP_CA_T>(T.sc, du[r], dv[r], dT[r], Db[0][r], Db[1][r], Db[2][r], Du, Dv, DT, gu, gv, gT); break;
            case SIDE_MPP_CA_U: side_column_vjp<SIDE_MPP_CA_U>(T.sc, du[r], dv[r], dT[r], Db[0][r], Db[1][r], Db[2][r], Du, Dv, DT, gu, gv, gT); break;
            default: break;  // CA only: piecewise-constant diffusivity
          }
          float gq = qd == 0 ? gu : (qd == 1 ? gv : gT);
          if (lane == 31) gq = 0.f;
          float dn = __shfl_up_sync(0xffffffffu, gq, 1);
          if (lane == 0) dn = 0.f;
          xbar[r] = lam[r] + (dn - gq);
        }
      }
      bar_sync_named(bar_id, 256);  // the side arrays are rewritten by the next sub-step's stages
      if (sub == 0) {
        const int fr = frame_of(nstep);
        if (fr >= 0) loss_frame(xp, fr);  // the saved frame is the state before the step's first implicit solve
      }
    } else {
      if (sub == 0) {  // X still holds the input of stage 0 = x_n
        const int fr = frame_of(nstep);
        if (fr >= 0) loss_frame(X, fr);
      }
    }
  }
  if (qd < 3 && active) {
    reinterpret_cast<float4*>(xb_g)[0] = make_float4(xbar[0], xbar[1], xbar[2], xbar[3]);
    reinterpret_cast<float4*>(xb_g)[1] = make_float4(xbar[4], xbar[5], xbar[6], xbar[7]);
    if (COT && a.x0bar != nullptr) {
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const int col = col0 + cg0 + r;
        if (col < a.ncol) a.x0bar[(size_t)col * 96 + 32 * qd + lane] = xbar[r];
      }
    }
  }
  // squared-error sums: fixed-order reduction (warp shuffles, then the six sums over the warps of a field)
  for (int o = 16; o > 0; o >>= 1) { lp += __shfl_xor_sync(0xffffffffu, lp, o); lg += __shfl_xor_sync(0xffffffffu, lg, o); }
  if (lane == 0) { red[2 * warp] = lp; red[2 * warp + 1] = lg; }
  tc_fence_before();
  __syncthreads();
  if (tid < 6) {
    const int q = tid % 3, kind = tid / 3;
    float s = 0.f;
    for (int w = 0; w < TC_NT / 32; ++w)
      if ((w & 3) == q) s += red[2 * w + kind];
    a.lpart[(size_t)blockIdx.x * 8 + tid] += s;
  }
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tb), "r"(512));
}

// ---- weight gradient: one contraction over every (column, stage) of the launch ------------------------------------------
struct WgradArgs {
  AuxD aux;
  int n_tiles, n_e;  // records of this launch: (tile t, evaluation e < n_e); x / z record aux.ev0 + e, d record e
  float* part;       // [gridDim.x][WG_COLS][128] accumulator images, added to (zeroed by the host before the first launch)
};
constexpr int WG_NT = 576;    // two halves of 8 converter warps + one MMA-issuing warp each (warps 16, 17)
constexpr int WG_HT = 256;    // converter threads of a half
constexpr int WG_BAR = 288;   // threads at a half's barrier
constexpr int WG_COLS = 448;  // N1 + 2 N2 + 96 <= 448
// Sub-records summed in tensor memory before the sums are added to the CTA's FP32 image. One accumulation over every record
// of a launch loses accuracy with its length: at 2 304 columns x 124 steps (~1 500 sub-records per CTA) the weight gradient
// was 1.5e-4 from FP64 where the FP32 oracle is 9e-6 off; blocks of 128 give 1.6e-5 (blocks of 32: 8e-6 at about twice the
// cost). Measured on a B200 at 1000 W: the bench.py config-3 step takes 356 ms instead of 347 ms.
constexpr int WG_BLOCK = 128;

__device__ __forceinline__ uint64_t wg_desc(uint32_t saddr, uint32_t lbo_bytes) {  // K-major, no swizzle, SBO = 128
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)(128 >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void tc_mma_ss(uint32_t d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d),
               "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
               : "memory");
}

// The CTA is two independent halves of 8 warps (own operand planes, own mbarrier and named barrier, own accumulator columns),
// free-running against each other so that one half's global fetch / hi-lo split overlaps the other's MMAs:
//   half 0: dW1 += [X;1] d1^T   (M 128 x N1)   and  dW3 += [a2;1] d3^T (M 128 x 96)      arrays x, z2, d1, d3
//   half 1: dW2 += [a1;1] d2^T  as two row blocks (rows 0..127, rows 128..) of M 128 x N2   arrays z1, d2
// Operand planes of a half: hi planes of its arrays (A operands first), then the lo planes; every array is the record image
// [column quad][row][4] itself. A operands are read as M = 128 rows: rows past an array's end run into the arrays behind
// it (finite values whose accumulator rows are never read). Records are fetched through registers one record ahead and
// pulled into L2 two records ahead.
//
// One array of a half: ID 0 x, 1 z1, 2 z2, 3 d1, 4 d2, 5 d3; NV = float4 per thread (rows <= 32 NV)
template <int ID_, int NV_>
struct WgArr {
  static constexpr int ID = ID_, NV = NV_;
};
template <int ACT, int ID>
__device__ __forceinline__ float4 wg_role(const TcD& T, int row, float4 v) {
  const float4 one = make_float4(1.f, 1.f, 1.f, 1.f), zero = make_float4(0.f, 0.f, 0.f, 0.f);
  if constexpr (ID == 0) {
    if (row == 96) v = one; else if (row > 96) v = zero;
  } else if constexpr (ID == 1) {
    if (row < 3 * T.h1) { v.x = tc_act<ACT>(T.act1, v.x); v.y = tc_act<ACT>(T.act1, v.y); v.z = tc_act<ACT>(T.act1, v.z); v.w = tc_act<ACT>(T.act1, v.w); }
    else v = row == 3 * T.h1 ? one : zero;
  } else if constexpr (ID == 2) {
    if (row < 3 * T.h2) { v.x = tc_act<ACT>(T.act2, v.x); v.y = tc_act<ACT>(T.act2, v.y); v.z = tc_act<ACT>(T.act2, v.z); v.w = tc_act<ACT>(T.act2, v.w); }
    else v = row == 3 * T.h2 ? one : zero;
  } else if constexpr (ID == 3) {
    if (row >= 3 * T.h1) v = zero;
  } else if constexpr (ID == 4) {
    if (row >= 3 * T.h2) v = zero;
  } else {
    if ((row & 31) == 31) v = zero;
  }
  return v;
}

template <int ACT, int HALF>
__device__ __forceinline__ void wgrad_half(const TcD& T, const TcB& B, const WgradArgs& a, uint8_t* smem, uint64_t* mbar, uint32_t tb) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, ht = tid & (WG_HT - 1);
  const bool is_mma = warp >= 16;  // this half's issuing warp: no fetch / convert work, so the MMA issue is off the converters' path
  // arrays in plane order (A operands first); NV = float4 per thread of a 16-column sub-record (4 column quads x rows)
  using A0 = std::conditional_t<HALF == 0, WgArr<0, 2>, WgArr<1, 3>>;
  using A1 = std::conditional_t<HALF == 0, WgArr<2, 2>, WgArr<4, 2>>;
  using A2 = WgArr<3, 3>;  // half 0 only
  using A3 = WgArr<5, 2>;  // half 0 only
  const int rows_all[6] = {a.aux.rx, a.aux.r1, a.aux.r2, a.aux.r1, a.aux.r2, a.aux.r3};
  float* const src_all[6] = {a.aux.x, a.aux.z1, a.aux.z2, a.aux.d1, a.aux.d2, a.aux.d3};
  const int r0 = rows_all[A0::ID], r1 = rows_all[A1::ID], r2 = HALF == 0 ? rows_all[A2::ID] : 0, r3 = HALF == 0 ? rows_all[A3::ID] : 0;
  const int o0 = 0, o1 = 4 * r0, o2 = o1 + 4 * r1, o3 = o2 + 4 * r2, set4 = o3 + 4 * r3;  // float4 offsets inside a plane set (16 columns)
  const int set4_h0 = 4 * (a.aux.rx + a.aux.r2 + a.aux.r1 + a.aux.r3);
  // planes of this half: buffer 0 hi, lo, buffer 1 hi, lo
  float4* planes = reinterpret_cast<float4*>(smem) + (HALF ? 4 * set4_h0 : 0);
  const int n_rec = a.n_tiles * a.n_e;
  float4 b0[A0::NV], b1[A1::NV], b2[HALF == 0 ? A2::NV : 1], b3[HALF == 0 ? A3::NV : 1];
  int w0[A0::NV], w1[A1::NV], w2[HALF == 0 ? A2::NV : 1], w3[HALF == 0 ? A3::NV : 1];  // row of this thread's j-th float4
#pragma unroll
  for (int j = 0; j < A0::NV; ++j) w0[j] = (ht + j * WG_HT) % r0;
#pragma unroll
  for (int j = 0; j < A1::NV; ++j) w1[j] = (ht + j * WG_HT) % r1;
  if constexpr (HALF == 0) {
#pragma unroll
    for (int j = 0; j < A2::NV; ++j) w2[j] = (ht + j * WG_HT) % r2;
#pragma unroll
    for (int j = 0; j < A3::NV; ++j) w3[j] = (ht + j * WG_HT) % r3;
  }
  // sub-record u of this CTA: record blockIdx.x + (u >> 1) gridDim.x, column half u & 1 (column quads 4 (u & 1) ..).
  // (tile, evaluation) of the fetch and prefetch streams are advanced incrementally (no division in the loop)
  struct Cur { int t, e; };
  Cur cf, cp;
  { const int rec = blockIdx.x; cf.t = rec / a.n_e; cf.e = rec - cf.t * a.n_e; cp = cf; }
  const int estep = gridDim.x;
  auto advance = [&](Cur& c) { c.e += estep; while (c.e >= a.n_e) { c.e -= a.n_e; ++c.t; } };
  auto sub_ptr = [&](int idk, int rows, const Cur& c, int u) -> const float4* {
    const size_t r = idk < 3 ? (size_t)c.t * a.aux.n_eval + a.aux.ev0 + c.e : (size_t)c.t * a.aux.n_eval_d + c.e;
    return reinterpret_cast<const float4*>(src_all[idk] + r * (size_t)(32 * rows)) + (u & 1) * 4 * rows;
  };
  auto fetch1 = [&](auto arr, int rows, float4* buf, int u) {
    using AR = decltype(arr);
    const float4* p = sub_ptr(AR::ID, rows, cf, u);
#pragma unroll
    for (int j = 0; j < AR::NV; ++j) {
      const int idx = ht + j * WG_HT;
      if (idx < 4 * rows) buf[j] = __ldcs(p + idx);
    }
  };
  auto pref1 = [&](auto arr, int rows, int u) {
    using AR = decltype(arr);
    const float4* p = sub_ptr(AR::ID, rows, cp, u);
    if (8 * ht < 4 * rows) prefetch_l2(p + 8 * ht);
  };
  auto conv1 = [&](auto arr, int rows, int off, const float4* buf, const int* rw, float4* hi, float4* lo) {
    using AR = decltype(arr);
#pragma unroll
    for (int j = 0; j < AR::NV; ++j) {
      const int idx = ht + j * WG_HT;
      if (idx < 4 * rows) {
        const float4 v = wg_role<ACT, AR::ID>(T, rw[j], buf[j]);
        float4 vh, vl;
        vh.x = tf32_hi(v.x); vh.y = tf32_hi(v.y); vh.z = tf32_hi(v.z); vh.w = tf32_hi(v.w);
        vl.x = v.x - vh.x; vl.y = v.y - vh.y; vl.z = v.z - vh.z; vl.w = v.w - vh.w;
        hi[off + idx] = vh;
        lo[off + idx] = vl;
      }
    }
  };
  auto fetch = [&](int u) {  // called for u = 0, 1, 2, ... in order
    fetch1(A0{}, r0, b0, u); fetch1(A1{}, r1, b1, u);
    if constexpr (HALF == 0) { fetch1(A2{}, r2, b2, u); fetch1(A3{}, r3, b3, u); }
    if (u & 1) advance(cf);
  };
  auto prefetch = [&](int u) {  // called for u = 1, 2, 3, ... in order
    if ((u & 1) == 0) advance(cp);
    pref1(A0{}, r0, u); pref1(A1{}, r1, u);
    if constexpr (HALF == 0) { pref1(A2{}, r2, u); pref1(A3{}, r3, u); }
  };
  auto convert = [&](float4* hi, float4* lo) {
    conv1(A0{}, r0, o0, b0, w0, hi, lo); conv1(A1{}, r1, o1, b1, w1, hi, lo);
    if constexpr (HALF == 0) { conv1(A2{}, r2, o2, b2, w2, hi, lo); conv1(A3{}, r3, o3, b3, w3, hi, lo); }
  };
  const uint32_t id1 = tc_idesc(128, B.N1), id2 = tc_idesc(128, B.N2), id3 = tc_idesc(128, 96);
  // accumulators -> this CTA's image (added: the image carries the sum over the blocks and launches). Image columns: dW1
  // [0,N1), dW2 rows 0..127 [N1,N1+N2), rows 128.. [N1+N2,N1+2N2), dW3 [N1+2N2,+96)
  auto drain = [&]() {  // two 8-column chunks per round: their image loads are in flight together
    float* dst = a.part + (size_t)blockIdx.x * WG_COLS * 128 + 32 * (warp & 3) + lane;
    const uint32_t tl = tb + ((uint32_t)(32 * (warp & 3)) << 16);
    const int ncols = HALF == 0 ? B.N1 + 96 : 2 * B.N2;
    auto col = [&](int c) { return HALF == 0 ? (c < B.N1 ? c : c + 2 * B.N2) : B.N1 + c; };
    for (int c0 = 8 * ((warp >> 2) & 1); c0 < ncols; c0 += 32) {
      const bool two = c0 + 16 < ncols;
      float v[16], o[16];
      tmem_ld8(tl + c0, v);
      if (two) tmem_ld8(tl + c0 + 16, v + 8);
      const int i0 = col(c0), i1 = col(c0 + 16);
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = dst[(size_t)(i0 + i) * 128];
      if (two) {
#pragma unroll
        for (int i = 0; i < 8; ++i) o[8 + i] = dst[(size_t)(i1 + i) * 128];
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) dst[(size_t)(i0 + i) * 128] = o[i] + v[i];
      if (two) {
#pragma unroll
        for (int i = 0; i < 8; ++i) dst[(size_t)(i1 + i) * 128] = o[8 + i] + v[8 + i];
      }
    }
  };
  uint32_t parity[2] = {0u, 0u};
  const int n_mine = blockIdx.x < n_rec ? (n_rec - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  const int n_sub = 2 * n_mine;
  if (!is_mma) {
    if (n_sub > 0) fetch(0);
    for (int u = 1; u < 4 && u < n_sub; ++u) prefetch(u);
  }
  for (int u = 0; u < n_sub; ++u) {
    const int b = u & 1;
    float4* hi = planes + b * 2 * set4;
    float4* lo = hi + set4;
    if (!is_mma) {
      if (u >= 2) { mbar_wait(mbar + b, parity[b]); parity[b] ^= 1u; }  // the MMAs that read this buffer two sub-records ago are done
      if (u % WG_BLOCK == 0 && u > 0) {
        // end of an accumulation block: every MMA so far is done (the commit of sub-record u - 1 covers them; the wait of
        // sub-record u + 1 on the same phase then returns at once); the block's sums go to the image before sub-record u
        // restarts the accumulators
        mbar_wait(mbar + (b ^ 1), parity[b ^ 1]);
        tc_fence_after();
        drain();
      }
      convert(hi, lo);
      fence_proxy_async();
      tc_fence_before();
    }
    bar_sync_named(1 + HALF, WG_BAR);
    if (!is_mma) {
      if (u + 1 < n_sub) fetch(u + 1);  // in flight while the MMAs run
      if (u + 4 < n_sub) prefetch(u + 4);
    } else {
      tc_fence_after();
      if (elect_one()) {
        const uint32_t sh = smem_u32(hi), sl = smem_u32(lo);
#pragma unroll 1
        for (int pass = 0; pass < 3; ++pass) {
          const uint32_t sa = pass == 1 ? sl : sh, sb = pass == 0 ? sl : sh;  // hi*lo, lo*hi, hi*hi
#pragma unroll 1
          for (int s = 0; s < 2; ++s) {
            const uint32_t acc = (u % WG_BLOCK == 0 && pass == 0 && s == 0) ? 0u : 1u;
            auto D = [&](uint32_t base, int off, int rows, int row0) { return wg_desc(base + (uint32_t)(off + 2 * s * rows + row0) * 16, (uint32_t)rows * 16); };
            if constexpr (HALF == 0) {
              tc_mma_ss(tb, D(sa, o0, r0, 0), D(sb, o2, r2, 0), id1, acc);
              tc_mma_ss(tb + B.N1, D(sa, o1, r1, 0), D(sb, o3, r3, 0), id3, acc);
            } else {
              tc_mma_ss(tb, D(sa, o0, r0, 0), D(sb, o1, r1, 0), id2, acc);
              tc_mma_ss(tb + B.N2, D(sa, o0, r0, 128), D(sb, o1, r1, 0), id2, acc);
            }
          }
        }
        tc_commit(mbar + b);
      }
      __syncwarp();
    }
  }
  if (n_sub > 0 && !is_mma) {
    // the last two commits cover every MMA (a commit tracks all MMAs issued before it)
    const int bl = (n_sub - 1) & 1;
    if (n_sub >= 2) { mbar_wait(mbar + (bl ^ 1), parity[bl ^ 1]); }
    mbar_wait(mbar + bl, parity[bl]);
    tc_fence_after();
    drain();
  }
}

template <int ACT>
__global__ void __launch_bounds__(WG_NT, 1) wgrad_tc_kernel(const __grid_constant__ TcD T, const __grid_constant__ TcB B,
                                                            const __grid_constant__ WgradArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_wg[];
  const int tid = threadIdx.x, warp = tid >> 5;
  const int half = warp < 16 ? warp >> 3 : warp - 16;
  // 2 halves x 2 buffers x (hi, lo) x 16 columns = the bytes of one full hi + lo record
  const int total4 = 16 * (a.aux.rx + a.aux.r2 + a.aux.r1 + a.aux.r3) + 16 * (a.aux.r1 + a.aux.r2);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem_wg + (size_t)total4 * 16);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_wg + (size_t)total4 * 16 + 32);
  if (tid == 0) { for (int i = 0; i < 4; ++i) mbar_init(mbar + i, 1); fence_mbar_init(); }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tb = *tmem_slot;
  if (half == 0) wgrad_half<ACT, 0>(T, B, a, smem_wg, mbar, tb);
  else wgrad_half<ACT, 1>(T, B, a, smem_wg, mbar + 2, tb + 256);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tb), "r"(512));
}

// Reference contraction of the same records in plain FP32 (CPZ_WGRAD_REF=1: validation of wgrad_tc_kernel; slow). One thread
// per accumulator element (column c, lane l) of the image layout; the records are read with the same row rules.
template <int ACT>
__global__ void wgrad_ref_kernel(const __grid_constant__ TcD T, const __grid_constant__ TcB B, const __grid_constant__ WgradArgs a) {
  const int ncols = B.N1 + 2 * B.N2 + 96;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= ncols * 128) return;
  const int c = idx >> 7, l = idx & 127;
  int ka, rowa, kb, rowb;  // operand arrays / rows
  if (c < B.N1) { ka = 0; rowa = l; kb = 3; rowb = c; }
  else if (c < B.N1 + B.N2) { ka = 1; rowa = l; kb = 4; rowb = c - B.N1; }
  else if (c < B.N1 + 2 * B.N2) { ka = 1; rowa = 128 + l; kb = 4; rowb = c - B.N1 - B.N2; }
  else { ka = 2; rowa = l; kb = 5; rowb = c - B.N1 - 2 * B.N2; }
  const int rows[6] = {a.aux.rx, a.aux.r1, a.aux.r2, a.aux.r1, a.aux.r2, a.aux.r3};
  const float* src[6] = {a.aux.x, a.aux.z1, a.aux.z2, a.aux.d1, a.aux.d2, a.aux.d3};
  const int h1x3 = 3 * T.h1, h2x3 = 3 * T.h2;
  const int va = ka == 0 ? 96 : (ka == 1 ? h1x3 : h2x3);  // the ones row; rows above are zero
  const bool bvalid = kb == 3 ? rowb < h1x3 : (kb == 4 ? rowb < h2x3 : (rowb < 96 && (rowb & 31) != 31));
  float s = 0.f;
  if (rowa <= va && bvalid) {
    for (int rec = 0; rec < a.n_tiles * a.n_e; ++rec) {
      const int t = rec / a.n_e, e = rec - t * a.n_e;
      const float* pa = src[ka] + ((size_t)t * a.aux.n_eval + a.aux.ev0 + e) * 32 * rows[ka];
      const float* pb = src[kb] + ((size_t)t * a.aux.n_eval_d + e) * 32 * rows[kb];
      for (int col = 0; col < 32; ++col) {
        float av = 1.f;
        if (rowa < va) {
          av = pa[((col >> 2) * rows[ka] + rowa) * 4 + (col & 3)];
          if (ka == 1) av = tc_act<ACT>(T.act1, av);
          if (ka == 2) av = tc_act<ACT>(T.act2, av);
        }
        s = fmaf(av, pb[((col >> 2) * rows[kb] + rowb) * 4 + (col & 3)], s);
      }
    }
  }
  a.part[idx] += s;
}

// gradient in destructure order from the accumulator images: out[p] = sum over CTA images (fixed order)
static __global__ void wgrad_finish_kernel(const __grid_constant__ TcD T, const __grid_constant__ TcB B, const float* __restrict__ part,
                                           int n_img, int P, float* __restrict__ out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const int dims[4] = {96, T.h1, T.h2, T.nout};
  int c = -1, l = -1;
  for (int q = 0; q < 3 && c < 0; ++q)
    for (int layer = 0; layer < 3 && c < 0; ++layer) {
      const int K = dims[layer], N = dims[layer + 1];
      int in = -1, out_i = -1;
      if (p >= T.w_off[q][layer] && p < T.w_off[q][layer] + K * N) { const int e = p - T.w_off[q][layer]; in = e / N; out_i = e - in * N; }
      else if (p >= T.b_off[q][layer] && p < T.b_off[q][layer] + N) { in = -2; out_i = p - T.b_off[q][layer]; }
      if (in == -1) continue;
      if (layer == 0) {
        l = in == -2 ? 96 : in;
        c = q * T.h1 + out_i;
      } else if (layer == 1) {
        const int f = in == -2 ? 3 * T.h1 : q * T.h1 + in;
        l = f & 127;
        c = B.N1 + (f >> 7) * B.N2 + q * T.h2 + out_i;
      } else {
        l = in == -2 ? 3 * T.h2 : q * T.h2 + in;
        c = B.N1 + 2 * B.N2 + 32 * q + out_i;
      }
    }
  float s = 0.f;
  if (c >= 0)
    for (int t = 0; t < n_img; ++t) s += part[((size_t)t * WG_COLS + c) * 128 + l];
  out[p] = s;
}

}  // namespace cpz
