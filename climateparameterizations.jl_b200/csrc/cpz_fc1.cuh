// Small-batch training pass of the T-only NDE (BASELINE config 1: ONE column, convective adjustment + mPP base, forward solve +
// loss gradient): one CTA per column, no column padding.
//
// Replaces, for a handful of columns, what the reference does per simulation in train_neural_differential_equation!
// (free_convection/src/training.jl:44-71: solve_nde + Flux.mse + Zygote gradient through InterpolatingAdjoint) for the RHS of
// ConvectiveAdjustmentNDE (free_convection/src/convective_adjustment_nde.jl:33-48) with the mPP base of
// wind_mixing/src/NDE_training.jl:114-139 at u = v = 0. Same discrete adjoint as adjoint_kernel (cpz_adjoint.cuh); the
// difference is the mapping: with one column there is no batch dimension to tile over, so
//   * the weights stay in shared memory in Flux's [in][out] order and every layer is a mat-vec whose outputs are spread over
//     the 512 threads (output o, K quarter kq), partial sums combined through shared memory;
//   * every thread owns a FIXED set of weight-gradient entries in registers for the whole reverse sweep
//     (dW2: 32, dW1: 8, dW3: 8, biases: 3) — no gradient slab is read-modify-written per stage;
//   * the transposed products of the delta propagation read the same weight copy with a lane skew that keeps the
//     shared-memory banks distinct.
// The shared-memory weight copy is zero-padded to 32 x 128, 128 x 128, 128 x 32 so that every loop has a constant trip count
// (fully unrolled, loads ahead of the FMAs). The forward pass writes the RECORD of every stage evaluation (stage input, z1,
// a1, z2, a2: 544 floats, 226 MB for config 1) to HBM instead of sparse checkpoints; the reverse sweep streams them back one
// sub-step ahead with cp.async into a double buffer and recomputes nothing.
#pragma once
#include "cpz_device.cuh"
#include "cpz_tc.cuh"  // pcr32: tridiagonal solve across the lanes of a warp

namespace cpz {

constexpr int FC1_NT = 512;

struct Fc1D {
  int h1, h2;        // hidden widths (<= 128); input 32, output 31
  int act1, act2;
  int w_off[3], b_off[3];
  int P;
};

struct Fc1Args {
  const float* theta;
  const float* x0;       // [ncol][32] (row stride x0_stride, 0 = 32)
  size_t x0_stride;
  const float* bcs;      // [ncol][2]
  const float* targets;  // [ncol][n_saved][32]
  float* xp;             // implicit diffusion: [ncol][n_sub][32] state before the implicit step of every sub-step
  float* records;        // [ncol][n_sub * n_stages][FC1_REC]: y (32), z1 (128), a1 (128), z2 (128), a2 (128) of every stage evaluation
  float* gpart;          // [ncol][P]: d(unnormalised loss of this column)/dtheta
  float* lpart;          // [ncol][8]: squared-error sum of the T profiles at index 2
  int ncol, n_saved, n_sub;  // n_sub = n_steps * n_substeps
  float wT, inv_prof;
  const float* cot;      // [ncol][n_saved][32] cotangent of the trajectory (cpz_solve_vjp), or null: loss mode (targets)
  float* x0bar;          // [ncol][32] cotangent of x0 (cot mode), or null
};

// zero-padded weight copy in shared memory
constexpr int FC1_W1 = 0, FC1_W2 = 32 * 128, FC1_W3 = FC1_W2 + 128 * 128, FC1_B1 = FC1_W3 + 128 * 32, FC1_B2 = FC1_B1 + 128,
              FC1_B3 = FC1_B2 + 128, FC1_WTOT = FC1_B3 + 32;

constexpr int FC1_REC = 544, FC1_Y = 0, FC1_Z1 = 32, FC1_A1 = 160, FC1_Z2 = 288, FC1_A2 = 416;  // floats of one stage record

struct Fc1Smem {
  int w, xs, xbar, ks, yb, rec, part, d1, d2, d3, nn, total_floats;
};
__host__ __device__ inline Fc1Smem fc1_smem_layout(int n_stages) {
  Fc1Smem L;
  int o = 0;
  auto take = [&](int n) { int r = o; o += (n + 3) & ~3; return r; };
  L.w = take(FC1_WTOT);
  L.xs = take(32); L.xbar = take(32);
  L.ks = take(n_stages * 32);   // forward: stage tendencies k_i
  L.yb = take(n_stages * 32);   // reverse: cotangents of the stage inputs
  L.rec = take(2 * n_stages * FC1_REC);  // forward: one scratch record; reverse: the records of two sub-steps (double buffer)
  L.part = take(4 * 128);       // partial sums: [4][128] or [16][32]
  L.d1 = take(128); L.d2 = take(128); L.d3 = take(32);
  L.nn = take(32);
  L.total_floats = o;
  return L;
}

__global__ void __launch_bounds__(FC1_NT, 1) fc1_train_kernel(const __grid_constant__ ModelD M, const __grid_constant__ Fc1D F,
                                                              const __grid_constant__ TableauD tab, const TimeD tm,
                                                              const __grid_constant__ Fc1Args a) {
  extern __shared__ __align__(16) float smem[];
  const int ns = tab.n_stages, nsub = tm.n_substeps;
  const Fc1Smem L = fc1_smem_layout(ns);
  float* wsm = smem + L.w;
  float* xs = smem + L.xs;
  float* xbar = smem + L.xbar;
  float* ks = smem + L.ks;
  float* yb = smem + L.yb;
  float* recs = smem + L.rec;
  float* part = smem + L.part;
  float* d1s = smem + L.d1;
  float* d2s = smem + L.d2;
  float* d3s = smem + L.d3;
  float* nns = smem + L.nn;

  const int t = threadIdx.x, lane = t & 31;
  const int o128 = t & 127, kq4 = t >> 7;   // (output, K quarter) of the 128-wide layers
  const int o32 = t & 31, kq16 = t >> 5;    // (output, K sixteenth) of the 31-wide output layer
  const int col = blockIdx.x;
  const int h1 = F.h1, h2 = F.h2;
  const float* W1 = wsm + FC1_W1;  // [32][128]
  const float* W2 = wsm + FC1_W2;  // [128][128]
  const float* W3 = wsm + FC1_W3;  // [128][32]
  const float* B1 = wsm + FC1_B1;
  const float* B2 = wsm + FC1_B2;
  const float* B3 = wsm + FC1_B3;
  const float Nf = M.rc.Nf, AN = M.rc.A[2] * M.rc.Nf;
  const bool mpp = (M.flags & F_MPP) != 0, ca = (M.flags & F_CA) != 0;
  // CPZ_FLAG_IMPLICIT_DIFFUSION: the stages carry the NN and boundary fluxes only; the diffusive / convective-adjustment flux acts
  // in a backward-Euler solve at the start of every sub-step (warp 0: lane <-> level, cyclic reduction across the warp)
  const bool implicit = (M.flags & F_IMPLICIT) != 0;
  const bool mpp_e = mpp && !implicit, ca_e = ca && !implicit;
  const float hstep = tm.dt / (float)nsub;

  for (int i = t; i < FC1_WTOT; i += FC1_NT) {
    float w = 0.f;
    if (i < FC1_W2) { const int k = i >> 7, o = i & 127; if (o < h1) w = __ldg(a.theta + F.w_off[0] + k * h1 + o); }
    else if (i < FC1_W3) { const int k = (i - FC1_W2) >> 7, o = i & 127; if (k < h1 && o < h2) w = __ldg(a.theta + F.w_off[1] + k * h2 + o); }
    else if (i < FC1_B1) { const int k = (i - FC1_W3) >> 5, o = i & 31; if (k < h2 && o < 31) w = __ldg(a.theta + F.w_off[2] + k * 31 + o); }
    else if (i < FC1_B2) { const int o = i - FC1_B1; if (o < h1) w = __ldg(a.theta + F.b_off[0] + o); }
    else if (i < FC1_B3) { const int o = i - FC1_B2; if (o < h2) w = __ldg(a.theta + F.b_off[1] + o); }
    else { const int o = i - FC1_B3; if (o < 31) w = __ldg(a.theta + F.b_off[2] + o); }
    wsm[i] = w;
  }
  if (t < 32) {
    xs[t] = __ldg(a.x0 + (size_t)col * (a.x0_stride ? a.x0_stride : (size_t)32) + t);
    xbar[t] = 0.f;
  }
  const float bc0 = __ldg(a.bcs + (size_t)col * 2), bc1 = __ldg(a.bcs + (size_t)col * 2 + 1);
  __syncthreads();

  // ---- MLP forward at the stage input y; the pre-activations / activations go to z1o, a1o, z2o, a2o; result in nns[0..30] ----
  auto mlp_forward = [&](const float* __restrict__ y, float* __restrict__ g) {  // g: this evaluation's record in HBM
    float* z1o = recs + FC1_Z1; float* a1o = recs + FC1_A1; float* z2o = recs + FC1_Z2; float* a2o = recs + FC1_A2;
    {  // layer 1: K = 32 split in four
      const float* w = W1 + (8 * kq4) * 128 + o128;
      const float4 y0 = reinterpret_cast<const float4*>(y + 8 * kq4)[0], y1 = reinterpret_cast<const float4*>(y + 8 * kq4)[1];
      float acc0 = w[0] * y0.x, acc1 = w[128] * y0.y;
      acc0 = fmaf(w[256], y0.z, acc0); acc1 = fmaf(w[384], y0.w, acc1);
      acc0 = fmaf(w[512], y1.x, acc0); acc1 = fmaf(w[640], y1.y, acc1);
      acc0 = fmaf(w[768], y1.z, acc0); acc1 = fmaf(w[896], y1.w, acc1);
      part[kq4 * 128 + o128] = acc0 + acc1;
    }
    __syncthreads();
    if (t < 128) {
      float z = 0.f, av = 0.f;
      if (t < h1) {
        z = (part[t] + part[128 + t]) + (part[256 + t] + part[384 + t]) + B1[t];
        av = act_fwd(F.act1, z);
      }
      z1o[t] = z; a1o[t] = av;
      g[FC1_Z1 + t] = z; g[FC1_A1 + t] = av;
    }
    __syncthreads();
    {  // layer 2: K = h1 (<= 128) split in four
      float acc0 = 0.f, acc1 = 0.f, acc2_ = 0.f, acc3_ = 0.f;
      const float* w = W2 + (32 * kq4) * 128 + o128;
      const float4* av = reinterpret_cast<const float4*>(a1o + 32 * kq4);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float4 v = av[q];
        acc0 = fmaf(w[(4 * q) * 128], v.x, acc0); acc1 = fmaf(w[(4 * q + 1) * 128], v.y, acc1);
        acc2_ = fmaf(w[(4 * q + 2) * 128], v.z, acc2_); acc3_ = fmaf(w[(4 * q + 3) * 128], v.w, acc3_);
      }
      part[kq4 * 128 + o128] = (acc0 + acc1) + (acc2_ + acc3_);
    }
    __syncthreads();
    if (t < 128) {
      float z = 0.f, av = 0.f;
      if (t < h2) {
        z = (part[t] + part[128 + t]) + (part[256 + t] + part[384 + t]) + B2[t];
        av = act_fwd(F.act2, z);
      }
      z2o[t] = z; a2o[t] = av;
      g[FC1_Z2 + t] = z; g[FC1_A2 + t] = av;
    }
    __syncthreads();
    {  // layer 3: 31 outputs, K = h2 split in sixteen
      const float* w = W3 + (8 * kq16) * 32 + o32;
      const float4 v0 = reinterpret_cast<const float4*>(a2o + 8 * kq16)[0], v1 = reinterpret_cast<const float4*>(a2o + 8 * kq16)[1];
      float acc0 = w[0] * v0.x, acc1 = w[32] * v0.y;
      acc0 = fmaf(w[64], v0.z, acc0); acc1 = fmaf(w[96], v0.w, acc1);
      acc0 = fmaf(w[128], v1.x, acc0); acc1 = fmaf(w[160], v1.y, acc1);
      acc0 = fmaf(w[192], v1.z, acc0); acc1 = fmaf(w[224], v1.w, acc1);
      part[kq16 * 32 + o32] = acc0 + acc1;
    }
    __syncthreads();
    if (t < 32) {
      float s = 0.f;
      if (t < 31) {
#pragma unroll
        for (int q = 0; q < 16; ++q) s += part[q * 32 + t];
        s += B3[t];
      }
      nns[t] = s;
    }
    __syncwarp();
  };

  // tendency of level `lane` from the stage input y and the NN fluxes in nns (warp 0 only)
  auto tendency = [&](const float* __restrict__ y) -> float {
    float Fl = bc0;  // flux at face lane (face 0: bottom boundary)
    if (lane >= 1) {
      const float G = Nf * (y[lane] - y[lane - 1]);
      Fl = nns[lane - 1];
      if (mpp_e) Fl -= fc_mpp_cnu(M, G) * G;
      if (ca_e) Fl -= fminf(0.f, M.rc.K_ca * G);
    }
    float Fu = __shfl_down_sync(0xffffffffu, Fl, 1);
    if (lane == 31) Fu = bc1;
    return -AN * (Fu - Fl);
  };

  // diffusivity D at face lane+1 (flux -D G, G = Nf (x[lane+1] - x[lane])) and dD/dG: [mPP] c_T nu/Pr + [CA] K [G < 0]
  auto face_D = [&](float G, float& dDdG) -> float {
    float D = 0.f;
    dDdG = 0.f;
    if (mpp) D += fc_mpp_cnu(M, G, &dDdG);
    if (ca && M.rc.K_ca * G < 0.f) D += M.rc.K_ca;
    return D;
  };
  // x <- L(D(x))^-1 x over one sub-step (warp 0); the incoming state goes to gxp for the reverse sweep
  auto implicit_fwd = [&](float* gxp) {
    const float xv = xs[lane];
    gxp[lane] = xv;
    float dd;
    const float dq = __shfl_down_sync(0xffffffffu, xv, 1) - xv;
    const float rup = lane == 31 ? 0.f : hstep * AN * Nf * face_D(Nf * dq, dd);
    float rdn = __shfl_up_sync(0xffffffffu, rup, 1);
    const float dqdn = __shfl_up_sync(0xffffffffu, dq, 1);
    if (lane == 0) rdn = 0.f;
    // incremental form: L (x' - x) = r_up (x_up - x) - r_dn (x - x_dn)
    xs[lane] = xv + pcr32(-rdn, 1.f + rdn + rup, -rup, rup * dq - rdn * dqdn);
  };

  // one Runge–Kutta step from xs (in place); the record of stage i goes to g0 + i * FC1_REC
  auto rk_step = [&](float* g0, float* gxp) {
    float* y = recs + FC1_Y;
    if (implicit) {
      if (t < 32) implicit_fwd(gxp);
      __syncwarp();
    }
    for (int i = 0; i < ns; ++i) {
      float* g = g0 + (size_t)i * FC1_REC;
      if (t < 32) {
        float yv = 0.f;
        for (int j = 0; j < i; ++j) yv = fmaf(tab.a[i][j], ks[j * 32 + t], yv);
        yv = fmaf(hstep, yv, xs[t]);
        y[t] = yv;
        g[FC1_Y + t] = yv;
      }
      __syncthreads();
      mlp_forward(y, g);
      if (t < 32) ks[i * 32 + t] = tendency(y);
      __syncwarp();
    }
    if (t < 32) {
      float acc = 0.f;
      for (int i = 0; i < ns; ++i) acc = fmaf(tab.b[i], ks[i * 32 + t], acc);
      xs[t] = fmaf(hstep, acc, xs[t]);
    }
    __syncthreads();
  };

  // ---- forward pass; every stage record goes to HBM ---------------------------------------------------------------------------
  float* grec = a.records + (size_t)col * a.n_sub * ns * FC1_REC;
  float* gxp0 = implicit ? a.xp + (size_t)col * a.n_sub * 32 : nullptr;
  for (int r = 0; r < a.n_sub; ++r) rk_step(grec + (size_t)r * ns * FC1_REC, implicit ? gxp0 + (size_t)r * 32 : nullptr);
  __threadfence();  // the records are read back by other threads of this CTA through cp.async (L2)

  // ---- reverse sweep -------------------------------------------------------------------------------------------------------
  auto frame_of = [&](int step) -> int {
    if (tm.save_stride <= 0) return step == tm.n_steps ? 0 : -1;
    return (step % tm.save_stride == 0) ? step / tm.save_stride : -1;
  };
  float sse = 0.f;
  auto loss_frame = [&](const float* __restrict__ x, int fr) {  // warp 0
    if (a.cot != nullptr) {
      xbar[lane] += __ldg(a.cot + ((size_t)col * a.n_saved + fr) * 32 + lane);
      return;
    }
    const float d = x[lane] - __ldg(a.targets + ((size_t)col * a.n_saved + fr) * 32 + lane);
    sse = fmaf(d, d, sse);
    xbar[lane] += a.wT * 2.f * a.inv_prof * d;
  };
  float acc1[8], acc2[32], acc3[8], db1 = 0.f, db2 = 0.f, db3 = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) { acc1[i] = 0.f; acc3[i] = 0.f; }
#pragma unroll
  for (int i = 0; i < 32; ++i) acc2[i] = 0.f;

  if (t < 32) {
    const int fr = frame_of(tm.n_steps);
    if (fr >= 0) loss_frame(xs, fr);
  }
  // records of sub-step r -> buffer b (16-byte cp.async; the records were written by this CTA: visible after the barrier)
  const int rec4 = ns * FC1_REC / 4;  // float4 per sub-step
  auto prefetch = [&](int r, int b) {
    const float4* src = reinterpret_cast<const float4*>(grec + (size_t)r * ns * FC1_REC);
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(recs + (size_t)b * ns * FC1_REC);
    for (int i4 = t; i4 < rec4; i4 += FC1_NT)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * i4), "l"(src + i4) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  __syncthreads();
  if (a.n_sub > 0) prefetch(a.n_sub - 1, 0);
  float xp_next = (implicit && t < 32 && a.n_sub > 0) ? gxp0[(size_t)(a.n_sub - 1) * 32 + t] : 0.f;  // written by this thread
  {
    for (int r = a.n_sub - 1; r >= 0; --r) {
      const int b = (a.n_sub - 1 - r) & 1;
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      __syncthreads();  // buffer b complete for every thread; nobody still reads buffer b ^ 1
      if (r > 0) prefetch(r - 1, b ^ 1);
      const float* rb = recs + (size_t)b * ns * FC1_REC;
      const float xp_cur = xp_next;
      if (implicit && t < 32 && r > 0) xp_next = gxp0[(size_t)(r - 1) * 32 + t];  // in flight during this sub-step's stages
      for (int i = ns - 1; i >= 0; --i) {
        const float* rec = rb + i * FC1_REC;
        const float* y = rec + FC1_Y;
        // B0 (warp 0): kbar_i, cotangent of the face fluxes = delta3, direct part of Ybar_i through the diffusive flux
        if (t < 32) {
          float kb = tab.b[i] * xbar[t];
          for (int j = i + 1; j < ns; ++j) kb = fmaf(tab.a[j][i], yb[j * 32 + t], kb);
          kb *= hstep;
          const float kbm = __shfl_up_sync(0xffffffffu, kb, 1);
          float Fb = 0.f, Gb = 0.f;  // face lane (>= 1)
          if (lane >= 1) {
            Fb = -AN * (kbm - kb);
            const float G = Nf * (y[lane] - y[lane - 1]);
            float dFdG = 0.f;
            if (mpp_e) { float dc; const float c = fc_mpp_cnu(M, G, &dc); dFdG -= fmaf(G, dc, c); }
            if (ca_e && M.rc.K_ca * G < 0.f) dFdG -= M.rc.K_ca;
            Gb = Fb * dFdG;
            d3s[lane - 1] = Fb;
          } else {
            d3s[31] = 0.f;
          }
          float Gbu = __shfl_down_sync(0xffffffffu, Gb, 1);
          if (lane == 31) Gbu = 0.f;
          yb[i * 32 + t] = Nf * (Gb - Gbu);
        }
        __syncthreads();
        // B1: dW3 += a2 d3^T, db3; abar2 = W3 d3
        {
          const float d3 = d3s[o32];
          const float* av = rec + FC1_A2 + 8 * kq16;
#pragma unroll
          for (int q = 0; q < 8; ++q) acc3[q] = fmaf(av[q], d3, acc3[q]);
          if (t < 31) db3 += d3s[t];
          // row k = o128 of W3 over the outputs (8 kq4 + q + k) mod 32: the row-dependent rotation keeps the banks distinct
          const float* w = W3 + o128 * 32;
          float s0 = 0.f, s1 = 0.f;
#pragma unroll
          for (int q = 0; q < 8; q += 2) {
            const int oa = (8 * kq4 + q + o128) & 31, oc = (8 * kq4 + q + 1 + o128) & 31;
            s0 = fmaf(w[oa], d3s[oa], s0);
            s1 = fmaf(w[oc], d3s[oc], s1);
          }
          part[kq4 * 128 + o128] = s0 + s1;
        }
        __syncthreads();
        if (t < 128) {
          float d = 0.f;
          if (t < h2) d = ((part[t] + part[128 + t]) + (part[256 + t] + part[384 + t])) * act_grad(F.act2, rec[FC1_Z2 + t]);
          d2s[t] = d;
          db2 += d;
        }
        __syncthreads();
        // B3: dW2 += a1 d2^T; abar1 = W2 d2
        {
          const float d2 = d2s[o128];
          const float4* av = reinterpret_cast<const float4*>(rec + FC1_A1 + 32 * kq4);
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 v = av[q];
            acc2[4 * q] = fmaf(v.x, d2, acc2[4 * q]); acc2[4 * q + 1] = fmaf(v.y, d2, acc2[4 * q + 1]);
            acc2[4 * q + 2] = fmaf(v.z, d2, acc2[4 * q + 2]); acc2[4 * q + 3] = fmaf(v.w, d2, acc2[4 * q + 3]);
          }
          // row k = o128 of W2 over the outputs 32 kq4 + (q + lane) mod 32 (lane rotation: distinct banks at row stride 128)
          float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
          const float* w = W2 + o128 * 128 + 32 * kq4;
          const float* dv = d2s + 32 * kq4;
#pragma unroll
          for (int q = 0; q < 32; q += 4) {
            const int oa = (q + lane) & 31, ob = (q + 1 + lane) & 31, oc = (q + 2 + lane) & 31, od = (q + 3 + lane) & 31;
            s0 = fmaf(w[oa], dv[oa], s0); s1 = fmaf(w[ob], dv[ob], s1);
            s2 = fmaf(w[oc], dv[oc], s2); s3 = fmaf(w[od], dv[od], s3);
          }
          part[kq4 * 128 + o128] = (s0 + s1) + (s2 + s3);
        }
        __syncthreads();
        if (t < 128) {
          float d = 0.f;
          if (t < h1) d = ((part[t] + part[128 + t]) + (part[256 + t] + part[384 + t])) * act_grad(F.act1, rec[FC1_Z1 + t]);
          d1s[t] = d;
          db1 += d;
        }
        __syncthreads();
        // B5: dW1 += y d1^T; Ybar_i += W1 d1 (thread (k = t / 16, oq = t % 16): outputs oq, oq + 16, ...)
        {
          const float d1 = d1s[o128];
          const float* yv = y + 8 * kq4;
#pragma unroll
          for (int q = 0; q < 8; ++q) acc1[q] = fmaf(yv[q], d1, acc1[q]);
          const int k = t >> 4, oq = t & 15;
          const float* w = W1 + k * 128 + oq;
          float s = 0.f;
#pragma unroll
          for (int q = 0; q < 8; ++q) s = fmaf(w[16 * q], d1s[oq + 16 * q], s);
          s += __shfl_xor_sync(0xffffffffu, s, 8);
          s += __shfl_xor_sync(0xffffffffu, s, 4);
          s += __shfl_xor_sync(0xffffffffu, s, 2);
          s += __shfl_xor_sync(0xffffffffu, s, 1);
          if (oq == 0) yb[i * 32 + k] += s;
        }
        __syncthreads();
      }
      if (t < 32) {
        float s = xbar[t];
        for (int i = 0; i < ns; ++i) s += yb[i * 32 + t];
        xbar[t] = s;
        if (implicit) {
          // VJP of x' = L(D(x))^-1 x: L is symmetric, lambda = L^-1 xbar' with the same coefficients; cotangent of r at face
          // lane+1 is -(lambda_up - lambda)(x'_up - x'); through D(G) to the level differences of the incoming state x
          const float xq = rb[FC1_Y + lane];  // x' = the input of stage 0
          float dd;
          const float G = Nf * (__shfl_down_sync(0xffffffffu, xp_cur, 1) - xp_cur);
          const float rup = lane == 31 ? 0.f : hstep * AN * Nf * face_D(G, dd);
          float rdn = __shfl_up_sync(0xffffffffu, rup, 1);
          if (lane == 0) rdn = 0.f;
          const float lam = pcr32(-rdn, 1.f + rdn + rup, -rup, s);
          const float lup = __shfl_down_sync(0xffffffffu, lam, 1), xup = __shfl_down_sync(0xffffffffu, xq, 1);
          const float Gb = lane == 31 ? 0.f : -(lup - lam) * (xup - xq) * hstep * AN * Nf * dd;  // cotangent of G at face lane+1
          float Gdn = __shfl_up_sync(0xffffffffu, Gb, 1);
          if (lane == 0) Gdn = 0.f;
          xbar[t] = lam + Nf * (Gdn - Gb);
        }
        if (r % nsub == 0) {
          const int fr = frame_of(r / nsub);
          if (fr >= 0) {
            if (a.cot != nullptr) {
              xbar[lane] += __ldg(a.cot + ((size_t)col * a.n_saved + fr) * 32 + lane);
            } else if (implicit) {  // the saved frame is the state before the step's first implicit solve
              const float d = xp_cur - __ldg(a.targets + ((size_t)col * a.n_saved + fr) * 32 + lane);
              sse = fmaf(d, d, sse);
              xbar[lane] += a.wT * 2.f * a.inv_prof * d;
            } else {
              loss_frame(rb + FC1_Y, fr);  // the input of stage 0 is the sub-step's start state
            }
          }
        }
      }
    }
  }

  // ---- results --------------------------------------------------------------------------------------------------------------
  float* gp = a.gpart + (size_t)col * F.P;
  if (o128 < h1) {
#pragma unroll
    for (int q = 0; q < 8; ++q) gp[F.w_off[0] + (8 * kq4 + q) * h1 + o128] = acc1[q];
  }
  if (o128 < h2) {
#pragma unroll
    for (int q = 0; q < 32; ++q)
      if (32 * kq4 + q < h1) gp[F.w_off[1] + (32 * kq4 + q) * h2 + o128] = acc2[q];
  }
  if (o32 < 31) {
#pragma unroll
    for (int q = 0; q < 8; ++q)
      if (8 * kq16 + q < h2) gp[F.w_off[2] + (8 * kq16 + q) * 31 + o32] = acc3[q];
  }
  if (t < h1) gp[F.b_off[0] + t] = db1;
  if (t < h2) gp[F.b_off[1] + t] = db2;
  if (t < 31) gp[F.b_off[2] + t] = db3;
  if (t < 32) {
    for (int o = 16; o > 0; o >>= 1) sse += __shfl_xor_sync(0xffffffffu, sse, o);
    if (t < 8) a.lpart[(size_t)col * 8 + t] = t == 2 ? sse : 0.f;
    if (a.x0bar != nullptr) a.x0bar[(size_t)col * 32 + lane] = xbar[lane];
  }
}

// out[p] = sum over columns of gpart[col][p] (fixed order)
static __global__ void fc1_reduce_kernel(const float* __restrict__ gpart, int ncol, int P, float* __restrict__ out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  float s = 0.f;
  for (int c = 0; c < ncol; ++c) s += gpart[(size_t)c * P + p];
  out[p] = s;
}

}  // namespace cpz
