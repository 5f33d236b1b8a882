// Tensor-core (tcgen05) forward solve: eligibility, weight image, launcher.
#include <algorithm>
#include <cstdio>
#include <cstdlib>

#include "cpz_launch.h"
#include "cpz_tc.cuh"
#include "cpz_nnfree.cuh"

namespace cpz {

// face-diffusivity mode and folded constants (see side_column in cpz_tc.cuh)
static void side_constants(const ModelD& M, int& side_mode, SideC& C) {
  const RhsC& rc = M.rc;
  const bool mpp = (M.flags & F_MPP) || M.variant == RHS_INFER;
  const bool ca = (M.flags & F_CA) != 0;
  side_mode = SIDE_NONE;
  if (mpp) side_mode = (M.variant == RHS_INFER && ca) ? ((M.flags & F_CA_LITERAL_U) ? SIDE_MPP_CA_U : SIDE_MPP_CA_T) : SIDE_MPP;
  else if (ca) side_mode = SIDE_CA_ONLY;
  const double Nf = rc.Nf, L2E = 1.4426950408889634;
  C.e = M.variant == RHS_TRAIN ? (float)(rc.eps / Nf) : 0.f;
  C.su2 = (float)((double)rc.sig_u * rc.sig_u); C.sv2 = (float)((double)rc.sig_v * rc.sig_v);
  C.k1 = (float)(2.0 * rc.inv_dRi * (rc.BzC / Nf) * L2E);
  C.k2 = (float)(2.0 * rc.inv_dRi * rc.Ric * L2E);
  C.a0 = (float)(Nf * rc.c[0] * rc.nu0); C.a1 = (float)(Nf * rc.c[0] * rc.nu_m);
  C.b0 = (float)(Nf * rc.c[1] * rc.nu0); C.b1 = (float)(Nf * rc.c[1] * rc.nu_m);
  C.t0 = (float)(Nf * rc.c[2] * rc.inv_Pr * rc.nu0); C.t1 = (float)(Nf * rc.c[2] * rc.inv_Pr * rc.nu_m);
  C.kap = (float)(Nf * rc.c[2] * rc.kappa);
}

// The tcgen05 kernel covers the production wind_mixing nets (wind_mixing/train_NDE.jl:103: three Chains
// Dense(96,h1,act) -> Dense(h1,h2,act) -> Dense(h2,31)) with 3*h1 <= 160 and h2 <= 32; everything else runs on the
// FP32 SIMT kernel (cpz_solve.cuh).
bool tc_plan(const cpz_model* m, TcD& T, std::string& why) {
  const cpz_model_desc& d = m->desc;
  if (d.n_fields != 3 || d.Nz != 32 || d.n_nets != 3) { why = "needs the u/v/T model with three nets at Nz = 32"; return false; }
  if (d.variant != CPZ_RHS_TRAIN && d.variant != CPZ_RHS_INFER) { why = "variant"; return false; }
  if (d.flags & (CPZ_FLAG_SMOOTH_NN | CPZ_FLAG_SMOOTH_RI)) { why = "smoothing filters"; return false; }
  const cpz_net_desc& n0 = d.nets[0];
  if (n0.n_layers != 3 || n0.sizes[0] != 96 || n0.sizes[3] != 31) { why = "net depth/shape"; return false; }
  for (int q = 1; q < 3; ++q) {
    const cpz_net_desc& n = d.nets[q];
    if (n.n_layers != 3) { why = "net depth"; return false; }
    for (int l = 0; l <= 3; ++l) if (n.sizes[l] != n0.sizes[l]) { why = "nets differ in shape"; return false; }
    for (int l = 0; l < 3; ++l) if (n.act[l] != n0.act[l]) { why = "nets differ in activation"; return false; }
  }
  if (n0.act[2] != CPZ_ACT_IDENTITY) { why = "output activation"; return false; }
  T = TcD{};
  T.h1 = n0.sizes[1]; T.h2 = n0.sizes[2]; T.nout = 31;
  T.act1 = n0.act[0]; T.act2 = n0.act[1]; T.act3 = n0.act[2];
  if (3 * T.h1 > 160 || T.h2 > 32 || T.h1 < 1 || T.h2 < 1) { why = "hidden widths outside 3*h1 <= 160, h2 <= 32"; return false; }
  T.n1b = 3 * T.h1 > 128 ? 3 * T.h1 - 128 : 0;
  // the H1 / H2 planes hold one net's units in K (h1 <= 53 <= 8 * TC_K2S): every K row a layer-2 / layer-3 chain reads
  T.k3_steps = T.h2 <= 24 ? 3 : 4;
  T.h1_rows = 8 * TC_K2S;
  T.h2_rows = 8 * T.k3_steps;
  const int K2 = 8 * TC_K2S, K3 = 8 * T.k3_steps;
  if (2 * K2 + 2 * K3 > 192) { why = "layer-2/3 stacks exceed the 192 free TMEM columns"; return false; }
  T.c_a2hi = 192; T.c_a2lo = 192 + K2; T.c_a3hi = 192 + 2 * K2; T.c_a3lo = 192 + 2 * K2 + K3;
  const ModelD& M = m->fwd.M;
  int found = 0;
  for (int i = 0; i < M.n_gemm; ++i) {
    const GemmD& g = M.gemm[i];
    if (g.net < 0 || g.net >= 3 || g.layer < 0 || g.layer >= 3) { why = "plan"; return false; }
    T.w_off[g.net][g.layer] = g.w_off; T.b_off[g.net][g.layer] = g.b_off;
    ++found;
  }
  if (found != 9) { why = "plan"; return false; }
  side_constants(M, T.side_mode, T.sc);
  const TcSmem L = tc_smem_layout(T, m->tab.n_stages);
  if ((size_t)L.total > m->ctx->smem_optin) { why = "shared memory"; return false; }
  return true;
}

std::string tc_describe(const cpz_model* m) {
  TcD T;
  std::string why;
  char line[512];
  if (getenv("CPZ_NO_TC") != nullptr) return "forward kernel: fp32-simt (CPZ_NO_TC set)\n";
  if (m->desc.n_nets == 0 && m->desc.n_fields == 3 && m->desc.Nz == 32 && m->desc.variant != CPZ_RHS_FREE_CONVECTION &&
      !(m->desc.flags & (CPZ_FLAG_SMOOTH_NN | CPZ_FLAG_SMOOTH_RI)))
    return "forward kernel: nn-free warp-per-columns (2 columns per warp, no block barriers)\n";
  if (m->desc.variant == CPZ_RHS_FREE_CONVECTION && closure_uses_tc(m) && !(m->desc.flags & CPZ_FLAG_IMPLICIT_DIFFUSION))
    return "forward kernel: tcgen05 3xTF32, columns on the M side (128-column tiles, activations in TMEM, weights in shared memory)\n";
  if (!tc_plan(m, T, why)) return "forward kernel: fp32-simt (tcgen05 path not eligible: " + why + ")\n";
  const TcSmem L = tc_smem_layout(T, m->tab.n_stages);
  snprintf(line, sizeof(line),
           "forward kernel: tcgen05 3xTF32 (weights in TMEM; %d column groups x %d columns, %d threads; layer-1 rows %d+%d, "
           "layer-2 %d K steps, layer-3 %d K steps, the three nets in one N=48 chain; MMAs per RHS and group %d; smem %d B)\n",
           TC_NG, TC_GN, TC_NT, 3 * T.h1 - T.n1b, T.n1b, TC_K2S, T.k3_steps,
           36 * (T.n1b > 0 ? 2 : 1) + 3 * TC_K2S + 3 * T.k3_steps, L.total);
  return line;
}

template <int ACT, int K3S>
static int launch_tc_t(cpz_model* m, const TcD& T, const SolveArgs& a, const TcArgs& ta) {
  const TcSmem L = tc_smem_layout(T, m->tab.n_stages);
  // 28-column tiles (7 real columns per thread) when that does not add a wave: 4 096 columns then make 147 CTAs instead
  // of 128 and use every SM; checkpointing solves keep the adjoint's 32-column tile layout
  const int sms = m->ctx->sm_count > 0 ? m->ctx->sm_count : 148;
  const int t32 = (a.ncol + 31) / 32, t28 = (a.ncol + 27) / 28;
  const bool aux = a.aux.x != nullptr;  // segment pass of the tensor-core adjoint
  const bool seven = !aux && !((m->desc.flags & CPZ_FLAG_IMPLICIT_DIFFUSION) != 0 && !a.rhs_only) && a.ckpt == nullptr && getenv("CPZ_TC_CPT8") == nullptr && (t28 + sms - 1) / sms <= (t32 + sms - 1) / sms && t28 > t32;
  auto kern = a.rhs_only ? (seven ? solve_tc_kernel<ACT, K3S, false, true, 7> : solve_tc_kernel<ACT, K3S, false, true, 8>)
                         : (seven ? solve_tc_kernel<ACT, K3S, false, false, 7> : solve_tc_kernel<ACT, K3S, false, false, 8>);
  if (aux) kern = solve_tc_kernel<ACT, K3S, false, false, 8, true>;
  const bool impl = (m->desc.flags & CPZ_FLAG_IMPLICIT_DIFFUSION) != 0 && !a.rhs_only;
  if (impl) kern = aux ? solve_tc_kernel<ACT, K3S, false, false, 8, true, true> : solve_tc_kernel<ACT, K3S, false, false, 8, false, true>;
  CPZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total));
  const int n_tiles = (seven ? t28 : t32) * ((aux && a.split) ? 2 : 1);  // split segment pass: two CTAs per tile
  if (getenv("CPZ_TC_PROF") != nullptr && !a.rhs_only && !seven && !aux && !(m->desc.flags & CPZ_FLAG_IMPLICIT_DIFFUSION)) {  // debug: per-phase cycle counters of CTA 0
    auto pk = solve_tc_kernel<ACT, K3S, true>;
    CPZ_CUDA(cudaFuncSetAttribute(pk, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total));
    SolveArgs ap = a;
    unsigned long long* dcnt = nullptr;
    CPZ_CUDA(cudaMalloc(&dcnt, 224 * sizeof(unsigned long long)));
    CPZ_CUDA(cudaMemsetAsync(dcnt, 0, 224 * sizeof(unsigned long long), m->ctx->stream));
    ap.prof = dcnt;
    pk<<<n_tiles, TC_NT, L.total, m->ctx->stream>>>(m->fwd.M, T, m->tab, m->tm, ap, ta);
    unsigned long long hc[32 + 192];
    CPZ_CUDA(cudaMemcpyAsync(hc, dcnt, sizeof(hc), cudaMemcpyDeviceToHost, m->ctx->stream));
    CPZ_CUDA(cudaStreamSynchronize(m->ctx->stream));
    cudaFree(dcnt);
    const double nr = (double)m->tm.n_steps * m->tm.n_substeps * m->tab.n_stages;
    double tot = 0;
    for (int i = 0; i < 8; ++i) tot += hc[i] / nr;
    fprintf(stderr, "[cpz tc prof] warp 0 E1 detail: tmem ld %.0f | act+stores %.0f | fences %.0f | bar2 wait %.0f\n", hc[12] / nr, hc[13] / nr, hc[14] / nr, hc[2] / nr);
    fprintf(stderr, "[cpz tc prof] cycles per RHS (warp 0): bar1 %.0f | wait L1 %.0f | E1+bar %.0f | wait L2 %.0f | E2+bar %.0f | wait L3 %.0f | "
            "E3+stencil %.0f | RK+writeX %.0f | total %.0f || quadrant-3 warp: issue L1 %.0f faces %.0f wait L1 %.0f E1 x2 %.0f\n",
            hc[0] / nr, hc[1] / nr, hc[2] / nr, hc[3] / nr, hc[4] / nr, hc[5] / nr, hc[6] / nr, hc[7] / nr, tot, hc[8] / nr, hc[9] / nr,
            hc[10] / nr, hc[11] / nr);
    fprintf(stderr, "[cpz tc prof] RHS start clocks, group0 (delta to previous) / group1 - group0:");
    for (int i = 1; i < 96; i += 5) fprintf(stderr, " %lld/%lld", (long long)(hc[32 + 2 * i] - hc[32 + 2 * i - 2]), (long long)(hc[33 + 2 * i] - hc[32 + 2 * i]));
    fprintf(stderr, "\n");
    m->ctx->launches++;
    return CPZ_OK;
  }
  kern<<<n_tiles, TC_NT, L.total, m->ctx->stream>>>(m->fwd.M, T, m->tab, m->tm, a, ta);
  CPZ_CUDA(cudaGetLastError());
  m->ctx->launches++;
  return CPZ_OK;
}

// NN-free u/v/T model (`DE`): warp-per-columns kernel without block barriers. 1 = not eligible.
int launch_solve_nnfree(cpz_model* m, const SolveArgs& a) {
  const cpz_model_desc& d = m->desc;
  if (getenv("CPZ_NO_TC") != nullptr) return 1;
  if (d.n_nets != 0 || d.n_fields != 3 || d.Nz != 32) return 1;
  if (d.variant != CPZ_RHS_TRAIN && d.variant != CPZ_RHS_INFER) return 1;
  if (d.flags & (CPZ_FLAG_SMOOTH_NN | CPZ_FLAG_SMOOTH_RI)) return 1;
  SideC sc; int mode;
  side_constants(m->fwd.M, mode, sc);
  // 2 columns per warp keep every SM busy at a few thousand columns; 4 amortise the per-warp overhead at large batches
  const int NC = (getenv("CPZ_NNFREE_NC") ? atoi(getenv("CPZ_NNFREE_NC")) : (a.ncol >= 32768 ? 4 : 2));
  const int warps = ((a.ckpt != nullptr ? ((a.ncol + 31) & ~31) : a.ncol) + NC - 1) / NC;
  const int grid = (warps + NF_WARPS - 1) / NF_WARPS;
  const size_t smem = (size_t)m->tab.n_stages * NF_WARPS * 32 * 3 * NC * sizeof(float);
  if (NC == 4) solve_nnfree_kernel<4><<<grid, NF_WARPS * 32, smem, m->ctx->stream>>>(m->fwd.M, sc, mode, m->tab, m->tm, a);
  else solve_nnfree_kernel<2><<<grid, NF_WARPS * 32, smem, m->ctx->stream>>>(m->fwd.M, sc, mode, m->tab, m->tm, a);
  CPZ_CUDA(cudaGetLastError());
  m->ctx->launches++;
  return CPZ_OK;
}

// u/v/T closure step on the tcgen05 kernel (CLOSURE instantiation): the MLP evaluation is solve_tc_kernel's, the implicit mPP
// step its cyclic reduction; the face diffusivities are evaluated in the model's scaled variables with constants rebuilt for
// the closure (no eps, kappa_ca, the closure's own dz). 1 = not eligible (the FP32 SIMT kernel takes it).
template <int ACT, int K3S>
static int launch_closure_tc_t(cpz_model* m, const ModelD& M2, const TcD& T, const TcArgs& ta, int grid) {
  const TcSmem L = tc_smem_layout(T, m->tab.n_stages);
  auto kern = solve_tc_kernel<ACT, K3S, false, false, 8, false, false, true>;
  CPZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total));
  SolveArgs a{};
  a.theta = m->d_theta;
  kern<<<grid, TC_NT, L.total, m->ctx->stream>>>(M2, T, m->tab, m->tm, a, ta);
  CPZ_CUDA(cudaGetLastError());
  m->ctx->launches++;
  return CPZ_OK;
}

int launch_closure_uvt_tc(cpz_model* m, const ClosureUvtD& cd, const ClosureUvtArgs& ca) {
  if (getenv("CPZ_NO_TC") != nullptr) return 1;
  TcD T;
  std::string why;
  if (!tc_plan(m, T, why)) return 1;
  // the model description with the closure's rules: inference-style Richardson number (no eps), mPP always on, the
  // convective-adjustment switch on dT/dz with kappa_ca, B_z built from the closure's own dz
  ModelD M2 = m->fwd.M;
  M2.variant = RHS_INFER;
  M2.flags = F_MPP | (cd.ca ? F_CA : 0);
  M2.rc.kappa = cd.kappa_ca;
  M2.rc.BzC = (float)((double)cd.g_alpha * (double)cd.sig[2] * (double)M2.rc.Nf / (double)cd.inv_dz);
  M2.rc.nu0 = cd.nu0; M2.rc.nu_m = cd.nu_m; M2.rc.Ric = cd.Ric; M2.rc.inv_dRi = cd.inv_dRi; M2.rc.inv_Pr = cd.inv_Pr;
  side_constants(M2, T.side_mode, T.sc);
  const size_t need = (size_t)TC_WCOLS * 128;
  if (m->b_wimg.cap < need) {
    if (m->b_wimg.p) cudaFree(m->b_wimg.p);
    m->b_wimg.p = nullptr; m->b_wimg.cap = 0;
    CPZ_CUDA(cudaMalloc(&m->b_wimg.p, need * sizeof(float)));
    m->b_wimg.cap = need;
    m->wimg_ver = 0;
  }
  if (m->wimg_ver != m->theta_ver || ca.theta != m->d_theta) {  // the image is a function of theta only: rebuilt when it changed
    tc_image_kernel<<<(int)((need + 255) / 256), 256, 0, m->ctx->stream>>>(T, ca.theta, m->b_wimg.p);
    CPZ_CUDA(cudaGetLastError());
    m->ctx->launches++;
    m->wimg_ver = ca.theta == m->d_theta ? m->theta_ver : 0;
  }
  TcArgs ta{};
  const char* cstg = getenv("CPZ_TC_CL_STAGGER");
  ta.wimg = m->b_wimg.p; ta.stagger_ns = cstg ? atoi(cstg) : 0;
  TcClosure& C = ta.cl;
  for (int q = 0; q < 3; ++q) { C.f[q] = ca.f[q]; C.top[q] = cd.top[q]; C.inv_sig[q] = cd.inv_sig[q]; }
  for (int i = 0; i < 6; ++i) { C.mu[i] = cd.mu[i]; C.sig[i] = cd.sig[i]; }
  C.dzf = ca.dzf; C.out = ca.out; C.ncol = ca.ncol; C.n_tiles = (ca.ncol + TC_CT - 1) / TC_CT;
  C.inv_dz = cd.inv_dz;
  // hsub A_q N (N c_q nu) = hsub tau N^2 nu / H^2 must equal dt nu / dz^2 = cd.r nu
  const double H = m->desc.H, tau = m->desc.tau, N = M2.rc.Nf;
  C.hsub = (float)((double)cd.r * H * H / (tau * N * N));
  const int sms = m->ctx->sm_count > 0 ? m->ctx->sm_count : 148;
  const int grid = std::min(C.n_tiles, sms);
  const bool k3 = T.k3_steps == 3;
  if (T.act1 == T.act2 && T.act1 == ACT_MISH) return k3 ? launch_closure_tc_t<ACT_MISH, 3>(m, M2, T, ta, grid) : launch_closure_tc_t<ACT_MISH, 4>(m, M2, T, ta, grid);
  if (T.act1 == T.act2 && T.act1 == ACT_RELU) return k3 ? launch_closure_tc_t<ACT_RELU, 3>(m, M2, T, ta, grid) : launch_closure_tc_t<ACT_RELU, 4>(m, M2, T, ta, grid);
  return k3 ? launch_closure_tc_t<-1, 3>(m, M2, T, ta, grid) : launch_closure_tc_t<-1, 4>(m, M2, T, ta, grid);
}

// true when launch_solve_tc would take a checkpointing solve of this model
bool solve_tc_eligible(cpz_model* m) {
  if (getenv("CPZ_NO_TC") != nullptr) return false;
  TcD T;
  std::string why;
  return tc_plan(m, T, why);
}

// returns 1 when the model is not eligible (caller falls back to the SIMT kernel), 0 on success, <0 on error
int launch_solve_tc(cpz_model* m, const SolveArgs& a) {
  if (getenv("CPZ_NO_TC") != nullptr) return 1;
  TcD T;
  std::string why;
  if (!tc_plan(m, T, why)) return 1;
  const size_t need = (size_t)TC_WCOLS * 128;
  if (m->b_wimg.cap < need) {
    if (m->b_wimg.p) cudaFree(m->b_wimg.p);
    m->b_wimg.p = nullptr; m->b_wimg.cap = 0;
    CPZ_CUDA(cudaMalloc(&m->b_wimg.p, need * sizeof(float)));
    m->b_wimg.cap = need;
    m->wimg_ver = 0;
  }
  if (m->wimg_ver != m->theta_ver || a.theta != m->d_theta) {  // the image is a function of theta only: rebuilt when it changed
    tc_image_kernel<<<(int)((need + 255) / 256), 256, 0, m->ctx->stream>>>(T, a.theta, m->b_wimg.p);
    CPZ_CUDA(cudaGetLastError());
    m->ctx->launches++;
    m->wimg_ver = a.theta == m->d_theta ? m->theta_ver : 0;
  }
  const char* stg = getenv("CPZ_TC_STAGGER");
  TcArgs ta{};
  ta.wimg = m->b_wimg.p; ta.stagger_ns = stg ? atoi(stg) : 1600;
  const bool k3 = T.k3_steps == 3;
  if (T.act1 == T.act2 && T.act1 == ACT_MISH) return k3 ? launch_tc_t<ACT_MISH, 3>(m, T, a, ta) : launch_tc_t<ACT_MISH, 4>(m, T, a, ta);
  if (T.act1 == T.act2 && T.act1 == ACT_RELU) return k3 ? launch_tc_t<ACT_RELU, 3>(m, T, a, ta) : launch_tc_t<ACT_RELU, 4>(m, T, a, ta);
  return k3 ? launch_tc_t<-1, 3>(m, T, a, ta) : launch_tc_t<-1, 4>(m, T, a, ta);
}

}  // namespace cpz
