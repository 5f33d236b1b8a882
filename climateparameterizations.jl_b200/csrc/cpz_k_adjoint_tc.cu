// Tensor-core adjoint (cpz_adjoint_tc.cuh): eligibility, buffers, and the per-segment launch sequence
//   segment forward pass (solve_tc_kernel<AUX>) -> adjoint_tc_kernel -> wgrad_tc_kernel,   last segment first.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "cpz_launch.h"
#include "cpz_adjoint_tc.cuh"

namespace cpz {

bool tc_plan(const cpz_model* m, TcD& T, std::string& why);  // cpz_k_tc.cu

static int ensure_buf(DevBuf& b, size_t floats) {
  if (floats <= b.cap) return CPZ_OK;
  if (b.p) CPZ_CUDA(cudaFree(b.p));
  b.p = nullptr; b.cap = 0;
  CPZ_CUDA(cudaMalloc(&b.p, std::max<size_t>(floats, 4) * sizeof(float)));
  b.cap = floats;
  return CPZ_OK;
}

// The tensor-core adjoint covers what the tcgen05 forward solve covers (implicit-diffusion step included), minus the
// mPP-parameter gradient. CPZ_NO_TC_ADJ=1 forces the FP32 SIMT adjoint for A/B runs.
bool adjoint_tc_eligible(cpz_model* m, std::string* why_out) {
  std::string why;
  TcD T;
  TcB B;
  bool ok = true;
  if (getenv("CPZ_NO_TC") != nullptr || getenv("CPZ_NO_TC_ADJ") != nullptr) { why = "disabled by CPZ_NO_TC / CPZ_NO_TC_ADJ"; ok = false; }
  else if (getenv("CPZ_PROF") != nullptr) { why = "CPZ_PROF profiles the FP32 kernels"; ok = false; }
  else if (!tc_plan(m, T, why)) ok = false;
  else if (!tc_bwd_plan(T, B)) { why = "transposed weight images exceed tensor memory"; ok = false; }
  else {
    const TcBSmem L = tc_bwd_smem_layout(B, m->tab.n_stages);
    AuxD A{};
    tc_aux_rows(T, A);
    const size_t wg_smem = (size_t)2 * 8 * (A.rx + 2 * A.r1 + 2 * A.r2 + A.r3) * 16 + 64;
    if ((size_t)L.total > m->ctx->smem_optin || wg_smem > m->ctx->smem_optin) { why = "shared memory"; ok = false; }
  }
  if (why_out) *why_out = why;
  return ok;
}

template <int ACT>
static int launch_reverse_t(cpz_model* m, const TcD& T, const TcB& B, const AdjTcArgs& aa, const TimeD& tm, int n_ctas, const WgradArgs& wa,
                            int wg_grid, size_t wg_smem, bool ref) {
  const TcBSmem L = tc_bwd_smem_layout(B, m->tab.n_stages);
  const bool impl = (m->desc.flags & CPZ_FLAG_IMPLICIT_DIFFUSION) != 0;
  auto kern = aa.cot != nullptr ? (impl ? adjoint_tc_kernel<ACT, true, true> : adjoint_tc_kernel<ACT, false, true>)
                                : (impl ? adjoint_tc_kernel<ACT, true, false> : adjoint_tc_kernel<ACT, false, false>);
  CPZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total));
  kern<<<n_ctas, TC_NT, L.total, m->ctx->stream>>>(m->fwd.M, T, B, m->tab, tm, aa);
  CPZ_CUDA(cudaGetLastError());
  m->ctx->launches++;
  if (ref) {
    const int n = (B.N1 + 2 * B.N2 + 96) * 128;
    wgrad_ref_kernel<ACT><<<(n + 127) / 128, 128, 0, m->ctx->stream>>>(T, B, wa);
  } else {
    auto wk = wgrad_tc_kernel<ACT>;
    CPZ_CUDA(cudaFuncSetAttribute(wk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wg_smem));
    wk<<<wg_grid, WG_NT, wg_smem, m->ctx->stream>>>(T, B, wa);
  }
  CPZ_CUDA(cudaGetLastError());
  m->ctx->launches++;
  return CPZ_OK;
}

// Forward solve with checkpoints, then the reverse sweep. The per-stage records X_i, z1, z2 of as many steps as the memory
// budget holds ("record segment": a multiple of ckpt_stride steps, all of them when they fit) are written by ONE forward
// launch — the checkpointing forward pass itself for the last record segment, a re-integration from a checkpoint for the
// earlier ones — and consumed by reverse launches of `rs` steps each (the d1..d3 records only live from a reverse launch to
// its weight-gradient launch). Budget: CPZ_ADJ_AUX_GB, default the free device memory minus 8 GB of head-room.
// On return m->b_red[0,P) holds the sum over the local columns of d(unnormalised loss)/dtheta and *lpart_out / *n_lpart the
// per-tile squared-error sums (stride 8).
int loss_grad_tc(cpz_model* m, const float* x0, const float* bcs, const float* Q, const float* targets, size_t ncol,
                 const float* loss_w, float inv_prof, float inv_grad, int n_saved, int n_ckpt, const float** lpart_out, int* n_lpart,
                 CotPair cp) {
  TcD T;
  TcB B;
  std::string why;
  if (!tc_plan(m, T, why) || !tc_bwd_plan(T, B)) return fail(CPZ_ERR_INVALID, "tensor-core adjoint not eligible: %s", why.c_str());
  cudaStream_t st = m->ctx->stream;
  const int P = (int)m->P, S = 96;
  const int n_tiles = ((int)ncol + 31) / 32;
  const TimeD tm_full = m->tm;
  const int cs = tm_full.ckpt_stride, ns = m->tab.n_stages, nsub = tm_full.n_substeps, n_steps = tm_full.n_steps;
  const int epst = nsub * ns;  // stage evaluations per step
  AuxD A{};
  tc_aux_rows(T, A);
  const size_t xz_rows = (size_t)A.rx + A.r1 + A.r2, d_rows = (size_t)A.r1 + A.r2 + A.r3;
  const bool implicit = (m->desc.flags & CPZ_FLAG_IMPLICIT_DIFFUSION) != 0;
  // floats per step: x / z records of every stage evaluation (+ the pre-implicit state of every sub-step), d records
  const size_t xp_step = implicit ? (size_t)n_tiles * nsub * A.rx * 32 : 0;
  const size_t xz_step = (size_t)n_tiles * epst * xz_rows * 32 + xp_step, d_step = (size_t)n_tiles * epst * d_rows * 32;
  int rc;
  if ((rc = ensure_buf(m->b_ckpt, (size_t)n_tiles * n_ckpt * S * 32))) return rc;
  if ((rc = ensure_buf(m->b_bwimg, (size_t)B.n_wcols * 128))) return rc;
  const bool ref = getenv("CPZ_WGRAD_REF") != nullptr;
  const int sms = m->ctx->sm_count > 0 ? m->ctx->sm_count : 148;
  // few tiles (config 3 on 4 or 8 GPUs: 72 / 36 tiles): one column group per CTA, two CTAs per tile, so that the forward
  // pass with records and the reverse sweep use twice the SMs and a group does not share its SM (CPZ_TC_SPLIT=0 disables)
  const char* split_env = getenv("CPZ_TC_SPLIT");
  const int split = (split_env ? atoi(split_env) != 0 : 2 * n_tiles <= sms) ? 1 : 0;
  const int n_ctas = n_tiles * (split ? 2 : 1);
  // reverse launches: as many steps as 4 GB of d records hold
  const int rs = (int)std::max<size_t>(1, std::min<size_t>((size_t)n_steps, ((size_t)1 << 30) / std::max<size_t>(d_step, 1)));
  const int wg_grid = ref ? 1 : (int)std::min<size_t>((size_t)sms, (size_t)n_tiles * epst);
  // [xbar: n_tiles*96*32][lpart: n_tiles*8][accumulator images: wg_grid*WG_COLS*128]
  const size_t f_xbar = (size_t)n_tiles * S * 32, f_lp = (size_t)n_ctas * 8, f_img = (size_t)wg_grid * WG_COLS * 128;
  if ((rc = ensure_buf(m->b_tcadj, f_xbar + f_lp + f_img))) return rc;
  // record segment length from the memory budget
  size_t budget;  // floats for the x / z records
  if (const char* gb = getenv("CPZ_ADJ_AUX_GB")) {
    budget = (size_t)(atof(gb) * 1e9 / sizeof(float));
  } else {
    size_t free_b = 0, total_b = 0;
    CPZ_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const size_t have = free_b + m->b_aux.cap * sizeof(float);
    const size_t keep = ((size_t)8 << 30) + (size_t)rs * d_step * sizeof(float);
    budget = have > keep ? (have - keep) / sizeof(float) : 0;
  }
  int seg_len = (int)std::min<size_t>((size_t)n_steps, budget / std::max<size_t>(xz_step, 1));
  if (seg_len < n_steps) seg_len = std::max(cs, seg_len / cs * cs);  // record segments start on checkpoints
  // boundaries: the LAST record segment is the longest one that fits (it costs no re-integration), the steps before it
  // are cut into segments of seg_len from the start; every boundary is a checkpointed step
  const int s_last = seg_len >= n_steps ? 0 : (n_steps - seg_len + cs - 1) / cs * cs;
  std::vector<int> bnd;
  for (int b = 0; b < s_last; b += seg_len) bnd.push_back(b);
  bnd.push_back(s_last);
  bnd.push_back(n_steps);
  const int nrseg = (int)bnd.size() - 1;
  {
    static int told_len = -1;
    if (getenv("CPZ_VERBOSE") != nullptr && told_len != seg_len) {
      told_len = seg_len;
      fprintf(stderr, "[cpz] tensor-core adjoint: %zu columns, stage records of %d of %d steps per forward launch (%.2f GB), %d record "
                      "segment(s), reverse launches of %d steps, %s\n", ncol, seg_len, n_steps, (double)seg_len * xz_step * 4e-9, nrseg, rs,
              split ? "one column group per CTA (two CTAs per tile)" : "two column groups per CTA");
    }
  }
  if ((rc = ensure_buf(m->b_aux, (size_t)seg_len * xz_step + (size_t)rs * d_step))) return rc;
  float* xbar = m->b_tcadj.p;
  float* lpart = xbar + f_xbar;
  float* img = lpart + f_lp;
  CPZ_CUDA(cudaMemsetAsync(lpart, 0, (f_lp + f_img) * sizeof(float), st));
  const size_t n_xz = (size_t)n_tiles * seg_len * epst, n_d = (size_t)n_tiles * rs * epst;  // records
  float* p = m->b_aux.p;
  A.x = p; p += n_xz * A.rx * 32;
  A.z1 = p; p += n_xz * A.r1 * 32;
  A.z2 = p; p += n_xz * A.r2 * 32;
  A.d1 = p; p += n_d * A.r1 * 32;
  A.d2 = p; p += n_d * A.r2 * 32;
  A.d3 = p; p += n_d * A.r3 * 32;
  A.xp = implicit ? p : nullptr;
  A.n_stages = ns;
  A.n_eval = seg_len * epst;
  A.n_eval_d = rs * epst;

  // (1) forward with checkpoints; it also writes the records of the last record segment
  SolveArgs fa{};
  fa.theta = m->d_theta; fa.x0 = x0; fa.bcs = bcs; fa.Q = Q; fa.traj = nullptr; fa.ckpt = m->b_ckpt.p;
  fa.ncol = (int)ncol; fa.n_saved = n_saved; fa.n_ckpt = n_ckpt; fa.rhs_only = 0;
  fa.aux = A;
  fa.aux.ev_skip = s_last * epst;
  fa.split = split;
  if ((rc = launch_solve_tc(m, fa))) return rc > 0 ? fail(CPZ_ERR_INVALID, "tcgen05 forward solve not eligible") : rc;

  tc_bwd_image_kernel<<<(B.n_wcols * 128 + 255) / 256, 256, 0, st>>>(T, B, m->d_theta, m->b_bwimg.p);
  CPZ_CUDA(cudaGetLastError());
  m->ctx->launches++;

  // (2) record segments, last first
  const size_t SL = (size_t)S * 32;
  const size_t wg_smem = (size_t)2 * 8 * (xz_rows + d_rows) * 16 + 64;
  for (int seg = nrseg - 1; seg >= 0; --seg) {
    const int a0 = bnd[seg], a1 = bnd[seg + 1];
    if (seg != nrseg - 1) {  // re-integrate [a0, a1) from the checkpoint at step a0
      SolveArgs sa{};
      sa.theta = m->d_theta; sa.x0 = x0; sa.bcs = bcs; sa.Q = Q; sa.traj = nullptr; sa.ckpt = nullptr;
      sa.ncol = (int)ncol; sa.n_saved = n_saved; sa.n_ckpt = 0; sa.rhs_only = 0;
      sa.x0_tile = m->b_ckpt.p + (size_t)(a0 / cs) * SL; sa.x0_tile_stride = (size_t)n_ckpt * SL;
      sa.aux = A;
      sa.aux.ev_skip = 0;
      sa.split = split;
      m->tm = tm_full;
      m->tm.step0 = tm_full.step0 + a0;
      m->tm.n_steps = a1 - a0;
      m->tm.save_stride = 0;
      rc = launch_solve_tc(m, sa);
      m->tm = tm_full;
      if (rc) return rc > 0 ? fail(CPZ_ERR_INVALID, "tcgen05 forward solve not eligible") : rc;
    }
    for (int n1 = a1; n1 > a0; n1 -= std::min(rs, n1 - a0)) {
      const int n0 = n1 - std::min(rs, n1 - a0);
      AdjTcArgs aa{};
      aa.wimg = m->b_bwimg.p; aa.theta = m->d_theta; aa.targets = targets; aa.cot = cp.cot;
      aa.x0bar = n0 == 0 ? cp.x0bar : nullptr;  // the launch that ends the reverse sweep at step 0
      aa.xN = m->b_ckpt.p + (size_t)(n_ckpt - 1) * SL; aa.xN_stride = (size_t)n_ckpt * SL;
      aa.xbar = xbar; aa.lpart = lpart; aa.aux = A;
      aa.aux.ev0 = (n0 - a0) * epst;
      aa.ncol = (int)ncol; aa.n_saved = n_saved; aa.first = n1 == n_steps ? 1 : 0;
      aa.seg_step0 = n0; aa.seg_steps = n1 - n0; aa.split = split;
      for (int q = 0; q < 6; ++q) aa.w[q] = loss_w[q];
      aa.inv_prof = inv_prof; aa.inv_grad = inv_grad;
      WgradArgs wa{};
      wa.aux = aa.aux; wa.n_tiles = n_tiles; wa.n_e = (n1 - n0) * epst; wa.part = img;
      const bool mish = T.act1 == T.act2 && T.act1 == ACT_MISH, relu = T.act1 == T.act2 && T.act1 == ACT_RELU;
      if (mish) rc = launch_reverse_t<ACT_MISH>(m, T, B, aa, tm_full, n_ctas, wa, wg_grid, wg_smem, ref);
      else if (relu) rc = launch_reverse_t<ACT_RELU>(m, T, B, aa, tm_full, n_ctas, wa, wg_grid, wg_smem, ref);
      else rc = launch_reverse_t<-1>(m, T, B, aa, tm_full, n_ctas, wa, wg_grid, wg_smem, ref);
      if (rc) return rc;
    }
  }
  // (3) gradient in destructure order
  wgrad_finish_kernel<<<(P + 255) / 256, 256, 0, st>>>(T, B, img, wg_grid, P, m->b_red.p);
  CPZ_CUDA(cudaGetLastError());
  m->ctx->launches++;
  *lpart_out = lpart;
  *n_lpart = n_ctas;
  return CPZ_OK;
}

}  // namespace cpz
