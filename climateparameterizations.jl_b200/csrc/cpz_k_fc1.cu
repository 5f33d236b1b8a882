// Small-batch training pass of the T-only NDE (cpz_fc1.cuh): eligibility and launcher.
#include <algorithm>
#include <cstdlib>

#include "cpz_launch.h"
#include "cpz_fc1.cuh"

namespace cpz {

static int fc1_ensure(DevBuf& b, size_t floats) {
  if (floats <= b.cap) return CPZ_OK;
  if (b.p) CPZ_CUDA(cudaFree(b.p));
  b.p = nullptr; b.cap = 0;
  CPZ_CUDA(cudaMalloc(&b.p, std::max<size_t>(floats, 4) * sizeof(float)));
  b.cap = floats;
  return CPZ_OK;
}

static bool fc1_plan(const cpz_model* m, Fc1D& F) {
  const cpz_model_desc& d = m->desc;
  if (d.variant != CPZ_RHS_FREE_CONVECTION || d.n_fields != 1 || d.n_nets != 1 || d.Nz != 32) return false;
  if (d.flags & ~(uint32_t)(CPZ_FLAG_MPP | CPZ_FLAG_CA | CPZ_FLAG_IMPLICIT_DIFFUSION)) return false;  // constant boundary fluxes
  const cpz_net_desc& n = d.nets[0];
  if (n.n_layers != 3 || n.sizes[0] != 32 || n.sizes[3] != 31 || n.act[2] != CPZ_ACT_IDENTITY) return false;
  if (n.sizes[1] < 1 || n.sizes[1] > 128 || n.sizes[2] < 1 || n.sizes[2] > 128) return false;
  F = Fc1D{};
  F.h1 = n.sizes[1]; F.h2 = n.sizes[2]; F.act1 = n.act[0]; F.act2 = n.act[1];
  F.P = (int)m->P;
  const ModelD& M = m->fwd.M;
  int found = 0;
  for (int i = 0; i < M.n_gemm; ++i) {
    const GemmD& g = M.gemm[i];
    if (g.net != 0 || g.layer < 0 || g.layer > 2) return false;
    F.w_off[g.layer] = g.w_off; F.b_off[g.layer] = g.b_off; ++found;
  }
  return found == 3;
}

// One CTA per column pays off while the columns are too few to fill 32-column tiles on more than a handful of SMs;
// CPZ_FC1_MAX_NCOL overrides the limit (0 disables the path).
bool fc1_eligible(const cpz_model* m, size_t ncol) {
  const char* e = getenv("CPZ_FC1_MAX_NCOL");
  const size_t max_ncol = e ? (size_t)atoi(e) : 32;
  if (ncol == 0 || ncol > max_ncol) return false;
  if (getenv("CPZ_PROF") != nullptr) return false;  // the phase counters live in the tile kernels
  Fc1D F;
  if (!fc1_plan(m, F)) return false;
  if (m->tab.n_stages > CPZ_MAX_STAGES) return false;
  // stage records of the whole solve (config 1: 226 MB per column)
  if (ncol * (size_t)m->tm.n_steps * m->tm.n_substeps * m->tab.n_stages * FC1_REC * sizeof(float) > ((size_t)8 << 30)) return false;
  const Fc1Smem L = fc1_smem_layout(m->tab.n_stages);
  return (size_t)L.total_floats * sizeof(float) <= m->ctx->smem_optin;
}

// Leaves the sum over the columns of d(unnormalised loss)/dtheta in m->b_red[0,P) and returns the per-column squared-error
// sums (stride 8).
int loss_grad_fc1(cpz_model* m, const float* x0, const float* bcs, const float* targets, size_t ncol, float wT, float inv_prof,
                  int n_saved, const float** lpart_out, CotPair cp) {
  Fc1D F;
  if (!fc1_plan(m, F)) return fail(CPZ_ERR_INVALID, "single-column training kernel not eligible");
  const int P = F.P;
  const int n_sub = m->tm.n_steps * m->tm.n_substeps;
  int rc;
  if ((rc = fc1_ensure(m->b_ckpt, ncol * (size_t)n_sub * m->tab.n_stages * FC1_REC))) return rc;
  if ((rc = fc1_ensure(m->b_part, ncol * ((size_t)P + 8)))) return rc;
  const bool implicit = (m->desc.flags & CPZ_FLAG_IMPLICIT_DIFFUSION) != 0;
  if (implicit && (rc = fc1_ensure(m->b_scr, ncol * (size_t)n_sub * 32))) return rc;
  Fc1Args a{};
  a.theta = m->d_theta; a.x0 = x0; a.x0_stride = 0; a.bcs = bcs; a.targets = targets; a.cot = cp.cot; a.x0bar = cp.x0bar;
  a.records = m->b_ckpt.p; a.xp = implicit ? m->b_scr.p : nullptr; a.gpart = m->b_part.p; a.lpart = m->b_part.p + ncol * (size_t)P;
  a.ncol = (int)ncol; a.n_saved = n_saved; a.n_sub = n_sub; a.wT = wT; a.inv_prof = inv_prof;
  const Fc1Smem L = fc1_smem_layout(m->tab.n_stages);
  const size_t smem = (size_t)L.total_floats * sizeof(float);
  CPZ_CUDA(cudaFuncSetAttribute(fc1_train_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  fc1_train_kernel<<<(unsigned)ncol, FC1_NT, smem, m->ctx->stream>>>(m->fwd.M, F, m->tab, m->tm, a);
  CPZ_CUDA(cudaGetLastError());
  m->ctx->launches++;
  fc1_reduce_kernel<<<(P + 255) / 256, 256, 0, m->ctx->stream>>>(a.gpart, (int)ncol, P, m->b_red.p);
  CPZ_CUDA(cudaGetLastError());
  m->ctx->launches++;
  *lpart_out = a.lpart;
  return CPZ_OK;
}

}  // namespace cpz
