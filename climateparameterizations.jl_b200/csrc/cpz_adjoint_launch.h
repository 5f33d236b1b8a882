// Launcher of adjoint_kernel<CT,NT,WS,COT> shared by the 32-column (cpz_k_adjoint.cu) and small-tile (cpz_k_small.cu) translation
// units, and of the single-evaluation pullbacks (cpz_k_rhs_vjp.cu, cpz_k_closure_vjp.cu, cpz_k_closure_uvt_vjp.cu).
#pragma once
#include <cstdio>
#include <cstdlib>

#include "cpz_launch.h"

namespace cpz {

template <int CT, int NT, bool WS>
static int launch_adjoint_t(cpz_model* m, const Plan& plan, const AdjArgs& a, int grid) {
  const AdjSmem L = adjoint_smem_layout(plan.M, CT);
  const size_t smem = (size_t)L.total_floats * sizeof(float);
  if (smem > m->ctx->smem_optin) return fail(CPZ_ERR_INVALID, "adjoint kernel needs %zu B shared memory, device allows %zu", smem, m->ctx->smem_optin);
  auto kern = a.cot != nullptr ? adjoint_kernel<CT, NT, WS, true> : adjoint_kernel<CT, NT, WS, false>;
  CPZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  static const bool prof = getenv("CPZ_PROF") != nullptr;
  if (prof) {
    AdjArgs ap = a;
    unsigned long long* d = nullptr;
    CPZ_CUDA(cudaMalloc(&d, 8 * sizeof(unsigned long long)));
    CPZ_CUDA(cudaMemsetAsync(d, 0, 8 * sizeof(unsigned long long), m->ctx->stream));
    ap.prof = d;
    kern<<<grid, NT, smem, m->ctx->stream>>>(plan.M, m->tab, m->tm, ap);
    unsigned long long hc[8];
    CPZ_CUDA(cudaMemcpyAsync(hc, d, sizeof(hc), cudaMemcpyDeviceToHost, m->ctx->stream));
    CPZ_CUDA(cudaStreamSynchronize(m->ctx->stream));
    cudaFree(d);
    const int tiles0 = (a.n_tiles + grid - 1) / grid;  // tiles processed by CTA 0
    const double nrk = (double)m->tm.n_steps * m->tm.n_substeps * tiles0, nst = nrk * m->tab.n_stages;
    fprintf(stderr, "[cpz prof adjoint] cycles per RK step: fwd-recompute(5 stages) %.0f | per reverse stage: combine+store %.0f mlp-fwd %.0f stencil-vjp %.0f bwd-L0 %.0f bwd-L1 %.0f bwd-L2+ %.0f\n",
            hc[0] / nrk, hc[1] / nst, hc[2] / nst, hc[3] / nst, hc[4] / nst, hc[5] / nst, hc[6] / nst);
    m->ctx->launches++;
    return CPZ_OK;
  }
  kern<<<grid, NT, smem, m->ctx->stream>>>(plan.M, m->tab, m->tm, a);
  CPZ_CUDA(cudaGetLastError());
  m->ctx->launches++;
  return CPZ_OK;
}

// Launcher of a single-evaluation pullback on the adjoint plan (VJP_NT threads, VJP_CT-column tiles, the caller has checked
// has_bwd): kern_ws / kern_wg are its instantiations with the weights in shared memory / streamed from global memory, taking
// the plan's ModelD and then `args`. scratch_rows: rows of the activation arena and zarena (adjacent in adjoint_smem_layout)
// that the kernel borrows as scratch outside the MLP.
template <class... Args>
static int launch_vjp_t(cpz_model* m, void (*kern_ws)(ModelD, Args...), void (*kern_wg)(ModelD, Args...), const char* name,
                        int scratch_rows, int grid, const Args&... args) {
  const ModelD& M = m->bwd.M;
  if (M.arena_floats + M.flux_off < scratch_rows)
    return fail(CPZ_ERR_INVALID, "%s: the adjoint plan's activation arena (%d rows) is smaller than the %d rows of the kernel's scratch",
                name, M.arena_floats + M.flux_off, scratch_rows);
  const AdjSmem L = adjoint_smem_layout(M, VJP_CT);  // the adjoint plan was built to fit this layout
  const size_t smem = (size_t)L.total_floats * sizeof(float);
  if (smem > m->ctx->smem_optin) return fail(CPZ_ERR_INVALID, "%s kernel needs %zu B shared memory, device allows %zu", name, smem, m->ctx->smem_optin);
  auto kern = M.w_in_smem ? kern_ws : kern_wg;
  CPZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, VJP_NT, smem, m->ctx->stream>>>(M, args...);
  CPZ_CUDA(cudaGetLastError());
  m->ctx->launches++;
  return CPZ_OK;
}

}  // namespace cpz
