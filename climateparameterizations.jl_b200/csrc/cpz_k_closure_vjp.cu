// Gyre closure-step pullback kernel instantiations (closure_vjp_kernel, cpz_closure_vjp.cuh) and their launcher.
#include "cpz_launch.h"
#include "cpz_closure_vjp.cuh"

namespace cpz {

template <bool WS>
static int launch_closure_vjp_t(cpz_model* m, const ClosureD& cd, const ClosureVjpArgs& a, int grid) {
  constexpr int CT = 32, NT = 256;
  const AdjSmem L = adjoint_smem_layout(m->bwd.M, CT);  // the adjoint plan was built to fit this layout
  const size_t smem = (size_t)L.total_floats * sizeof(float);
  if (smem > m->ctx->smem_optin) return fail(CPZ_ERR_INVALID, "closure_vjp kernel needs %zu B shared memory, device allows %zu", smem, m->ctx->smem_optin);
  auto kern = closure_vjp_kernel<CT, NT, WS>;
  CPZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, NT, smem, m->ctx->stream>>>(m->bwd.M, cd, a);
  CPZ_CUDA(cudaGetLastError());
  m->ctx->launches++;
  return CPZ_OK;
}

int launch_closure_vjp(cpz_model* m, const ClosureD& cd, const ClosureVjpArgs& a, int grid) {
  if (!m->has_bwd) return fail(CPZ_ERR_INVALID, "adjoint plan unavailable: %s", m->bwd_err.c_str());
  const ModelD& M = m->bwd.M;
  // the Thomas scratch lives in the activation arena and zarena, which are adjacent in adjoint_smem_layout
  if (M.arena_floats + M.flux_off < closure_vjp_scratch_rows(M.Nz))
    return fail(CPZ_ERR_INVALID, "closure_vjp: the adjoint plan's activation arena (%d rows) is smaller than the %d rows of the Thomas scratch",
                M.arena_floats + M.flux_off, closure_vjp_scratch_rows(M.Nz));
  return M.w_in_smem ? launch_closure_vjp_t<true>(m, cd, a, grid) : launch_closure_vjp_t<false>(m, cd, a, grid);
}

}  // namespace cpz
