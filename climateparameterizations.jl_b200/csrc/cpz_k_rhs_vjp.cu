// RHS pullback kernel instantiations (rhs_vjp_kernel, cpz_rhs_vjp.cuh) and their launcher.
#include "cpz_launch.h"

namespace cpz {

template <bool WS>
static int launch_rhs_vjp_t(cpz_model* m, const VjpArgs& a, int grid) {
  constexpr int CT = 32, NT = 256;
  const AdjSmem L = adjoint_smem_layout(m->bwd.M, CT);  // the adjoint plan was built to fit this layout
  const size_t smem = (size_t)L.total_floats * sizeof(float);
  if (smem > m->ctx->smem_optin) return fail(CPZ_ERR_INVALID, "rhs_vjp kernel needs %zu B shared memory, device allows %zu", smem, m->ctx->smem_optin);
  auto kern = rhs_vjp_kernel<CT, NT, WS>;
  CPZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, NT, smem, m->ctx->stream>>>(m->bwd.M, a);
  CPZ_CUDA(cudaGetLastError());
  m->ctx->launches++;
  return CPZ_OK;
}

int launch_rhs_vjp(cpz_model* m, const VjpArgs& a, int grid) {
  if (!m->has_bwd) return fail(CPZ_ERR_INVALID, "rhs_vjp needs the adjoint plan: %s", m->bwd_err.c_str());
  return m->bwd.M.w_in_smem ? launch_rhs_vjp_t<true>(m, a, grid) : launch_rhs_vjp_t<false>(m, a, grid);
}

}  // namespace cpz
