// Gyre closure-step pullback kernel instantiations (closure_vjp_kernel, cpz_closure_vjp.cuh) and their launcher.
#include "cpz_adjoint_launch.h"
#include "cpz_closure_vjp.cuh"

namespace cpz {

int launch_closure_vjp(cpz_model* m, const ClosureD& cd, const ClosureVjpArgs& a, int grid) {
  return launch_vjp_t(m, closure_vjp_kernel<VJP_CT, VJP_NT, true>, closure_vjp_kernel<VJP_CT, VJP_NT, false>, "closure_vjp",
                      closure_vjp_scratch_rows(m->bwd.M.Nz), grid, cd, a);
}

}  // namespace cpz
