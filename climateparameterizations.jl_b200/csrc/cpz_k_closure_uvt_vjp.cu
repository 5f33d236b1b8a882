// u/v/T closure-step pullback kernel instantiations (closure_uvt_vjp_kernel, cpz_closure_uvt_vjp.cuh) and their launcher.
#include "cpz_adjoint_launch.h"
#include "cpz_closure_uvt_vjp.cuh"

namespace cpz {

int launch_closure_uvt_vjp(cpz_model* m, const ClosureUvtD& cd, const ClosureUvtVjpArgs& a, int grid) {
  return launch_vjp_t(m, closure_uvt_vjp_kernel<VJP_CT, VJP_NT, true>, closure_uvt_vjp_kernel<VJP_CT, VJP_NT, false>,
                      "closure_uvt_vjp", closure_uvt_vjp_scratch_rows(m->bwd.M.Nz), grid, cd, a);
}

}  // namespace cpz
