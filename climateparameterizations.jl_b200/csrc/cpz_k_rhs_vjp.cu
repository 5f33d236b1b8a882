// RHS pullback kernel instantiations (rhs_vjp_kernel, cpz_rhs_vjp.cuh) and their launcher.
#include "cpz_adjoint_launch.h"

namespace cpz {

int launch_rhs_vjp(cpz_model* m, const VjpArgs& a, int grid) {
  return launch_vjp_t(m, rhs_vjp_kernel<VJP_CT, VJP_NT, true>, rhs_vjp_kernel<VJP_CT, VJP_NT, false>, "rhs_vjp", 0, grid, a);
}

}  // namespace cpz
