// Tangent kernel instantiations (rhs_jvp_kernel, solve_jvp_kernel, cpz_jvp.cuh) and their launchers.
#include "cpz_adjoint_launch.h"
#include "cpz_jvp.cuh"

namespace cpz {

int launch_rhs_jvp(cpz_model* m, const JvpArgs& a, int grid) {
  return launch_vjp_t(m, rhs_jvp_kernel<VJP_CT, VJP_NT, true>, rhs_jvp_kernel<VJP_CT, VJP_NT, false>, "rhs_jvp", 0, grid, a);
}

int launch_solve_jvp(cpz_model* m, const JvpArgs& a, int grid) {
  return launch_vjp_t(m, solve_jvp_kernel<VJP_CT, VJP_NT, true>, solve_jvp_kernel<VJP_CT, VJP_NT, false>, "solve_jvp", 0, grid,
                      m->tab, m->tm, a);
}

}  // namespace cpz
