// Launchers implemented in the per-kernel translation units (compiled in parallel).
#pragma once
#include "cpz_internal.h"
#include "cpz_solve.cuh"
#include "cpz_adjoint.cuh"
#include "cpz_rhs_vjp.cuh"
#include "cpz_closure.cuh"
#include "cpz_closure_uvt.cuh"

namespace cpz {
int launch_solve(cpz_model* m, const SolveArgs& a);
int launch_flux(cpz_model* m, const SolveArgs& a);  // rhs_only == 2 on the FP32 kernel with the adjoint plan's face-flux rows
int launch_solve_tc(cpz_model* m, const SolveArgs& a);
bool solve_tc_eligible(cpz_model* m);
int launch_solve_nnfree(cpz_model* m, const SolveArgs& a);
int launch_solve_fc_tc(cpz_model* m, const SolveArgs& a);   // T-only nets on tcgen05; 1 = not eligible
bool closure_uses_tc(const cpz_model* m);  // NN-free u/v/T model; 1 = not eligible
// one line for cpz_model_describe: which forward kernel this model runs on and why
std::string tc_describe(const cpz_model* m);  // 1 = not eligible, use the SIMT kernel
int launch_adjoint(cpz_model* m, const AdjArgs& a, int grid);
// pullback of one RHS evaluation on the adjoint plan (cpz_k_rhs_vjp.cu): persistent grid, one gradient slab per CTA
int launch_rhs_vjp(cpz_model* m, const VjpArgs& a, int grid);
// tensor-core adjoint (cpz_k_adjoint_tc.cu): checkpointing forward solve + reverse sweep; leaves the summed gradient in
// m->b_red[0,P) and returns the per-tile squared-error sums (stride 8)
bool adjoint_tc_eligible(cpz_model* m, std::string* why);
int loss_grad_tc(cpz_model* m, const float* x0, const float* bcs, const float* Q, const float* targets, size_t ncol,
                 const float* loss_w, float inv_prof, float inv_grad, int n_saved, int n_ckpt, const float** lpart_out, int* n_lpart);
// 4-, 8- and 16-column-tile instantiations (cpz_k_small.cu, cpz_k_small8.cu, cpz_k_small16.cu); CT selects the plan
int launch_solve_small(cpz_model* m, const SolveArgs& a, int CT);
int launch_adjoint_small(cpz_model* m, const AdjArgs& a, int grid, int CT);
// column tile the training pass (checkpointing forward + adjoint) uses for `ncol` columns
int train_tile(const cpz_model* m, size_t ncol);
// small-batch T-only training pass, one CTA per column (cpz_k_fc1.cu)
bool fc1_eligible(const cpz_model* m, size_t ncol);
int loss_grad_fc1(cpz_model* m, const float* x0, const float* bcs, const float* targets, size_t ncol, float wT, float inv_prof,
                  int n_saved, const float** lpart_out);
int launch_closure(cpz_model* m, const ClosureD& cd, const ClosureArgs& a);
int launch_closure_uvt(cpz_model* m, const ClosureUvtD& cd, const ClosureUvtArgs& a);
int launch_closure_uvt_tc(cpz_model* m, const ClosureUvtD& cd, const ClosureUvtArgs& a);  // tcgen05 flavour (cpz_k_tc.cu); 1 = not eligible
int launch_reduce_slabs(cpz_model* m, const float* part, int n_slabs, int P, float* out);
int launch_pack_loss(cpz_model* m, const float* lpart, int n_slabs, int stride, float ncol, float* pack_tail);
int launch_finalize_loss(cpz_model* m, const float* pack_tail, const float* w6, float inv_prof, float inv_grad, float* loss_out);
int launch_loss_traj(cpz_model* m, const float* traj, const float* tgt, int ncol, int n_saved, int S, int Nz, int nf, float* lpart);
// counts non-finite values of rows [ncol] x [S] (row stride `stride` floats) into the context's device counter
int launch_check_finite(cpz_ctx* c, const float* p, size_t stride, int ncol, int S);
// host flavours: begin_host_call zeroes the per-call counter; report_nonfinite reads it (synchronises the stream) and
// returns CPZ_ERR_NONFINITE when the call produced non-finite values
int begin_host_call(cpz_ctx* c);
int report_nonfinite(cpz_ctx* c, const char* what);
int launch_scale(cpz_model* m, float* g, int P, const float* pack_tail);
int launch_adam(cpz_model* m, const float* g, float lr, float b1, float b2, float eps);
}  // namespace cpz
