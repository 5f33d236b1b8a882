/*
 * cpz.h — C ABI of libcpz.so, the B200-native NDE column engine.
 *
 * This header is the drop-in boundary for the one hot path of
 * CliMA/ClimateParameterizations.jl (OceanParameterizations.jl): the batched
 * neural-differential-equation (NDE) column solve and its parameter gradient.
 * The reference has no FFI; each entry point below names the de-facto operator
 * seam (reference file:line, relative to the reference checkout) it replaces.
 * A Julia host reaches these through `ccall` (see INTEGRATION.md), the Python
 * host mirror through `ctypes`.
 *
 * Conventions
 *   - C linkage, POD arguments only. Every entry point returns 0 on success and
 *     a negative cpz_status otherwise; cpz_last_error() gives the message.
 *   - All arrays are float32. A batched state is [ncol][n_fields*Nz] with each
 *     column's profile contiguous (Julia Array{Float32,2} of size (nf*Nz, ncol));
 *     trajectories are [ncol][n_saved][n_fields*Nz] (Julia (nf*Nz, n_saved, ncol)).
 *     Index 0 of a profile is the bottom level, index Nz-1 the surface level.
 *   - Pointers passed to the host flavour are HOST pointers owned by the caller
 *     and only read/written during the call. The *_dev flavour takes DEVICE
 *     pointers on the context's device and enqueues on the context's stream
 *     without synchronising.
 *   - Handles are not thread-safe; one host thread drives one context.
 *   - There is no CPU fallback: every compute entry point fails with
 *     CPZ_ERR_CUDA when no sm_100-class device is usable.
 */
#ifndef CPZ_H
#define CPZ_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CPZ_VERSION_MAJOR 0
#define CPZ_VERSION_MINOR 1

#define CPZ_MAX_LAYERS 6
#define CPZ_MAX_NETS 3

typedef enum {
  CPZ_OK = 0,
  CPZ_ERR_INVALID = -1,   /* bad argument / unsupported configuration */
  CPZ_ERR_CUDA = -2,      /* CUDA runtime error, or no usable device   */
  CPZ_ERR_NONFINITE = -3, /* NaN/Inf detected in a result (IEEE semantics are kept, this only reports) */
  CPZ_ERR_COLLECTIVE = -4 /* the host-supplied allreduce hook failed   */
} cpz_status;

/* Right-hand-side variants (SURVEY §8a / Appendix A). */
typedef enum {
  /* wind_mixing/src/NDE_training.jl:83-165  predict_flux + predict_NDE (training RHS, eps on gradients) */
  CPZ_RHS_TRAIN = 0,
  /* wind_mixing/src/training_postprocessing.jl:55-153  solve_NDE_mutating's NDE! (inference RHS, no eps) */
  CPZ_RHS_INFER = 1,
  /* free_convection/src/free_convection_nde.jl:29-38 and convective_adjustment_nde.jl:33-48 (T-only) */
  CPZ_RHS_FREE_CONVECTION = 2
} cpz_rhs_variant;

/* Flags (bitmask in cpz_model_desc.flags). */
#define CPZ_FLAG_MPP              (1u << 0) /* modified Pacanowski–Philander diffusivity (NDE_training.jl:114-139); on the T-only
                                              * variant: the same rule at u = v = 0 (shear gradients 0 + eps), added to the NN
                                              * flux as -sigma_T/(sigma_wT H) nu/Pr dT/dz — BASELINE config 1 "CA + mPP base" */
#define CPZ_FLAG_CA               (1u << 1) /* convective adjustment (training_postprocessing.jl:118-124; convective_adjustment_nde.jl:44-47) */
#define CPZ_FLAG_ZERO_WEIGHTS     (1u << 2) /* conditions.zero_weights boundary handling (NDE_training.jl:104-112,129-133) */
#define CPZ_FLAG_SMOOTH_NN        (1u << 3) /* filters.interior on NN output (NDE_training.jl:98-102) */
#define CPZ_FLAG_SMOOTH_RI        (1u << 4) /* filters.face on Ri (NDE_training.jl:121-123) */
#define CPZ_FLAG_DIURNAL          (1u << 5) /* time-dependent wT_top (NDE_training.jl:68-81, data_containers.jl:135) */
#define CPZ_FLAG_CA_LITERAL_U     (1u << 6) /* CA switch tests du/dz>0 exactly as training_postprocessing.jl:120 (default tests dT/dz>0) */
#define CPZ_FLAG_IMPLICIT_DIFFUSION (1u << 8) /* the diffusive / convective-adjustment part of the flux is left out of the RHS and
                                               * applied by a backward-Euler tridiagonal solve (diffusivities of the incoming state)
                                               * at the start of every (sub-)step, the way the reference integrates inside Oceananigans
                                               * (modified_pacanowski_philander!, NDE_oceananigans.jl:61-101; convective_adjustment!,
                                               * oceananigans_nn.jl:13-40); the NN flux, Coriolis and boundary fluxes stay explicit.
                                               * Removes the stability sub-steps of explicit diffusion (SURVEY 8f-1). */
#define CPZ_FLAG_DIURNAL_UNSHIFTED (1u << 7) /* infer variant: diurnal top flux without the -s_wT(0) shift, as training_postprocessing.jl:142-144 */

/* Activations (Flux 0.11.6 / NNlib 0.7.20 definitions). */
typedef enum {
  CPZ_ACT_IDENTITY = 0,
  CPZ_ACT_RELU = 1,
  CPZ_ACT_MISH = 2,      /* x*tanh(softplus(x)) */
  CPZ_ACT_SWISH = 3,     /* x*sigmoid(x)        */
  CPZ_ACT_LEAKYRELU = 4, /* max(0.01x, x)       */
  CPZ_ACT_TANH = 5
} cpz_activation;

/* Fixed-step explicit integrators. TSIT5 is the tableau of OrdinaryDiffEq's Tsit5, the one
 * fixed-step call in the reference (free_convection/convective_adjustment.jl:137). */
typedef enum { CPZ_INT_EULER = 0, CPZ_INT_RK4 = 1, CPZ_INT_TSIT5 = 2 } cpz_integrator;

/* One Flux.Chain of Dense layers. Input is the full scaled state (n_fields*Nz),
 * output the Nz-1 interior faces. */
typedef struct {
  int32_t n_layers;                  /* number of Dense layers, 1..CPZ_MAX_LAYERS */
  int32_t sizes[CPZ_MAX_LAYERS + 1]; /* sizes[0]=input, sizes[n_layers]=output     */
  int32_t act[CPZ_MAX_LAYERS];       /* cpz_activation per layer                   */
} cpz_net_desc;

/* POD description of one NDE model; replaces the (constants, scalings, conditions, NN_sizes)
 * NamedTuples of prepare_parameters_NDE_training (NDE_training.jl:1-44) and the
 * FreeConvectionNDEParameters vector (free_convection_nde.jl:49-62). */
typedef struct {
  int32_t Nz;        /* levels, 4..64 (benchmarked at 32)              */
  int32_t n_fields;  /* 3 = (u,v,T) wind_mixing, 1 = T-only free_convection */
  int32_t variant;   /* cpz_rhs_variant                                */
  uint32_t flags;    /* CPZ_FLAG_*                                     */
  int32_t n_nets;    /* 0 (NN-free `DE`, diffusivity_parameter_optimisation.jl:1-33), 1 (T-only) or 3 (uw,vw,wT) */
  cpz_net_desc nets[CPZ_MAX_NETS];
  /* constants (NDE_training.jl:23-33) */
  float H, tau, f, g, alpha, nu0, nu_m, Ric, dRi, Pr, kappa, eps;
  /* ZeroMeanUnitVarianceScaling mu, sigma for u, v, T, uw, vw, wT (feature_scaling.jl:7-23) */
  float mu[6];
  float sigma[6];
  float K_ca;           /* T-only non-dimensional convective-adjustment K (convective_adjustment_nde.jl:45: 10) */
  float diurnal_period; /* seconds; data_containers.jl:135 uses 24*60^2 */
  /* time integration */
  int32_t integrator;   /* cpz_integrator */
  float dt;             /* non-dimensional length of one step (one saved-frame interval = 1/1152 in the reference data) */
  float t0;             /* non-dimensional start time */
  int32_t n_steps;      /* steps per solve */
  int32_t n_substeps;   /* integrator sub-steps inside each step (stability of explicit diffusion) */
  int32_t save_stride;  /* save every save_stride-th step (frame 0 = initial condition is always saved); 0 = final state only */
  int32_t ckpt_stride;  /* adjoint: checkpoint the state every ckpt_stride steps */
} cpz_model_desc;

typedef struct cpz_ctx cpz_ctx;
typedef struct cpz_model cpz_model;

/* Allreduce hook for data-parallel training: sum `n` floats in place in the DEVICE buffer `buf`
 * over all ranks, enqueued on `stream` (a cudaStream_t). Return 0 on success. The host (torch.distributed /
 * NCCL.jl) owns the communicator; the library never initialises one. */
typedef int (*cpz_allreduce_fn)(void* user, float* buf, size_t n, void* stream);

/* ---- context ------------------------------------------------------------------------------- */
int cpz_version(void);                                   /* major*100+minor */
const char* cpz_last_error(void);                        /* thread-local message of the last failure */
int cpz_device_count(int* n);                            /* usable CUDA devices (0 is not an error here) */
size_t cpz_sizeof_model_desc(void);                      /* sizeof(cpz_model_desc) the library was built with (ABI check) */
size_t cpz_sizeof_closure_desc(void);
/* Create a context on CUDA device `device`. `stream` is a cudaStream_t to enqueue on (e.g. torch's current
 * stream) or NULL for a library-owned non-blocking stream. */
int cpz_ctx_create(int device, void* stream, cpz_ctx** out);
int cpz_ctx_destroy(cpz_ctx* ctx);
int cpz_ctx_set_allreduce(cpz_ctx* ctx, cpz_allreduce_fn fn, void* user, int rank, int world_size);
int cpz_ctx_synchronize(cpz_ctx* ctx);
int cpz_ctx_stream(cpz_ctx* ctx, void** stream_out);     /* the cudaStream_t kernels are launched on */
/* CPZ_ERR_NONFINITE reporting. The host flavours of cpz_solve / cpz_loss_grad / cpz_train_step return CPZ_ERR_NONFINITE
 * (after writing their results as computed) when the final saved frame or the loss holds a NaN/Inf. The *_dev flavours
 * cannot (they do not synchronise): they add to a device counter that this call reads (it synchronises the stream). */
int cpz_ctx_nonfinite_count(cpz_ctx* ctx, uint64_t* n);
/* Number of library kernels launched on this context since creation (for gpu_launches accounting). */
int cpz_ctx_launch_count(cpz_ctx* ctx, uint64_t* n);

/* ---- model --------------------------------------------------------------------------------- */
/* replaces prepare_parameters_NDE_training (NDE_training.jl:1-44) / FreeConvectionNDE (free_convection_nde.jl:1-47) */
int cpz_model_create(cpz_ctx* ctx, const cpz_model_desc* desc, cpz_model** out);
int cpz_model_destroy(cpz_model* m);
int cpz_model_n_params(const cpz_model* m, size_t* P);   /* total length of theta = sum over nets */
int cpz_model_n_saved(const cpz_model* m, int32_t* n);   /* frames a solve writes per column */
/* theta in Flux.destructure order: per net, per layer [vec(W) column-major (out x in); b]
 * (NDE_training.jl:11-13,37; nets concatenated uw,vw,wT). HOST pointers. */
int cpz_set_theta(cpz_model* m, const float* theta, size_t P);
int cpz_get_theta(cpz_model* m, float* theta, size_t P);
/* human-readable plan (tile shapes, phases, shared-memory use) of the forward and adjoint kernels */
int cpz_model_describe(const cpz_model* m, char* buf, size_t buf_len);
/* change time-stepping fields (n_steps, n_substeps, dt, t0, save_stride, ckpt_stride, integrator) without rebuilding */
int cpz_model_set_time(cpz_model* m, int32_t integrator, float dt, float t0, int32_t n_steps, int32_t n_substeps,
                       int32_t save_stride, int32_t ckpt_stride);

/* ---- S1: RHS  f(x, p, t) -> dx ------------------------------------------------------------- */
/* replaces NDE(x,p,t,...) (NDE_training.jl:56-81), NDE! (training_postprocessing.jl:131-153),
 * dT/dt closures (free_convection_nde.jl:29-38, convective_adjustment_nde.jl:33-48).
 * x, dxdt: [ncol][nf*Nz]; bcs: [ncol][6] = (uw_b,uw_t,vw_b,vw_t,wT_b,wT_t) scaled, or [ncol][2] = (bottom,top) for T-only;
 * diurnal_Q: [ncol] buoyancy-flux amplitudes or NULL. */
int cpz_rhs(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, float* dxdt, size_t ncol);
int cpz_rhs_dev(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, float* dxdt, size_t ncol);

/* ---- S1 pullback: VJP of f(x, p, t) ------------------------------------------------------------ */
/* replaces the Zygote pullback of NDE that InterpolatingAdjoint(autojacvec=ZygoteVJP()) calls once per adjoint stage
 * (NDE_training.jl:291,304; free_convection/src/solve.jl:4-5), so that a host with its own time stepper (adaptive Tsit5 or
 * ROCK4, a continuous adjoint) can differentiate through cpz_rhs. With f_c = what cpz_rhs returns for column c on the same
 * inputs and ybar_c = dxdt_bar[c] ([ncol][nf*Nz]):
 *   x_bar[c]  = (df_c/dx_c)^T ybar_c                 [ncol][nf*Nz]
 *   theta_bar = sum_c (df_c/dtheta)^T ybar_c         [P], Flux.destructure order
 *   mpp_bar   = sum_c (df_c/dp)^T ybar_c             [5], p = (nu0, nu_m, dRi, Ric, Pr) unscaled, as cpz_loss_grad_mpp
 * Outputs are overwritten, not accumulated; each may be NULL, at least one must not be. theta_bar must be NULL when P = 0;
 * mpp_bar is refused where cpz_loss_grad_mpp refuses it. At relu kinks and the convective-adjustment switch the derivative
 * of the branch that was evaluated is taken. With CPZ_FLAG_IMPLICIT_DIFFUSION this is the pullback of the explicit part
 * cpz_rhs returns (mpp_bar = 0). The sums over columns are in a fixed order (bitwise reproducible); the allreduce hook is
 * not called (the sum over ranks is the host's) and there is no non-finite reporting. Needs the adjoint plan. */
int cpz_rhs_vjp(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, const float* dxdt_bar,
                float* x_bar, float* theta_bar, float* mpp_bar, size_t ncol);
int cpz_rhs_vjp_dev(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, const float* dxdt_bar,
                    float* x_bar, float* theta_bar, float* mpp_bar, size_t ncol);

/* total face fluxes of one RHS evaluation; replaces predict_flux (NDE_training.jl:83-147), predict_flux! (training_postprocessing.jl:
 * 105-128) and the per-frame wT reconstruction of solve_nde (free_convection/src/solve.jl:35-48).
 * flux: [ncol][n_fields][Nz+1] (scaled): faces 0 and Nz are the effective boundary fluxes, interior faces NN flux minus the
 * diffusive / convective-adjustment flux; D_c of it, times -tau/H sigma_flux/sigma_q (+ Coriolis), is cpz_rhs's result. */
int cpz_predict_flux(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, float* flux, size_t ncol);
int cpz_predict_flux_dev(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, float* flux, size_t ncol);

/* ---- S2/S6: forward solve ------------------------------------------------------------------- */
/* replaces Array(solve(prob, alg; p=[theta;BCs[i]], saveat)) (NDE_training.jl:291),
 * solve_NDE_mutating (training_postprocessing.jl:55-159), solve_nde (free_convection/src/solve.jl:1-6).
 * traj: [ncol][n_saved][nf*Nz]. */
int cpz_solve(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, float* traj, size_t ncol);
int cpz_solve_dev(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, float* traj, size_t ncol);

/* ---- S2 pullback: VJP of the solve ---------------------------------------------------------------------------------- */
/* replaces the Zygote pullback of Array(solve(prob, ...; sensealg = InterpolatingAdjoint(...))) that loss_NDE /
 * loss_gradient_NDE (NDE_training.jl:290-323) and nde_loss (free_convection/src/training.jl:55-62) take of the loss they
 * compute on the trajectory, so that a host can differentiate any loss of the solve, not only cpz_loss_grad's. With
 * traj_c = what cpz_solve writes for column c on the same inputs (current theta, mPP parameters and time settings) and
 * tbar_c = traj_bar[c] ([ncol][n_saved][nf*Nz], the layout of traj and targets):
 *   x0_bar[c] = (dtraj_c/dx0_c)^T tbar_c             [ncol][nf*Nz]; frame 0 is x0 itself when save_stride > 0
 *   theta_bar = sum_c (dtraj_c/dtheta)^T tbar_c      [P], Flux.destructure order
 *   mpp_bar   = sum_c (dtraj_c/dp)^T tbar_c          [5], p = (nu0, nu_m, dRi, Ric, Pr) unscaled, as cpz_loss_grad_mpp
 * This is the exact discrete adjoint of the engine's fixed-step map, computed by cpz_loss_grad's kernels (checkpointing
 * forward, then the reverse sweep) with traj_bar in place of the loss terms; kinks are handled as there. Outputs are
 * overwritten, not accumulated; each may be NULL, at least one must not be. theta_bar must be NULL when P = 0; mpp_bar is
 * refused where cpz_loss_grad_mpp refuses it, and an implicit-diffusion model where cpz_loss_grad refuses it. The sums
 * over columns are in a fixed order; the allreduce hook is not called (the sum over ranks is the host's) and there is no
 * non-finite reporting. The argument checks are cpz_loss_grad's with traj_bar in place of targets; the device scratch is
 * cpz_loss_grad's. */
int cpz_solve_vjp(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, const float* traj_bar,
                  float* x0_bar, float* theta_bar, float* mpp_bar, size_t ncol);
int cpz_solve_vjp_dev(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, const float* traj_bar,
                      float* x0_bar, float* theta_bar, float* mpp_bar, size_t ncol);

/* ---- S1 / S2 pushforwards: JVPs of f(x, p, t) and of the solve ------------------------------------------------------ */
/* Forward-mode derivatives for hosts that need J v: Rosenbrock / Newton-Krylov integrators (J v per column, or the dense
 * S x S Jacobian of a column from S replicated columns with unit tangents), forward sensitivities wrt few parameters, the
 * tangent-linear model. With f_c = what cpz_rhs returns and traj_c = what cpz_solve writes for column c on the same inputs:
 *   dxdt_dot[c] = (df_c/dx) x_dot[c] + (df_c/dtheta) theta_dot + (df_c/dp) mpp_dot                     [ncol][nf*Nz]
 *   traj_dot[c] = (dtraj_c/dx0) x0_dot[c] + (dtraj_c/dtheta) theta_dot + (dtraj_c/dp) mpp_dot          [ncol][n_saved][nf*Nz]
 * Tangents: x_dot / x0_dot [ncol][nf*Nz], theta_dot [P] in Flux.destructure order, mpp_dot [5] wrt p = (nu0, nu_m, dRi, Ric,
 * Pr) unscaled (the meaning cpz_loss_grad_mpp uses). A NULL tangent counts as zero; at least one must be given. theta_dot
 * is refused when P = 0, mpp_dot where cpz_loss_grad_mpp refuses it. dxdt_dot / traj_dot are required; dxdt / traj are
 * optional and receive the primal result of the same pass. Outputs are overwritten, not accumulated. ncol must be positive.
 * With CPZ_FLAG_IMPLICIT_DIFFUSION cpz_rhs_jvp differentiates the explicit part cpz_rhs returns (mpp_dot contributes 0), and
 * cpz_solve_jvp the whole split step, backward-Euler solve included. At relu kinks, the convective-adjustment switch and
 * CPZ_FLAG_CA_LITERAL_U the derivative of the evaluated branch is taken, as in the pullbacks. Nothing is summed over
 * columns: a column's result depends only on its own inputs (bitwise batch invariance); the allreduce hook is not called
 * and there is no non-finite reporting. Both run FP32 SIMT kernels on the adjoint plan (a model without one is refused with
 * the planner's reason); traj therefore comes from the FP32 pass and differs from cpz_solve's 3xTF32 result for the
 * production nets by rounding. */
int cpz_rhs_jvp(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, const float* x_dot,
                const float* theta_dot, const float* mpp_dot, float* dxdt, float* dxdt_dot, size_t ncol);
int cpz_rhs_jvp_dev(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, const float* x_dot,
                    const float* theta_dot, const float* mpp_dot, float* dxdt, float* dxdt_dot, size_t ncol);
int cpz_solve_jvp(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, const float* x0_dot,
                  const float* theta_dot, const float* mpp_dot, float* traj, float* traj_dot, size_t ncol);
int cpz_solve_jvp_dev(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, const float* x0_dot,
                      const float* theta_dot, const float* mpp_dot, float* traj, float* traj_dot, size_t ncol);

/* ---- S3: objective and gradient ------------------------------------------------------------- */
/* replaces loss_NDE / loss_gradient_NDE + Zygote gradient (NDE_training.jl:290-333; loss.jl:1-42) and
 * nde_loss (free_convection/src/training.jl:55-62).
 * targets: [ncol][n_saved][nf*Nz]; loss_w[6]: weights of (u,v,T,du/dz,dv/dz,dT/dz) (loss.jl:33-42);
 * loss_out[7]: the six weighted components then their sum; grad_out[P] (destructure order) or NULL for loss only.
 * With an allreduce hook set, sums are global over ranks (ncol_global = sum of ncol).
 * Device scratch kept by the model between calls: the step checkpoints, and, depending on the path the model takes
 * (cpz_model_describe names it):
 *   - tensor-core adjoint (production u/v/T nets): per-stage records of as many steps as the free device memory minus 8 GB
 *     holds (73 KB per column-step; all steps when they fit, otherwise one checkpoint-aligned segment at a time with
 *     re-integration; CPZ_ADJ_AUX_GB in the environment sets the budget);
 *   - FP32 adjoint behind the tcgen05 forward solve: the stage tendencies of the forward pass when they fit
 *     (ceil(ncol/32)*32 * n_steps * n_substeps * n_stages * nf*Nz floats; CPZ_NO_KSTORE=1 disables it);
 *   - single-column training kernel (T-only model, ncol <= 32): the record of every stage evaluation
 *     (ncol * n_steps * n_substeps * n_stages * 544 floats, at most 8 GB; larger jobs take the tile kernels). */
int cpz_loss_grad(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, const float* targets,
                  size_t ncol, const float* loss_w, float* loss_out, float* grad_out);
int cpz_loss_grad_dev(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, const float* targets,
                      size_t ncol, const float* loss_w, float* loss_out_dev, float* grad_out_dev);

/* ---- S3 for the NN-free base closure: gradient wrt the five mPP parameters ---------------------------------- */
/* replaces loss_mpp / loss_gradient_mpp + Zygote gradient of optimise_modified_pacanowski_philander
 * (wind_mixing/src/diffusivity_parameter_optimisation.jl:1-33,150-197): p = (nu0, nu_m, dRi, Ric, Pr) in the order `DE`
 * destructures it (:2). The parameters live in the model description; set/get below. The loss is cpz_loss_grad's;
 * grad_mpp_out[5] = d(total loss)/dp (unscaled parameters — the reference optimises p .* (1 ./ p_initial), so the host
 * multiplies by p_initial); grad_theta_out[P] may be NULL (and must be for a model without nets). */
int cpz_set_mpp_params(cpz_model* m, const float* p5);
int cpz_get_mpp_params(const cpz_model* m, float* p5);
int cpz_loss_grad_mpp(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, const float* targets,
                      size_t ncol, const float* loss_w, float* loss_out, float* grad_theta_out, float* grad_mpp_out);
int cpz_loss_grad_mpp_dev(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, const float* targets,
                          size_t ncol, const float* loss_w, float* loss_out_dev, float* grad_theta_out_dev, float* grad_mpp_out_dev);

/* ---- S3+S4: fused training iteration -------------------------------------------------------- */
/* forward + discrete adjoint + (allreduce) + ADAM update of the model's theta; replaces one GalacticOptim iteration
 * (NDE_training.jl:340-372) with Flux.ADAM(lr,(beta1,beta2)), eps=1e-8 semantics. loss_out[7] is the loss at the
 * theta BEFORE the update (what the reference callback sees). */
int cpz_train_step(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, const float* targets,
                   size_t ncol, const float* loss_w, float lr, float beta1, float beta2, float eps, float* loss_out);
int cpz_train_step_dev(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, const float* targets,
                       size_t ncol, const float* loss_w, float lr, float beta1, float beta2, float eps,
                       float* loss_out_host);
/* ADAM state for checkpoint/resume (data_writing.jl:28-78 stores eta/beta/state): m[P], v[P], beta_pow[2]. HOST pointers. */
int cpz_adam_get_state(cpz_model* m, float* mt, float* vt, float* beta_pow, size_t P);
int cpz_adam_set_state(cpz_model* m, const float* mt, const float* vt, const float* beta_pow, size_t P);

/* ---- S7: per-step NN closure inside a 3-D host model --------------------------------------- */
/* replaces convective_adjustment! + compute_neural_network_forcing! (free_convection/double_gyre_nn.jl:27-62,149-168).
 * T: [Nz][Ny][Nx] (x fastest = Julia (Nx,Ny,Nz)); y: [Ny] cell-centre y coordinates. */
typedef struct {
  int32_t Nx, Ny, Nz;
  float dz;            /* metres                                            */
  float dt;            /* host-model time step for the implicit adjustment  */
  float K;             /* convective-adjustment diffusivity, m^2/s          */
  float T_shift, T_div;/* T_profile = T_shift + T/T_div (double_gyre_nn.jl:156: 19.65, 20) */
  float mu_relax;      /* surface restoring rate (double_gyre_nn.jl:113: 1/day) */
  float T_mid, dT, Ly; /* T_reference(y) = T_mid + dT/Ly*y (double_gyre_nn.jl:110)  */
} cpz_closure_desc;
int cpz_closure_step(cpz_model* m, const cpz_closure_desc* c, const float* T, const float* y, float* forcing_out,
                     float* T_out);
int cpz_closure_step_dev(cpz_model* m, const cpz_closure_desc* c, const float* T, const float* y, float* forcing_out,
                         float* T_out);

/* pullback of cpz_closure_step at T on the same model and theta, for the cotangents forcing_bar of forcing_out and T_out_bar
 * of T_out (both [Nz][Ny][Nx]; either may be NULL = zero, not both). Lets a host that differentiates its gyre model (Zygote /
 * Enzyme over a Julia host, torch autograd over a Python one) chain through the closure and train the T-only net on the
 * discretisation it is deployed in:
 *   T_bar: [Nz][Ny][Nx] cotangent of the incoming T;
 *   theta_bar: [P], summed over all columns, destructure order.
 * T' = A(T)^-1 T is the implicit convective adjustment; the forcing depends on T' through the net and the surface restoring
 * flux, so theta_bar comes from forcing_bar alone (T_out_bar alone gives theta_bar = 0 exactly), and T_bar = A^-1 (T_out_bar
 * + the forcing path's cotangent of T') with A symmetric. y, T_mid, dT and Ly are additive constants and drop out, so the
 * pullback takes no y. At relu kinks and at the convective-adjustment switch the derivative is that of the branch the forward
 * evaluated. Outputs are overwritten, not accumulated, and each may be NULL (not both). The sums over columns run in a fixed
 * order (bitwise reproducible); the allreduce hook is not called and there is no non-finite reporting. The argument checks
 * are cpz_closure_step's; a model without the adjoint plan is refused with the planner's reason. */
int cpz_closure_step_vjp(cpz_model* m, const cpz_closure_desc* c, const float* T, const float* forcing_bar,
                         const float* T_out_bar, float* T_bar, float* theta_bar);
int cpz_closure_step_vjp_dev(cpz_model* m, const cpz_closure_desc* c, const float* T, const float* forcing_bar,
                             const float* T_out_bar, float* T_bar, float* theta_bar);

/* ---- S7b: per-step closure of the u/v/T NDE inside a host ocean model (SURVEY 8f-2) ---------- */
/* replaces the Simulation callback progress_neural_network (wind_mixing/src/NDE_oceananigans.jl:380-405): the NN forcing
 * chains NN_uw_forcing / NN_vw_forcing / NN_wT_forcing on the incoming state (:288-344; dz of [0; unscaled NN - shift;
 * top flux]) followed by modified_pacanowski_philander! (:61-101, diffusivities :17-58): a backward-Euler tridiagonal
 * solve of the vertical diffusion of u, v (nu) and T (nu_T) over dt, T'[bottom] kept. The model is a u/v/T model
 * (n_fields = 3, three nets); mu/sigma, g, alpha, nu0, nu_m, dRi, Ric, Pr come from its description. Everything here is
 * DIMENSIONAL. u, v, T: [Nz][Ny][Nx]; dz_flux_out: [3][Nz][Ny][Nx] = dz_uw_NN, dz_vw_NN, dz_wT_NN (the Forcing functions
 * apply the minus sign, :346-359); uvT_out: [3][Nz][Ny][Nx] = u', v', T'. A time-dependent wT_flux(t) (:129,332) is
 * evaluated by the caller and passed as wT_top. On the two boundary faces nu = nu_T = 0 (the reference's boundary-face
 * Ri comes from Oceananigans halo values; 0 is what its gradient boundary conditions give). */
typedef struct {
  int32_t Nx, Ny, Nz;
  float dz;                       /* metres (grid.dz = Lz/Nz)                          */
  float dt;                       /* host-model time step, seconds (:104: 60)          */
  float uw_top, vw_top, wT_top;   /* BCs.top fluxes (:112)                             */
  int32_t convective_adjustment;  /* nu_T = Ri > 0 ? nu/Pr : kappa_ca (:50-53)         */
  float kappa_ca;                 /* :52 hard-codes 1f0                                */
} cpz_closure_uvt_desc;
size_t cpz_sizeof_closure_uvt_desc(void);
int cpz_closure_step_uvt(cpz_model* m, const cpz_closure_uvt_desc* c, const float* u, const float* v, const float* T,
                         float* dz_flux_out, float* uvT_out);
int cpz_closure_step_uvt_dev(cpz_model* m, const cpz_closure_uvt_desc* c, const float* u, const float* v, const float* T,
                             float* dz_flux_out, float* uvT_out);

/* pullback of cpz_closure_step_uvt at (u, v, T) on the same model, theta and mPP parameters, for the cotangents dz_flux_bar of
 * dz_flux_out and uvT_bar of uvT_out (both [3][Nz][Ny][Nx]; either may be NULL = zero, not both). Lets a host that
 * differentiates its own ocean or column model (Zygote / Enzyme over a Julia host, torch autograd over a Python one) chain
 * through the closure and train the nets, or tune the base closure, on the discretisation they are deployed in:
 *   u_bar, v_bar, T_bar: [Nz][Ny][Nx] cotangents of the incoming fields;
 *   theta_bar: [P], summed over all columns, destructure order (NULL required when P = 0);
 *   mpp_bar[5]: wrt p = (nu0, nu_m, dRi, Ric, Pr), unscaled, as cpz_loss_grad_mpp (refused with smooth_Ri).
 * The step's outputs depend on the state through separate paths: dz_flux through the nets, (u', v', T') through the implicit
 * mPP step of the incoming state (the forcing is applied by the host), so theta_bar comes from dz_flux_bar alone and mpp_bar
 * from uvT_bar alone. uw_top, vw_top and wT_top are additive constants and drop out. T'[bottom] = T[bottom] and nu = 0 on
 * the two boundary faces are differentiated as the forward states them. At relu kinks and at the convective-adjustment
 * switch the derivative is that of the branch the forward evaluated. Outputs are overwritten, not accumulated, and each may
 * be NULL (not all). The sums over columns run in a fixed order (bitwise reproducible); the allreduce hook is not called
 * and there is no non-finite reporting. The argument checks are cpz_closure_step_uvt's; a model without the adjoint plan
 * (e.g. the 400-wide nets) is refused with the planner's reason. */
int cpz_closure_step_uvt_vjp(cpz_model* m, const cpz_closure_uvt_desc* c, const float* u, const float* v, const float* T,
                             const float* dz_flux_bar, const float* uvT_bar, float* u_bar, float* v_bar, float* T_bar,
                             float* theta_bar, float* mpp_bar);
int cpz_closure_step_uvt_vjp_dev(cpz_model* m, const cpz_closure_uvt_desc* c, const float* u, const float* v, const float* T,
                                 const float* dz_flux_bar, const float* uvT_bar, float* u_bar, float* v_bar, float* T_bar,
                                 float* theta_bar, float* mpp_bar);

#ifdef __cplusplus
}
#endif
#endif /* CPZ_H */
