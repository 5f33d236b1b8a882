// C ABI of libcpz.so (see include/cpz.h). Host-side orchestration: device buffers, launches, error reporting.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "cpz_launch.h"
#include "cpz_closure_uvt_vjp.cuh"
#include "cpz_closure_vjp.cuh"
#include "cpz_jvp.cuh"

namespace cpz {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
int cuda_fail(cudaError_t e, const char* what) {
  snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
  return CPZ_ERR_CUDA;
}

static int ensure(DevBuf& b, size_t floats) {
  if (floats <= b.cap) return CPZ_OK;
  if (b.p) CPZ_CUDA(cudaFree(b.p));
  b.p = nullptr; b.cap = 0;
  CPZ_CUDA(cudaMalloc(&b.p, std::max<size_t>(floats, 4) * sizeof(float)));
  b.cap = floats;
  return CPZ_OK;
}
static void release(DevBuf& b) {
  if (b.p) cudaFree(b.p);
  b.p = nullptr; b.cap = 0;
}

// Grid and reduction buffers of the single-evaluation pullbacks (cpz_rhs_vjp, cpz_closure_step_vjp,
// cpz_closure_step_uvt_vjp): a persistent grid of min(tiles, SMs) CTAs over VJP_CT-column tiles, each CTA with one
// weight-gradient slab in b_part and one LP row after the slabs. b_red is touched only when mpp_bar is wanted: host flavours
// stage theta_bar in b_red[0, P) and grow b_red to P + 16 beforehand, so the ensure here never reallocates an output they
// passed in.
struct SlabPullback {
  float* theta_bar;  // [P] output, or null
  float* mpp_bar;    // [5] output, or null
  size_t ncol;
  int n_tiles, grid;
  float* gpart;  // [grid][M.slab] weight-gradient slabs, zeroed when theta_bar is wanted
  float* lpart;  // [grid][LP], zeroed when mpp_bar is wanted: the five mPP-parameter sums at LP/2 .. LP/2+4
};

static int begin_slab_pullback(cpz_model* m, size_t ncol, float* theta_bar, float* mpp_bar, SlabPullback& sp) {
  cudaStream_t st = m->ctx->stream;
  sp.theta_bar = theta_bar; sp.mpp_bar = mpp_bar; sp.ncol = ncol;
  sp.n_tiles = (int)((ncol + VJP_CT - 1) / VJP_CT);
  sp.grid = std::min(sp.n_tiles, m->ctx->sm_count);
  const size_t slab = (size_t)m->bwd.M.slab;
  int rc;
  if ((rc = ensure(m->b_part, (size_t)sp.grid * (slab + LP)))) return rc;
  if (mpp_bar && (rc = ensure(m->b_red, m->P + 16))) return rc;
  sp.gpart = m->b_part.p;
  sp.lpart = m->b_part.p + (size_t)sp.grid * slab;
  if (theta_bar) CPZ_CUDA(cudaMemsetAsync(sp.gpart, 0, (size_t)sp.grid * slab * sizeof(float), st));
  if (mpp_bar) CPZ_CUDA(cudaMemsetAsync(sp.lpart, 0, (size_t)sp.grid * LP * sizeof(float), st));
  return CPZ_OK;
}

// theta_bar = the sum of the slabs; mpp_bar = the five mPP-parameter sums of the LP rows
static int finish_slab_pullback(cpz_model* m, const SlabPullback& sp) {
  const int P = (int)m->P;
  int rc;
  if (sp.theta_bar && (rc = launch_reduce_slabs(m, sp.gpart, sp.grid, P, sp.theta_bar))) return rc;
  if (sp.mpp_bar) {
    if ((rc = launch_pack_loss(m, sp.lpart, sp.grid, LP, (float)sp.ncol, m->b_red.p + P))) return rc;
    CPZ_CUDA(cudaMemcpyAsync(sp.mpp_bar, m->b_red.p + P + 8, 5 * sizeof(float), cudaMemcpyDeviceToDevice, m->ctx->stream));
  }
  return CPZ_OK;
}

// The mPP-parameter gradient (cpz_loss_grad_mpp, and mpp_bar of the pullbacks that run the model's own RHS)
static int check_mpp_grad(const cpz_model* m) {
  if (m->desc.n_fields != 3) return fail(CPZ_ERR_INVALID, "mPP-parameter gradient needs the u/v/T model");
  if (!((m->desc.flags & CPZ_FLAG_MPP) || m->desc.variant == CPZ_RHS_INFER)) return fail(CPZ_ERR_INVALID, "mPP-parameter gradient needs CPZ_FLAG_MPP");
  if (m->desc.flags & CPZ_FLAG_SMOOTH_RI) return fail(CPZ_ERR_INVALID, "mPP-parameter gradient is not available with smooth_Ri");
  return CPZ_OK;
}

static int n_saved_of(const TimeD& tm) { return tm.save_stride <= 0 ? 1 : tm.n_steps / tm.save_stride + 1; }
// checkpoints: step 0, every ckpt_stride-th step, and the final step (once)
static int n_ckpt_of(const TimeD& tm) {
  int n = tm.n_steps / tm.ckpt_stride + 1;
  if (tm.n_steps % tm.ckpt_stride != 0) ++n;
  return n;
}

static int check_model(const cpz_model* m) {
  if (!m || !m->ctx) return fail(CPZ_ERR_INVALID, "null model handle");
  return CPZ_OK;
}

static int bind_device(const cpz_ctx* c) {
  CPZ_CUDA(cudaSetDevice(c->device));
  return CPZ_OK;
}

static size_t solve_other_smem(const cpz_model_desc& d, int CT, int n_stages) {
  const int S = d.n_fields * d.Nz, nbc = d.n_fields == 3 ? 6 : 2;
  if ((d.flags & CPZ_FLAG_IMPLICIT_DIFFUSION) && n_stages < 2) n_stages = 2;  // scratch of the implicit-diffusion step
  return ((size_t)3 * CT * (S + 4) + (size_t)n_stages * S * CT + (size_t)nbc * CT + CT + 4) * sizeof(float) + ((sizeof(ModelD) + 15) / 16) * 16;
}

static int rebuild_plans(cpz_model* m) {
  std::string err;
  fill_tableau(m->desc.integrator, m->tab);
  m->tm.dt = m->desc.dt; m->tm.t0 = m->desc.t0; m->tm.n_steps = m->desc.n_steps; m->tm.n_substeps = m->desc.n_substeps;
  m->tm.save_stride = m->desc.save_stride; m->tm.ckpt_stride = m->desc.ckpt_stride; m->tm.step0 = 0;
  PlanOptions fo;
  fo.CT = m->CT; fo.NT = m->NT; fo.keep_all = false;
  fo.smem_budget = m->ctx->smem_optin;
  fo.other_smem_bytes = solve_other_smem(m->desc, m->CT, m->tab.n_stages);
  if (!build_plan(m->desc, fo, m->fwd, err)) return fail(CPZ_ERR_INVALID, "forward plan: %s", err.c_str());
  PlanOptions bo;
  bo.CT = m->CT; bo.NT = m->NT; bo.keep_all = true;
  bo.smem_budget = m->ctx->smem_optin;
  bo.other_smem_bytes = adjoint_other_smem(m->desc.n_fields * m->desc.Nz, m->desc.n_fields == 3 ? 6 : 2, m->CT);
  m->has_bwd = build_plan(m->desc, bo, m->bwd, m->bwd_err);
  m->implicit_adjoint_ok = true;  // adjoint_kernel carries implicit_vjp_tile
  for (int i = 0; i < cpz_model::N_SMALL; ++i) {
    const int cs = cpz_model::small_ct(i);
    PlanOptions fs = fo, bs = bo;
    std::string es;
    fs.CT = cs; fs.other_smem_bytes = solve_other_smem(m->desc, cs, m->tab.n_stages);
    bs.CT = cs; bs.other_smem_bytes = adjoint_other_smem(m->desc.n_fields * m->desc.Nz, m->desc.n_fields == 3 ? 6 : 2, cs);
    m->has_small[i] = m->has_bwd && build_plan(m->desc, fs, m->fwd_s[i], es) && build_plan(m->desc, bs, m->bwd_s[i], es);
    // every adjoint plan must describe the same gradient slab (one index map, one reduction kernel)
    if (m->has_small[i]) {
      const ModelD &A = m->bwd.M, &B = m->bwd_s[i].M;
      bool same = A.slab == B.slab && A.n_gemm == B.n_gemm;
      for (int gi = 0; same && gi < A.n_gemm; ++gi)
        same = A.gemm[gi].gw_off == B.gemm[gi].gw_off && A.gemm[gi].gb_off == B.gemm[gi].gb_off && A.gemm[gi].w_off == B.gemm[gi].w_off;
      m->has_small[i] = same;
    }
  }
  if (m->has_bwd && m->P > 0) {
    std::vector<int> map(m->P, 0);
    const ModelD& B = m->bwd.M;
    for (int gi = 0; gi < B.n_gemm; ++gi) {
      const GemmD& g = B.gemm[gi];
      const int njg = (g.N + 3) / 4;
      for (int k = 0; k < g.K; ++k)
        for (int j = 0; j < g.N; ++j)
          map[g.w_off + k * g.N + j] = g.gw_off + ((k / 4) * njg + j / 4) * 16 + (k % 4) * 4 + (j % 4);
      for (int j = 0; j < g.N; ++j) map[g.b_off + j] = g.gb_off + j;
    }
    if (!m->d_gmap) CPZ_CUDA(cudaMalloc(&m->d_gmap, m->P * sizeof(int)));
    CPZ_CUDA(cudaMemcpyAsync(m->d_gmap, map.data(), m->P * sizeof(int), cudaMemcpyHostToDevice, m->ctx->stream));
    CPZ_CUDA(cudaStreamSynchronize(m->ctx->stream));
  }
  return CPZ_OK;
}

}  // namespace cpz

using namespace cpz;

extern "C" {

int cpz_version(void) { return CPZ_VERSION_MAJOR * 100 + CPZ_VERSION_MINOR; }
const char* cpz_last_error(void) { return g_err; }

size_t cpz_sizeof_model_desc(void) { return sizeof(cpz_model_desc); }
size_t cpz_sizeof_closure_desc(void) { return sizeof(cpz_closure_desc); }

int cpz_device_count(int* n) {
  if (!n) return fail(CPZ_ERR_INVALID, "null pointer");
  int c = 0;
  cudaError_t e = cudaGetDeviceCount(&c);
  if (e != cudaSuccess) { cudaGetLastError(); c = 0; }
  *n = c;
  return CPZ_OK;
}

int cpz_ctx_create(int device, void* stream, cpz_ctx** out) {
  if (!out) return fail(CPZ_ERR_INVALID, "null out pointer");
  *out = nullptr;
  int cnt = 0;
  cudaError_t e = cudaGetDeviceCount(&cnt);
  if (e != cudaSuccess || cnt == 0) {
    cudaGetLastError();
    return fail(CPZ_ERR_CUDA, "no CUDA device available (%s); libcpz has no CPU fallback", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  }
  if (device < 0 || device >= cnt) return fail(CPZ_ERR_INVALID, "device %d out of range [0,%d)", device, cnt);
  CPZ_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  CPZ_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail(CPZ_ERR_CUDA, "device %d is sm_%d%d; libcpz is built for sm_100a only", device, prop.major, prop.minor);
  cpz_ctx* c = new (std::nothrow) cpz_ctx();
  if (!c) return fail(CPZ_ERR_INVALID, "out of host memory");
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->smem_optin = prop.sharedMemPerBlockOptin;
  if (stream) {
    c->stream = (cudaStream_t)stream;
  } else {
    cudaError_t es = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (es != cudaSuccess) { delete c; return cuda_fail(es, "cudaStreamCreateWithFlags"); }
    c->own_stream = true;
  }
  *out = c;
  return CPZ_OK;
}

int cpz_ctx_destroy(cpz_ctx* ctx) {
  if (!ctx) return CPZ_OK;
  cudaSetDevice(ctx->device);
  if (ctx->d_nonfinite) cudaFree(ctx->d_nonfinite);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  for (auto& e : ctx->chunk_ev) if (e) cudaEventDestroy(e);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return CPZ_OK;
}

int cpz_ctx_set_allreduce(cpz_ctx* ctx, cpz_allreduce_fn fn, void* user, int rank, int world_size) {
  if (!ctx) return fail(CPZ_ERR_INVALID, "null ctx");
  if (world_size < 1 || rank < 0 || rank >= world_size) return fail(CPZ_ERR_INVALID, "bad rank/world_size");
  ctx->allreduce = fn; ctx->allreduce_user = user; ctx->rank = rank; ctx->world = world_size;
  return CPZ_OK;
}

int cpz_ctx_synchronize(cpz_ctx* ctx) {
  if (!ctx) return fail(CPZ_ERR_INVALID, "null ctx");
  CPZ_CUDA(cudaSetDevice(ctx->device));
  CPZ_CUDA(cudaStreamSynchronize(ctx->stream));
  return CPZ_OK;
}

int cpz_ctx_stream(cpz_ctx* ctx, void** stream_out) {
  if (!ctx || !stream_out) return fail(CPZ_ERR_INVALID, "null pointer");
  *stream_out = (void*)ctx->stream;
  return CPZ_OK;
}

int cpz_ctx_nonfinite_count(cpz_ctx* ctx, uint64_t* n) {
  if (!ctx || !n) return fail(CPZ_ERR_INVALID, "null pointer");
  *n = 0;
  if (!ctx->d_nonfinite) return CPZ_OK;
  CPZ_CUDA(cudaSetDevice(ctx->device));
  unsigned int v = 0;
  CPZ_CUDA(cudaMemcpyAsync(&v, ctx->d_nonfinite, sizeof(v), cudaMemcpyDeviceToHost, ctx->stream));
  CPZ_CUDA(cudaStreamSynchronize(ctx->stream));
  *n = v;
  return CPZ_OK;
}

int cpz_ctx_launch_count(cpz_ctx* ctx, uint64_t* n) {
  if (!ctx || !n) return fail(CPZ_ERR_INVALID, "null pointer");
  *n = ctx->launches;
  return CPZ_OK;
}

int cpz_model_create(cpz_ctx* ctx, const cpz_model_desc* desc, cpz_model** out) {
  if (!ctx || !desc || !out) return fail(CPZ_ERR_INVALID, "null pointer");
  *out = nullptr;
  std::string err;
  if (!validate_desc(*desc, err)) return fail(CPZ_ERR_INVALID, "%s", err.c_str());
  int rc = bind_device(ctx);
  if (rc) return rc;
  cpz_model* m = new (std::nothrow) cpz_model();
  if (!m) return fail(CPZ_ERR_INVALID, "out of host memory");
  m->ctx = ctx;
  m->desc = *desc;
  m->P = count_params(*desc);
  rc = rebuild_plans(m);
  if (rc) { delete m; return rc; }
  const size_t pf = std::max<size_t>(m->P, 4);
  cudaError_t e = cudaMalloc(&m->d_theta, pf * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&m->d_m, pf * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&m->d_v, pf * sizeof(float));
  if (e == cudaSuccess) e = cudaMemsetAsync(m->d_theta, 0, pf * sizeof(float), ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(m->d_m, 0, pf * sizeof(float), ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(m->d_v, 0, pf * sizeof(float), ctx->stream);
  if (e != cudaSuccess) { cpz_model_destroy(m); return cuda_fail(e, "model allocation"); }
  *out = m;
  return CPZ_OK;
}

int cpz_model_destroy(cpz_model* m) {
  if (!m) return CPZ_OK;
  if (m->ctx) { cudaSetDevice(m->ctx->device); cudaStreamSynchronize(m->ctx->stream); }
  if (m->d_theta) cudaFree(m->d_theta);
  if (m->d_m) cudaFree(m->d_m);
  if (m->d_v) cudaFree(m->d_v);
  if (m->d_gmap) cudaFree(m->d_gmap);
  DevBuf* bufs[] = {&m->b_x0, &m->b_bcs, &m->b_q, &m->b_traj, &m->b_tgt, &m->b_ckpt, &m->b_scr, &m->b_part, &m->b_red, &m->b_out, &m->b_w, &m->b_wimg, &m->b_cimg, &m->b_fcscr, &m->b_kstore, &m->b_aux, &m->b_bwimg, &m->b_tcadj};
  for (DevBuf* b : bufs) release(*b);
  delete m;
  return CPZ_OK;
}

int cpz_model_n_params(const cpz_model* m, size_t* P) {
  if (!m || !P) return fail(CPZ_ERR_INVALID, "null pointer");
  *P = m->P;
  return CPZ_OK;
}

int cpz_model_n_saved(const cpz_model* m, int32_t* n) {
  if (!m || !n) return fail(CPZ_ERR_INVALID, "null pointer");
  *n = n_saved_of(m->tm);
  return CPZ_OK;
}

int cpz_model_describe(const cpz_model* m, char* buf, size_t buf_len) {
  if (!m || !buf || buf_len == 0) return fail(CPZ_ERR_INVALID, "null pointer");
  std::string s;
  char line[512];
  auto dump = [&](const char* name, const Plan& pl, size_t other) {
    const ModelD& M = pl.M;
    snprintf(line, sizeof(line), "%s plan: CT=%d NT=%d %s weights_in_smem=%d weight_smem=%zuB arena=%zuB other=%zuB arena_rows=%d flux_off=%d\n",
             name, m->CT, m->NT, pl.layer_major ? "layer-major" : "net-major", M.w_in_smem, pl.smem_weight_bytes, pl.arena_bytes, other,
             M.arena_floats, M.flux_off);
    s += line;
    for (int p = 0; p < M.n_phase; ++p) {
      snprintf(line, sizeof(line), "  phase %d: tiles=%d tile=%dcols x %douts ksplit=%d:", p, M.phase[p].n_tiles, M.phase[p].TC, M.phase[p].TO, M.phase[p].ksplit);
      s += line;
      for (int g = M.phase[p].g0; g < M.phase[p].g1; ++g) {
        const GemmD& G = M.gemm[g];
        snprintf(line, sizeof(line), " [net%d L%d K=%d N=%d TO=%d Npad=%d act=%d in=%d out=%d]", G.net, G.layer, G.K, G.N, G.TO, G.Npad, G.act, G.in_off, G.out_off);
        s += line;
      }
      s += "\n";
    }
  };
  s += tc_describe(m);
  {
    std::string why;
    if (m->P > 0 && adjoint_tc_eligible(const_cast<cpz_model*>(m), &why))
      s += "adjoint kernels: tcgen05 3xTF32 (stage records in HBM; reverse sweep with transposed weights in tensor memory; weight gradient as one contraction over columns x stages)\n";
    else if (m->P > 0)
      s += "adjoint kernels: fp32-simt (tensor-core adjoint not eligible: " + why + ")\n";
    if (m->P > 0 && fc1_eligible(m, 1))
      s += "small batches (<= 32 columns, CPZ_FC1_MAX_NCOL): one CTA per column, weights in shared memory, weight gradients in registers\n";
  }
  dump("forward", m->fwd, solve_other_smem(m->desc, m->CT, m->tab.n_stages));
  if (m->has_bwd) dump("adjoint", m->bwd, adjoint_other_smem(m->desc.n_fields * m->desc.Nz, m->desc.n_fields == 3 ? 6 : 2, m->CT));
  else s += "adjoint plan: unavailable (" + m->bwd_err + ")\n";
  auto pullback = [&](const char* what, const char* kernel, bool closure) {  // the single-evaluation pullbacks (launch_vjp_t)
    snprintf(line, sizeof(line), "%s: %s, fp32-simt, 32-column tiles%s on the adjoint plan, weights %s, persistent grid of min(tiles, %d) "
             "CTAs with one gradient slab each\n", what, kernel, closure ? " (32 consecutive x-columns)" : "",
             m->bwd.M.w_in_smem ? "in shared memory" : "streamed from global memory", m->ctx->sm_count);
    s += line;
  };
  if (m->has_bwd) pullback("rhs pullback (cpz_rhs_vjp)", "rhs_vjp_kernel", false);
  if (m->has_bwd && m->desc.n_fields == 3 && m->desc.n_nets == 3)
    pullback("u/v/T closure-step pullback (cpz_closure_step_uvt_vjp)", "closure_uvt_vjp_kernel", true);
  if (m->has_bwd && m->desc.n_fields == 1 && m->desc.n_nets == 1)
    pullback("gyre closure-step pullback (cpz_closure_step_vjp)", "closure_vjp_kernel", true);
  s += "solve pullback (cpz_solve_vjp): the cpz_loss_grad kernels above in cotangent mode (the trajectory cotangent replaces the "
       "loss terms at the saved frames; x0 cotangent stored at the end of the reverse sweep)\n";
  if (m->has_bwd) {
    snprintf(line, sizeof(line), "tangents (cpz_rhs_jvp, cpz_solve_jvp): rhs_jvp_kernel, solve_jvp_kernel, fp32-simt, 32-column tiles on "
             "the adjoint plan, weights %s, persistent grid of min(tiles, %d) CTAs; the solve's stage slots k and kdot in a per-CTA "
             "global scratch\n", m->bwd.M.w_in_smem ? "in shared memory" : "streamed from global memory", m->ctx->sm_count);
    s += line;
  }
  if (m->has_small[0]) {
    const int sms = m->ctx->sm_count > 0 ? m->ctx->sm_count : 148;
    snprintf(line, sizeof(line), "small-batch training pass: 4- / 8- / 16-column adjoint tiles while the batch fits one wave (up to %d / %d / %d columns)\n",
             4 * sms, 8 * sms, 16 * sms);
    s += line;
  }
  snprintf(buf, buf_len, "%s", s.c_str());
  return CPZ_OK;
}

int cpz_set_theta(cpz_model* m, const float* theta, size_t P) {
  int rc = check_model(m);
  if (rc) return rc;
  if (P != m->P) return fail(CPZ_ERR_INVALID, "theta length %zu != model parameters %zu", P, m->P);
  if (P == 0) return CPZ_OK;
  if (!theta) return fail(CPZ_ERR_INVALID, "null theta");
  if ((rc = bind_device(m->ctx))) return rc;
  CPZ_CUDA(cudaMemcpyAsync(m->d_theta, theta, P * sizeof(float), cudaMemcpyHostToDevice, m->ctx->stream));
  CPZ_CUDA(cudaStreamSynchronize(m->ctx->stream));
  m->theta_ver++;
  return CPZ_OK;
}

int cpz_get_theta(cpz_model* m, float* theta, size_t P) {
  int rc = check_model(m);
  if (rc) return rc;
  if (P != m->P) return fail(CPZ_ERR_INVALID, "theta length %zu != model parameters %zu", P, m->P);
  if (P == 0) return CPZ_OK;
  if (!theta) return fail(CPZ_ERR_INVALID, "null theta");
  if ((rc = bind_device(m->ctx))) return rc;
  CPZ_CUDA(cudaMemcpyAsync(theta, m->d_theta, P * sizeof(float), cudaMemcpyDeviceToHost, m->ctx->stream));
  CPZ_CUDA(cudaStreamSynchronize(m->ctx->stream));
  return CPZ_OK;
}

int cpz_model_set_time(cpz_model* m, int32_t integrator, float dt, float t0, int32_t n_steps, int32_t n_substeps,
                       int32_t save_stride, int32_t ckpt_stride) {
  int rc = check_model(m);
  if (rc) return rc;
  cpz_model_desc d = m->desc;
  d.integrator = integrator; d.dt = dt; d.t0 = t0; d.n_steps = n_steps; d.n_substeps = n_substeps;
  d.save_stride = save_stride; d.ckpt_stride = ckpt_stride;
  std::string err;
  if (!validate_desc(d, err)) return fail(CPZ_ERR_INVALID, "%s", err.c_str());
  const bool replan = d.integrator != m->desc.integrator;
  m->desc = d;
  if (replan) return rebuild_plans(m);
  fill_tableau(d.integrator, m->tab);
  m->tm.dt = dt; m->tm.t0 = t0; m->tm.n_steps = n_steps; m->tm.n_substeps = n_substeps;
  m->tm.save_stride = save_stride; m->tm.ckpt_stride = ckpt_stride; m->tm.step0 = 0;
  return CPZ_OK;
}

// ---- RHS ------------------------------------------------------------------------------------------------------------
int cpz_rhs_dev(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, float* dxdt, size_t ncol) {
  int rc = check_model(m);
  if (rc) return rc;
  if (ncol == 0) return CPZ_OK;
  if (!x || !bcs || !dxdt) return fail(CPZ_ERR_INVALID, "null array");
  if ((m->desc.flags & CPZ_FLAG_DIURNAL) && !diurnal_Q) return fail(CPZ_ERR_INVALID, "diurnal model needs diurnal_Q");
  if (ncol > (size_t)INT32_MAX / 512) return fail(CPZ_ERR_INVALID, "ncol too large");
  if ((rc = bind_device(m->ctx))) return rc;
  SolveArgs a{};
  a.theta = m->d_theta; a.x0 = x; a.bcs = bcs; a.Q = diurnal_Q; a.dxdt = dxdt; a.ncol = (int)ncol;
  a.rhs_only = 1; a.t_rhs = t; a.n_saved = 1; a.n_ckpt = 0;
  return launch_solve(m, a);
}

static int upload_inputs(cpz_model* m, const float* x0, const float* bcs, const float* Q, size_t ncol) {
  const size_t S = (size_t)m->fwd.M.S, nbc = (size_t)m->fwd.M.nbc;
  int rc;
  if ((rc = ensure(m->b_x0, ncol * S))) return rc;
  if ((rc = ensure(m->b_bcs, ncol * nbc))) return rc;
  cudaStream_t st = m->ctx->stream;
  CPZ_CUDA(cudaMemcpyAsync(m->b_x0.p, x0, ncol * S * sizeof(float), cudaMemcpyHostToDevice, st));
  CPZ_CUDA(cudaMemcpyAsync(m->b_bcs.p, bcs, ncol * nbc * sizeof(float), cudaMemcpyHostToDevice, st));
  if (Q) {
    if ((rc = ensure(m->b_q, ncol))) return rc;
    CPZ_CUDA(cudaMemcpyAsync(m->b_q.p, Q, ncol * sizeof(float), cudaMemcpyHostToDevice, st));
  }
  return CPZ_OK;
}

int cpz_rhs(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, float* dxdt, size_t ncol) {
  int rc = check_model(m);
  if (rc) return rc;
  if (ncol == 0) return CPZ_OK;
  if (!x || !bcs || !dxdt) return fail(CPZ_ERR_INVALID, "null array");
  if ((rc = bind_device(m->ctx))) return rc;
  if ((rc = upload_inputs(m, x, bcs, diurnal_Q, ncol))) return rc;
  const size_t S = (size_t)m->fwd.M.S;
  if ((rc = ensure(m->b_traj, ncol * S))) return rc;
  if ((rc = cpz_rhs_dev(m, m->b_x0.p, m->b_bcs.p, diurnal_Q ? m->b_q.p : nullptr, t, m->b_traj.p, ncol))) return rc;
  CPZ_CUDA(cudaMemcpyAsync(dxdt, m->b_traj.p, ncol * S * sizeof(float), cudaMemcpyDeviceToHost, m->ctx->stream));
  CPZ_CUDA(cudaStreamSynchronize(m->ctx->stream));
  return CPZ_OK;
}

// ---- RHS pullback ---------------------------------------------------------------------------------------------------
int cpz_rhs_vjp_dev(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, const float* dxdt_bar,
                    float* x_bar, float* theta_bar, float* mpp_bar, size_t ncol) {
  (void)t;  // boundary fluxes, diurnal forcing and t enter f additively: the cotangents do not depend on them
  int rc = check_model(m);
  if (rc) return rc;
  if (ncol == 0) return CPZ_OK;
  if (!x_bar && !theta_bar && !mpp_bar) return fail(CPZ_ERR_INVALID, "rhs_vjp: no output requested (x_bar, theta_bar and mpp_bar are all NULL)");
  if (!x || !bcs || !dxdt_bar) return fail(CPZ_ERR_INVALID, "null array");
  if ((m->desc.flags & CPZ_FLAG_DIURNAL) && !diurnal_Q) return fail(CPZ_ERR_INVALID, "diurnal model needs diurnal_Q");
  if (theta_bar && m->P == 0) return fail(CPZ_ERR_INVALID, "rhs_vjp: theta_bar requested but the model has no parameters");
  if (mpp_bar && (rc = check_mpp_grad(m))) return rc;
  if (!m->has_bwd) return fail(CPZ_ERR_INVALID, "adjoint plan unavailable: %s", m->bwd_err.c_str());
  if (ncol > (size_t)INT32_MAX / 512) return fail(CPZ_ERR_INVALID, "ncol too large");
  if ((rc = bind_device(m->ctx))) return rc;
  SlabPullback sp;
  if ((rc = begin_slab_pullback(m, ncol, theta_bar, mpp_bar, sp))) return rc;
  VjpArgs a{};
  a.theta = m->d_theta; a.x = x; a.ybar = dxdt_bar; a.xbar = x_bar; a.gpart = sp.gpart; a.lpart = sp.lpart;
  a.want_mlp = (x_bar || theta_bar) && m->P > 0; a.want_pgrad = mpp_bar != nullptr; a.ncol = (int)ncol; a.n_tiles = sp.n_tiles;
  if ((rc = launch_rhs_vjp(m, a, sp.grid))) return rc;
  return finish_slab_pullback(m, sp);
}

int cpz_rhs_vjp(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, const float* dxdt_bar,
                float* x_bar, float* theta_bar, float* mpp_bar, size_t ncol) {
  int rc = check_model(m);
  if (rc) return rc;
  if (ncol == 0) return CPZ_OK;
  if (!x || !bcs || !dxdt_bar) return fail(CPZ_ERR_INVALID, "null array");
  if ((rc = bind_device(m->ctx))) return rc;
  if ((rc = upload_inputs(m, x, bcs, diurnal_Q, ncol))) return rc;
  const size_t S = (size_t)m->fwd.M.S;
  cudaStream_t st = m->ctx->stream;
  // staging: ybar in b_tgt, x_bar in b_traj, theta_bar in b_red[0, P) (the pullback's reduction tail is b_red[P, P+16)),
  // mpp_bar in b_out
  if ((rc = ensure(m->b_tgt, ncol * S))) return rc;
  if ((rc = ensure(m->b_traj, ncol * S))) return rc;
  if ((rc = ensure(m->b_red, m->P + 16))) return rc;
  if ((rc = ensure(m->b_out, 8))) return rc;
  CPZ_CUDA(cudaMemcpyAsync(m->b_tgt.p, dxdt_bar, ncol * S * sizeof(float), cudaMemcpyHostToDevice, st));
  if ((rc = cpz_rhs_vjp_dev(m, m->b_x0.p, m->b_bcs.p, diurnal_Q ? m->b_q.p : nullptr, t, m->b_tgt.p, x_bar ? m->b_traj.p : nullptr,
                            theta_bar ? m->b_red.p : nullptr, mpp_bar ? m->b_out.p : nullptr, ncol)))
    return rc;
  if (x_bar) CPZ_CUDA(cudaMemcpyAsync(x_bar, m->b_traj.p, ncol * S * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (theta_bar) CPZ_CUDA(cudaMemcpyAsync(theta_bar, m->b_red.p, m->P * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (mpp_bar) CPZ_CUDA(cudaMemcpyAsync(mpp_bar, m->b_out.p, 5 * sizeof(float), cudaMemcpyDeviceToHost, st));
  CPZ_CUDA(cudaStreamSynchronize(st));
  return CPZ_OK;
}

// ---- RHS pushforward ------------------------------------------------------------------------------------------------
}  // extern "C"
namespace {
// Argument checks of cpz_rhs_jvp and cpz_solve_jvp (both flavours); binds the context's device
int check_jvp_args(cpz_model* m, const char* what, const float* x, const float* bcs, const float* Q, const float* x_dot,
                   const float* theta_dot, const float* mpp_dot, const float* y_dot, size_t ncol) {
  int rc = check_model(m);
  if (rc) return rc;
  if (ncol == 0) return fail(CPZ_ERR_INVALID, "ncol must be positive");
  if (!x || !bcs || !y_dot) return fail(CPZ_ERR_INVALID, "null array");
  if (!x_dot && !theta_dot && !mpp_dot) return fail(CPZ_ERR_INVALID, "%s: no tangent given (x_dot, theta_dot and mpp_dot are all NULL)", what);
  if ((m->desc.flags & CPZ_FLAG_DIURNAL) && !Q) return fail(CPZ_ERR_INVALID, "diurnal model needs diurnal_Q");
  if (theta_dot && m->P == 0) return fail(CPZ_ERR_INVALID, "%s: theta_dot given but the model has no parameters", what);
  if (mpp_dot && (rc = check_mpp_grad(m))) return rc;
  if (!m->has_bwd) return fail(CPZ_ERR_INVALID, "adjoint plan unavailable: %s", m->bwd_err.c_str());
  if (ncol > (size_t)INT32_MAX / 512) return fail(CPZ_ERR_INVALID, "ncol too large");
  return bind_device(m->ctx);
}

JvpArgs jvp_args(cpz_model* m, const float* x, const float* bcs, const float* Q, const float* x_dot, const float* theta_dot,
                 const float* mpp_dot, float* y, float* y_dot, size_t ncol, int& grid) {
  JvpArgs a{};
  a.theta = m->d_theta; a.theta_dot = theta_dot; a.pdot = mpp_dot; a.x = x; a.xdot = x_dot; a.bcs = bcs; a.Q = Q;
  a.y = y; a.ydot = y_dot; a.ncol = (int)ncol; a.n_tiles = (int)((ncol + VJP_CT - 1) / VJP_CT);
  grid = std::min(a.n_tiles, m->ctx->sm_count);
  return a;
}

// Host flavours: the inputs go to device staging (x, bcs, Q as upload_inputs does; x_dot in b_tgt, theta_dot in b_red, mpp_dot
// in b_out), the tangent output to b_traj and the primal output to b_ckpt.
int stage_jvp_inputs(cpz_model* m, const float* x, const float* bcs, const float* Q, const float* x_dot, const float* theta_dot,
                     const float* mpp_dot, size_t ncol, size_t out_floats, bool want_y) {
  int rc;
  if ((rc = upload_inputs(m, x, bcs, Q, ncol))) return rc;
  const size_t S = (size_t)m->fwd.M.S;
  cudaStream_t st = m->ctx->stream;
  if (x_dot) {
    if ((rc = ensure(m->b_tgt, ncol * S))) return rc;
    CPZ_CUDA(cudaMemcpyAsync(m->b_tgt.p, x_dot, ncol * S * sizeof(float), cudaMemcpyHostToDevice, st));
  }
  if (theta_dot) {
    if ((rc = ensure(m->b_red, m->P + 16))) return rc;
    CPZ_CUDA(cudaMemcpyAsync(m->b_red.p, theta_dot, m->P * sizeof(float), cudaMemcpyHostToDevice, st));
  }
  if (mpp_dot) {
    if ((rc = ensure(m->b_out, 8))) return rc;
    CPZ_CUDA(cudaMemcpyAsync(m->b_out.p, mpp_dot, 5 * sizeof(float), cudaMemcpyHostToDevice, st));
  }
  if ((rc = ensure(m->b_traj, out_floats))) return rc;
  if (want_y && (rc = ensure(m->b_ckpt, out_floats))) return rc;
  return CPZ_OK;
}
}  // namespace
extern "C" {

int cpz_rhs_jvp_dev(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, const float* x_dot,
                    const float* theta_dot, const float* mpp_dot, float* dxdt, float* dxdt_dot, size_t ncol) {
  int rc = check_jvp_args(m, "rhs_jvp", x, bcs, diurnal_Q, x_dot, theta_dot, mpp_dot, dxdt_dot, ncol);
  if (rc) return rc;
  int grid = 0;
  JvpArgs a = jvp_args(m, x, bcs, diurnal_Q, x_dot, theta_dot, mpp_dot, dxdt, dxdt_dot, ncol, grid);
  a.t = t;
  return launch_rhs_jvp(m, a, grid);
}

int cpz_rhs_jvp(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, const float* x_dot,
                const float* theta_dot, const float* mpp_dot, float* dxdt, float* dxdt_dot, size_t ncol) {
  int rc = check_jvp_args(m, "rhs_jvp", x, bcs, diurnal_Q, x_dot, theta_dot, mpp_dot, dxdt_dot, ncol);
  if (rc) return rc;
  const size_t n = ncol * (size_t)m->fwd.M.S;
  if ((rc = stage_jvp_inputs(m, x, bcs, diurnal_Q, x_dot, theta_dot, mpp_dot, ncol, n, dxdt != nullptr))) return rc;
  if ((rc = cpz_rhs_jvp_dev(m, m->b_x0.p, m->b_bcs.p, diurnal_Q ? m->b_q.p : nullptr, t, x_dot ? m->b_tgt.p : nullptr,
                            theta_dot ? m->b_red.p : nullptr, mpp_dot ? m->b_out.p : nullptr, dxdt ? m->b_ckpt.p : nullptr,
                            m->b_traj.p, ncol)))
    return rc;
  cudaStream_t st = m->ctx->stream;
  CPZ_CUDA(cudaMemcpyAsync(dxdt_dot, m->b_traj.p, n * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (dxdt) CPZ_CUDA(cudaMemcpyAsync(dxdt, m->b_ckpt.p, n * sizeof(float), cudaMemcpyDeviceToHost, st));
  CPZ_CUDA(cudaStreamSynchronize(st));
  return CPZ_OK;
}

// ---- predict_flux ---------------------------------------------------------------------------------------------------
int cpz_predict_flux_dev(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, float* flux, size_t ncol) {
  int rc = check_model(m);
  if (rc) return rc;
  if (ncol == 0) return CPZ_OK;
  if (!x || !bcs || !flux) return fail(CPZ_ERR_INVALID, "null array");
  if ((m->desc.flags & CPZ_FLAG_DIURNAL) && !diurnal_Q) return fail(CPZ_ERR_INVALID, "diurnal model needs diurnal_Q");
  if (ncol > (size_t)INT32_MAX / 512) return fail(CPZ_ERR_INVALID, "ncol too large");
  if ((rc = bind_device(m->ctx))) return rc;
  SolveArgs a{};
  a.theta = m->d_theta; a.x0 = x; a.bcs = bcs; a.Q = diurnal_Q; a.dxdt = flux; a.ncol = (int)ncol;
  a.rhs_only = 2; a.t_rhs = t; a.n_saved = 1; a.n_ckpt = 0;
  return launch_flux(m, a);
}

int cpz_predict_flux(cpz_model* m, const float* x, const float* bcs, const float* diurnal_Q, float t, float* flux, size_t ncol) {
  int rc = check_model(m);
  if (rc) return rc;
  if (ncol == 0) return CPZ_OK;
  if (!x || !bcs || !flux) return fail(CPZ_ERR_INVALID, "null array");
  if ((rc = bind_device(m->ctx))) return rc;
  if ((rc = upload_inputs(m, x, bcs, diurnal_Q, ncol))) return rc;
  const size_t rows = (size_t)m->fwd.M.nf * (m->fwd.M.Nz + 1);
  if ((rc = ensure(m->b_traj, ncol * rows))) return rc;
  if ((rc = cpz_predict_flux_dev(m, m->b_x0.p, m->b_bcs.p, diurnal_Q ? m->b_q.p : nullptr, t, m->b_traj.p, ncol))) return rc;
  CPZ_CUDA(cudaMemcpyAsync(flux, m->b_traj.p, ncol * rows * sizeof(float), cudaMemcpyDeviceToHost, m->ctx->stream));
  CPZ_CUDA(cudaStreamSynchronize(m->ctx->stream));
  return CPZ_OK;
}

// ---- forward solve ----------------------------------------------------------------------------------------------------
int cpz_solve_dev(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, float* traj, size_t ncol) {
  int rc = check_model(m);
  if (rc) return rc;
  if (ncol == 0) return CPZ_OK;
  if (!x0 || !bcs || !traj) return fail(CPZ_ERR_INVALID, "null array");
  if ((m->desc.flags & CPZ_FLAG_DIURNAL) && !diurnal_Q) return fail(CPZ_ERR_INVALID, "diurnal model needs diurnal_Q");
  if (ncol > (size_t)INT32_MAX / 512) return fail(CPZ_ERR_INVALID, "ncol too large");
  if ((rc = bind_device(m->ctx))) return rc;
  SolveArgs a{};
  a.theta = m->d_theta; a.x0 = x0; a.bcs = bcs; a.Q = diurnal_Q; a.traj = traj; a.ncol = (int)ncol;
  a.n_saved = n_saved_of(m->tm); a.n_ckpt = 0; a.rhs_only = 0;
  if ((rc = launch_solve(m, a))) return rc;
  // CPZ_ERR_NONFINITE reporting: the last saved frame is scanned on the device (a diverged explicit step shows up there)
  const size_t S = (size_t)m->fwd.M.S;
  return launch_check_finite(m->ctx, traj + (size_t)(a.n_saved - 1) * S, (size_t)a.n_saved * S, (int)ncol, (int)S);
}

int cpz_solve(cpz_model* m, const float* x0, const float* bcs, const float* diurnal_Q, float* traj, size_t ncol) {
  int rc = check_model(m);
  if (rc) return rc;
  if (ncol == 0) return CPZ_OK;
  if (!x0 || !bcs || !traj) return fail(CPZ_ERR_INVALID, "null array");
  // the same argument checks as cpz_solve_dev, made here because the chunked path below launches the kernels directly
  if ((m->desc.flags & CPZ_FLAG_DIURNAL) && !diurnal_Q) return fail(CPZ_ERR_INVALID, "diurnal model needs diurnal_Q");
  if (ncol > (size_t)INT32_MAX / 512) return fail(CPZ_ERR_INVALID, "ncol too large");
  if ((rc = bind_device(m->ctx))) return rc;
  if ((rc = begin_host_call(m->ctx))) return rc;
  if ((rc = upload_inputs(m, x0, bcs, diurnal_Q, ncol))) return rc;
  const size_t S = (size_t)m->fwd.M.S;
  const int n_saved = n_saved_of(m->tm);
  const size_t n = ncol * (size_t)n_saved * S;
  if ((rc = ensure(m->b_traj, n))) return rc;
  const float* dQ = diurnal_Q ? m->b_q.p : nullptr;
  // Long solves that save frames are cut into time chunks: while chunk k+1 integrates, the frames of chunk k go to the
  // host on a second stream (the trajectory is [ncol][n_saved][S], so a chunk is a 2-D sub-block).
  const TimeD tm_full = m->tm;
  const int n_frames = tm_full.save_stride > 0 ? tm_full.n_steps / tm_full.save_stride : 0;
  int n_chunks = 1;
  if (tm_full.save_stride > 0 && tm_full.n_steps % tm_full.save_stride == 0 && n * sizeof(float) >= ((size_t)64 << 20)) n_chunks = std::min(32, n_frames / 16);  // the un-overlapped tail is the last chunk's copy: 1/32 of the trajectory
  if (n_chunks > 1) {
    // The overlap needs a page-locked destination: cudaMemcpy2DAsync into pageable memory blocks the host until the copy
    // is done, so the next chunk's kernel would only be launched afterwards and chunking would be pure overhead.
    cudaPointerAttributes pa{};
    const cudaError_t pe = cudaPointerGetAttributes(&pa, traj);
    if (pe != cudaSuccess) cudaGetLastError();
    if (pe != cudaSuccess || pa.type != cudaMemoryTypeHost) n_chunks = 1;
  }
  if (n_chunks <= 1) {
    if ((rc = cpz_solve_dev(m, m->b_x0.p, m->b_bcs.p, dQ, m->b_traj.p, ncol))) return rc;
    CPZ_CUDA(cudaMemcpyAsync(traj, m->b_traj.p, n * sizeof(float), cudaMemcpyDeviceToHost, m->ctx->stream));
    CPZ_CUDA(cudaStreamSynchronize(m->ctx->stream));
    return report_nonfinite(m->ctx, "the final frame of the solve");
  }
  cpz_ctx* c = m->ctx;
  if (!c->copy_stream) {
    CPZ_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (auto& e : c->chunk_ev) CPZ_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  }
  const size_t pitch = (size_t)n_saved * S * sizeof(float);
  const int fpc = (n_frames + n_chunks - 1) / n_chunks;  // frames per chunk
  int f0 = 0;                                            // frames (after the initial one) already integrated
  for (int k = 0; f0 < n_frames; ++k) {
    const int nf = std::min(fpc, n_frames - f0);
    SolveArgs a{};
    a.theta = m->d_theta; a.bcs = m->b_bcs.p; a.Q = dQ; a.ncol = (int)ncol; a.n_saved = n_saved; a.n_ckpt = 0; a.rhs_only = 0;
    if (k == 0) { a.x0 = m->b_x0.p; a.traj = m->b_traj.p; }
    else { a.x0 = m->b_traj.p + (size_t)f0 * S; a.x0_stride = (size_t)n_saved * S; a.skip_frame0 = 1; a.traj = m->b_traj.p + (size_t)(f0 + 1) * S; }
    m->tm = tm_full;
    m->tm.step0 = f0 * tm_full.save_stride;  // stage times are t0 + (step0 + n) dt, bitwise those of a single launch
    m->tm.n_steps = nf * tm_full.save_stride;
    rc = launch_solve(m, a);
    m->tm = tm_full;
    if (rc) return rc;
    cudaEvent_t ev = c->chunk_ev[k & 1];
    CPZ_CUDA(cudaEventRecord(ev, c->stream));
    CPZ_CUDA(cudaStreamWaitEvent(c->copy_stream, ev, 0));
    const int first = k == 0 ? 0 : f0 + 1, count = k == 0 ? nf + 1 : nf;  // chunk 0 also carries the initial frame
    CPZ_CUDA(cudaMemcpy2DAsync(traj + (size_t)first * S, pitch, m->b_traj.p + (size_t)first * S, pitch, (size_t)count * S * sizeof(float), ncol,
                               cudaMemcpyDeviceToHost, c->copy_stream));
    f0 += nf;
  }
  if ((rc = launch_check_finite(c, m->b_traj.p + (size_t)(n_saved - 1) * S, (size_t)n_saved * S, (int)ncol, (int)S))) return rc;
  CPZ_CUDA(cudaStreamSynchronize(c->copy_stream));
  CPZ_CUDA(cudaStreamSynchronize(c->stream));
  return report_nonfinite(c, "the final frame of the solve");
}

}  // extern "C"

#include "cpz_capi_train.inc"
