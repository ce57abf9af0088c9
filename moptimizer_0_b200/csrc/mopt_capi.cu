// C ABI implementation (include/mopt_capi.h): contexts, the host-driven linearize / cost passes,
// the device-resident Levenberg-Marquardt driver and the optional NCCL shard reduction.
#include <dlfcn.h>

#include <cmath>
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "mopt_hyp_rule.h"
#include "mopt_internal.h"
#include "mopt_quant_rule.h"

using namespace mopt;

// ------------------------------------------------------------------------------ errors ----
namespace {
thread_local std::string g_last_error;
}
namespace mopt {
void set_last_error(const std::string& msg) { g_last_error = msg; }
int store_upload_async(mopt_store* st, int group, const void* host, int host_dtype, int64_t host_stride, int64_t first,
                       int64_t count);
}  // namespace mopt

// -------------------------------------------------------------------------------- NCCL ----
// Resolved at run time (dlopen) so the library has no link-time NCCL dependency and shares the
// copy already loaded by the host process (e.g. the one bundled with torch) when there is one.
namespace {
struct NcclApi {
  typedef struct ncclComm* comm_t;
  struct unique_id { char internal[MOPT_NCCL_ID_BYTES]; };
  int (*GetUniqueId)(unique_id*) = nullptr;
  int (*CommInitRank)(comm_t*, int, unique_id, int) = nullptr;
  int (*CommDestroy)(comm_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, comm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
  std::string why;
};
NcclApi& nccl() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* names[] = {getenv("MOPT_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    void* h = nullptr;
    for (const char* n : names) {
      if (!n) continue;
      h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (h) break;
    }
    if (!h) {
      api.why = std::string("cannot dlopen libnccl: ") + (dlerror() ? dlerror() : "?");
      return;
    }
    api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(h, "ncclGetUniqueId"));
    api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(h, "ncclCommInitRank"));
    api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(h, "ncclCommDestroy"));
    api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(dlsym(h, "ncclAllReduce"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(h, "ncclGetErrorString"));
    api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllReduce && api.GetErrorString;
    if (!api.ok) api.why = "libnccl is missing required symbols";
  });
  return api;
}
constexpr int kNcclFloat64 = 8;  // ncclFloat64 / ncclDouble (nccl.h)
constexpr int kNcclSum = 0;      // ncclSum

#define MOPT_NCCL_TRY(expr)                                                                       \
  do {                                                                                            \
    int _r = (expr);                                                                              \
    if (_r != 0) {                                                                                \
      set_last_error(std::string(#expr) + " failed: " + nccl().GetErrorString(_r));               \
      return MOPT_ERR_COMM;                                                                       \
    }                                                                                             \
  } while (0)
}  // namespace

// ----------------------------------------------------------------------------- kernels ----
namespace {

// model->setup(x) for one cost slot (and its finite-difference perturbations).  x travels as a
// kernel argument, so back-to-back asynchronous calls need no staging buffer.
__global__ void setup_kernel(CostSlot* slot, XArg x) { setup_cost(slot->cost, x.v, &slot->pb, threadIdx.x, blockDim.x); }

// levenberg_marquadt_dyn.cpp:15-26 (prepare) + the first setup(x0).
__global__ void lm_init_kernel(LmState* st, CostSlot* slots, LmInit in) {
  __shared__ LmStepShared s_sh;
  lm_init_warp(st, slots, in, &s_sh, threadIdx.x);
}

// One optimizer transition between passes; also publishes the done flag of this slot to the host.
__global__ void lm_step_kernel(LmState* st, const PassResult* trial, CostSlot* slots, int* flag, const int* xerr, int P,
                               int scalar_f32) {
  __shared__ LmStepShared s_sh;
  const int lane = threadIdx.x;
  if (*reinterpret_cast<const volatile int*>(xerr)) {  // a peer exchange timed out: `trial` is not a total
    if (lane == 0) {
      if (!st->done) lm_finish(st, MOPT_FATAL_ERROR);
      *flag = 1;
    }
    return;
  }
  const int done = lm_step_warp(st, trial, slots, &s_sh, lane, P, scalar_f32 != 0, LmStepIo{});
  if (lane == 0) *flag = done;
}

// The same solve through the warp-cooperative LDL^T (mopt_ldlt_solve with cooperative = 1; for tests).
__global__ void ldlt_warp_test_kernel(int n, const double* A, const double* rhs, double* out) {
  __shared__ LmSolveScratch sc;
  const int lane = threadIdx.x;
  for (int i = lane; i < n * n; i += 32) sc.A[i] = A[i];
  if (lane < n) sc.nb[lane] = rhs[lane];
  __syncwarp();
  if (n == 6) ldlt_solve_warp<double, 6>(n, sc.A, sc.nb, sc.d, sc.tmp, sc.y, sc.tr, lane);  // the unrolled instantiation
  else ldlt_solve_warp<double>(n, sc.A, sc.nb, sc.d, sc.tmp, sc.y, sc.tr, lane);
  if (lane < n) out[lane] = sc.d[lane];
}

// Consumer side of the NVLink peer exchange (mopt_pass.cuh peer_push): acquire every rank's sequence flag for
// this exchange, then sum the slots in rank order into `out` — identical bits on every rank.
__global__ void peer_reduce_kernel(XSlot* local, int world, unsigned long long seq, PassResult* out, int npk,
                                   const int* mode_ptr, int mode_override, int* err, int* err_dev) {
  const int mode = mode_override >= 0 ? mode_override : *mode_ptr;
  if (mode == PASS_SKIP) return;  // the optimizer finished: no rank pushed, nothing to wait for
  if (*reinterpret_cast<const volatile int*>(err_dev)) return;  // an earlier exchange already failed
  const int base = int(seq & 1ull) * kMaxWorld;
  __shared__ int s_ok;
  if (threadIdx.x == 0) {
    bool ok = true;
    const long long t0 = clock64();
    for (int r = 0; r < world && ok; ++r) {
      const unsigned long long* flag = &local[base + r].seq;
      for (;;) {
        unsigned long long v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
        if (v == seq) break;
        if (clock64() - t0 > 20000000000LL) {  // ~10 s: a peer died; fail loudly instead of hanging the GPU
          ok = false;
          break;
        }
        __nanosleep(64);
      }
    }
    if (!ok) {
      *err = 1;
      *err_dev = 1;
    }
    s_ok = ok ? 1 : 0;
    __threadfence_system();
  }
  __syncthreads();
  if (!s_ok) return;
  for (int k = threadIdx.x; k < npk; k += blockDim.x) {
    double s = 0.0;
    for (int r = 0; r < world; ++r) s += *reinterpret_cast<volatile double*>(&local[base + r].v[k]);
    out->v[k] = s;
  }
}

__global__ void ldlt_test_kernel(int n, double* A, const double* rhs, double* out) { ldlt_solve_dev<double>(n, A, rhs, out); }

}  // namespace

// ----------------------------------------------------------------------------- helpers ----
namespace {

// Where x holds a rotation vector (x[3..5] for the builtin point2point and camera models, the declared offset for a
// user model), or -1.
int rot_offset(int model) {
  if (model >= MOPT_MODEL_USER_BASE) return user_model_rot_offset(model);
  return (model == MOPT_MODEL_POINT2POINT || model == MOPT_MODEL_PINHOLE || model == MOPT_MODEL_PINHOLE_DISTORT) ? 3
                                                                                                               : -1;
}

}  // namespace

namespace mopt {

int validate_problem(const mopt_store* st, const mopt_problem* p, bool need_linearize) {
  MOPT_REQUIRE(st && p, "null store/problem");
  MOPT_REQUIRE(p->model == st->model, "problem.model differs from the store's model");
  const ModelShape sh = model_shape(p->model);
  MOPT_REQUIRE(sh.P >= 0, "unknown model kind");
  MOPT_REQUIRE(p->num_parameters == sh.P, "num_parameters does not match the builtin model");
  MOPT_REQUIRE(p->num_outputs == sh.O, "num_outputs does not match the builtin model");
  MOPT_REQUIRE(p->compute_dtype == MOPT_F32 || p->compute_dtype == MOPT_F64, "bad compute dtype");
  MOPT_REQUIRE(p->loss >= MOPT_LOSS_NONE && p->loss <= MOPT_LOSS_HUBER, "unknown loss kind");
  MOPT_REQUIRE(p->jacobian >= MOPT_JAC_ANALYTICAL && p->jacobian <= MOPT_JAC_CENTRAL, "unknown jacobian mode");
  if (need_linearize) {
    MOPT_REQUIRE(sh.P > 0, "this model has no parameters; only mopt_compute_cost is defined for it");
    if (p->jacobian == MOPT_JAC_ANALYTICAL && !sh.has_analytical) {
      // BaseModel::f_df throws for Jacobian-free models (include/moptimizer/model.h:66-70)
      set_last_error("Non implemented non-jacobian model function `f_df` being used.");
      return MOPT_ERR_UNSUPPORTED;
    }
  }
  if (p->model == MOPT_MODEL_POINT2POINT)
    MOPT_REQUIRE(p->variant >= MOPT_P2P_EXACT && p->variant <= MOPT_P2P_LEFT, "unknown point2point variant");
  MOPT_REQUIRE(p->manifold == MOPT_MANIFOLD_ADDITIVE || p->manifold == MOPT_MANIFOLD_SO3_LEFT, "unknown manifold");
  if (p->manifold == MOPT_MANIFOLD_SO3_LEFT)
    MOPT_REQUIRE(rot_offset(p->model) >= 0, "MOPT_MANIFOLD_SO3_LEFT needs a model whose x[3..5] is a rotation vector");
  if (p->has_covariance) {
    const int O = sh.O;
    for (int r = 0; r < O; ++r)
      for (int c = 0; c < r; ++c)
        if (p->covariance[r + c * O] != p->covariance[c + r * O]) {
          set_last_error("covariance must be symmetric (only the upper triangle of H is accumulated)");
          return MOPT_ERR_UNSUPPORTED;
        }
  }
  // no kernel reads an fp64 store into fp32 arithmetic (with_dtypes)
  if (st->dtype == MOPT_F64 && p->compute_dtype == MOPT_F32) {
    set_last_error("store dtype f64 with compute dtype f32 is not supported");
    return MOPT_ERR_UNSUPPORTED;
  }
  return MOPT_OK;
}

}  // namespace mopt

namespace {

void fill_cost(const mopt_problem* p, CostDev* c) {
  std::memset(c, 0, sizeof(*c));
  c->model = p->model; c->variant = p->variant; c->P = p->num_parameters; c->O = p->num_outputs;
  c->jacobian = p->jacobian; c->loss = p->loss; c->has_cov = p->has_covariance ? 1 : 0;
  c->compute_dtype = p->compute_dtype; c->loss_param = p->loss_param;
  c->manifold = p->manifold;
  c->rot_offset = rot_offset(p->model);
  c->so3_guard = ((p->flags & MOPT_FLAG_REFERENCE_FLOAT_GUARD) && p->compute_dtype == MOPT_F32) ? kSo3GuardF32 : kSo3GuardF64;
  const int O = p->num_outputs;
  for (int i = 0; i < O * O; ++i) c->cov[i] = p->has_covariance ? p->covariance[i] : ((i % (O + 1) == 0) ? 1.0 : 0.0);
  std::memcpy(c->consts, p->consts, sizeof(c->consts));
}

// Copy the cost constants of slot `i` to the device unless they are already there.
int stage_cost(mopt_ctx* ctx, int i, const mopt_problem* p) {
  CostDev c;
  fill_cost(p, &c);
  if (ctx->cached_valid[i] && std::memcmp(&c, &ctx->cached_cost[i], sizeof(c)) == 0) return MOPT_OK;
  // h_slot is reused as a pinned bounce buffer: wait until earlier copies from it have been consumed
  MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  ctx->h_slot->cost = c;
  MOPT_CUDA_TRY(cudaMemcpyAsync(&ctx->d_slots[i].cost, &ctx->h_slot->cost, sizeof(CostDev), cudaMemcpyHostToDevice, ctx->stream));
  MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  ctx->cached_cost[i] = c;
  ctx->cached_valid[i] = true;
  return MOPT_OK;
}

}  // namespace

namespace mopt {

PassArgs make_args(mopt_ctx* ctx, const mopt_store* st, int slot, int accumulate, int mode_override) {
  PassArgs a;
  std::memset(&a, 0, sizeof(a));
  for (int s = 0; s < kMaxStreams; ++s) a.streams.p[s] = st->streams[s];
  a.n = st->n;
  a.pb = &ctx->d_slots[slot].pb;
  a.cost = &ctx->d_slots[slot].cost;
  a.partials = ctx->d_partials;
  a.ticket = ctx->d_ticket;
  a.out = ctx->d_trial;
  a.accumulate = accumulate;
  a.mode_ptr = &ctx->d_lm->pass_mode;
  a.mode_override = mode_override;
  a.masked = st->may_have_invalid ? 1 : 0;
  return a;
}

}  // namespace mopt

namespace {

// `push`: this pass completes the rank-local result (last cost term), so its last CTA also pushes the packed
// result to every peer when the NVLink exchange is open.
// Host-driven passes of the analytical point2point model carry x into the kernel, which runs setup(x) itself
// (PassArgs::fused_setup): the step is one kernel instead of setup kernel + pass kernel.
// Sharded contexts too since round 2: with the second-generation kernel the 2-GPU A/B gives 0.3501 ms per lock-step
// step fused against 0.3565 ms with the setup kernel in front (round 1's kernel showed no difference,
// profiles/r1_fused_setup_ab_n2.txt); the packed results are bit-identical either way (bench.py check.vs_single_gpu
// compares a fused single-GPU context with the sharded ones).  MOPT_FUSED_SETUP=0 never fuses.
bool can_fuse_setup(const mopt_ctx* ctx, const mopt_problem* p, const mopt_store* st) {
  static const int env = [] {
    const char* e = getenv("MOPT_FUSED_SETUP");
    return (e && e[0]) ? (e[0] == '0' ? 0 : 1) : -1;
  }();
  if (env == 0) return false;
  // Finite differences of a parameter-only builtin model on the packed fp32 kernel (dense_f2_kernel, the condition of
  // launch_one in mopt_pass_dense.cu): a set is x +- h e_j, every CTA's first warp derives them itself.  (For the camera
  // models a set costs an so3::Exp and two matrix products per CTA: no gain over the set-up kernel, not fused.)
  if (p->model == MOPT_MODEL_EXP_CURVE && p->jacobian != MOPT_JAC_ANALYTICAL && st->dtype == MOPT_F32 &&
      p->compute_dtype == MOPT_F32 && !(p->flags & MOPT_FLAG_GENERIC_KERNEL) && !p->has_covariance &&
      !st->may_have_invalid && ctx->threads != 1024)
    return true;
  return p->model == MOPT_MODEL_POINT2POINT && p->jacobian == MOPT_JAC_ANALYTICAL &&
         p->manifold == MOPT_MANIFOLD_ADDITIVE;
}

}  // namespace

namespace mopt {

PassLaunch pass_launch(const mopt_ctx* ctx, const mopt_problem* p) {
  PassLaunch L{ctx->stream, ctx->num_sms, ctx->ctas_per_sm, ctx->threads};
  // finite differences over a common denominator (AFFINE_FD): the default with fp32 compute, opt-in with fp64
  L.affine_fd = (p->compute_dtype == MOPT_F32) ? !(p->flags & MOPT_FLAG_GENERIC_KERNEL)
                                               : ((p->flags & MOPT_FLAG_STABLE_FD) && !(p->flags & MOPT_FLAG_GENERIC_KERNEL));
  L.identity_cov = !p->has_covariance;
  return L;
}

}  // namespace mopt

namespace {

int launch_pass(mopt_ctx* ctx, const mopt_store* st, const mopt_problem* p, int slot, int accumulate, int mode_override,
                bool push, const XArg* fused_x = nullptr) {
  PassArgs a = make_args(ctx, st, slot, accumulate, mode_override);
  if (fused_x) {
    a.fused_setup = 1;
    a.x = *fused_x;
  }
  if (push && ctx->world > 1 && ctx->peers_open && ctx->exchange_enabled) {
    for (int r = 0; r < ctx->world; ++r) a.peer.base[r] = ctx->peer_base[r];
    a.peer.world = ctx->world;
    a.peer.rank = ctx->rank;
    a.peer.push = 1;
    a.peer.fused = ctx->fused_consumer ? 1 : 0;
    a.peer.err = ctx->d_xerr;
    a.peer.err_dev = ctx->d_xerr_dev;
    a.peer.seq = ++ctx->xseq;
  }
  const PassLaunch L = pass_launch(ctx, p);
  if (p->model >= MOPT_MODEL_USER_BASE)
    return launch_user(L, ctx->device, p->model, p->jacobian != MOPT_JAC_ANALYTICAL, st->dtype, p->compute_dtype, a);
  if (p->model == MOPT_MODEL_POINT2POINT && p->jacobian == MOPT_JAC_ANALYTICAL)
    return launch_p2p_moment(L, st->dtype, p->compute_dtype, p->loss,
                             p->variant == MOPT_P2P_EXACT || p->variant == MOPT_P2P_LEFT, a);
  // finite differences of an affine residual are affine in the source point: moment kernel with q = p
  // (mopt_setup.cuh fills the affine pieces); cost-only passes of this model take the same kernel
  if (p->model == MOPT_MODEL_POINT2POINT && !(p->flags & MOPT_FLAG_GENERIC_KERNEL))
    return launch_p2p_moment(L, st->dtype, p->compute_dtype, p->loss, false, a);
  if (is_wide(p->num_parameters)) return launch_wide(L, p->model, st->dtype, p->compute_dtype, a);
  return launch_dense(L, p->model, p->jacobian != MOPT_JAC_ANALYTICAL, st->dtype, p->compute_dtype, a);
}

// The analysis kernels below (score Gram, evaluation, quantile sweep, hypothesis scores) have one launcher each for
// builtin and run-time compiled models alike: the kernel resolves to a KernelDesc, and its grid follows from the same
// work items by the same rule (persistent_grid) whichever model it is.

// Score Gram sums (mopt_covariance_terms) of cost term `slot`, staged by setup_slot, into `out`: the Jacobian form
// launch_pass selects for the same problem (score_gram_kernel_desc picks the common-denominator differences where
// pass_launch's affine_fd and the model allow them, as launch_dense / launch_wide do).
int launch_cov_pass(mopt_ctx* ctx, const mopt_store* st, const mopt_problem* p, int slot, double* out) {
  PassLaunch L = pass_launch(ctx, p);
  const bool numeric = p->jacobian != MOPT_JAC_ANALYTICAL;
  int form = numeric ? COV_JAC_FD : COV_JAC_ANALYTICAL;
  if (p->model == MOPT_MODEL_POINT2POINT && (!numeric || !(p->flags & MOPT_FLAG_GENERIC_KERNEL)))
    form = COV_JAC_P2P_AFFINE;
  KernelDesc k;
  MOPT_TRY(p->model >= MOPT_MODEL_USER_BASE
               ? user_kernel(ctx->device, p->model, KIND_COV, st->dtype, p->compute_dtype, numeric, &k)
               : score_gram_kernel_desc(p->model, form, L.affine_fd, st->dtype, p->compute_dtype, &k));
  // work items as the pass kernels count them: 16-byte groups (P <= 6), residuals (wide tier); like the builtin dense
  // and wide passes, the kernel keeps its full occupancy whatever mopt_ctx_set_launch asks
  const ModelShape sh = model_shape(p->model);
  const int64_t items = sh.NS == 0 ? 1 : (sh.P <= 6 ? st->n / store_vec(st->dtype) : st->n);
  L.ctas_per_sm = 0;
  const int grid = persistent_grid(k.occupancy, k.threads, L, items);
  PassArgs a = make_args(ctx, st, slot, 0, PASS_LINEARIZE);
  CovArgs cv;
  cv.out = out;
  cv.qrot = (!numeric && (p->variant == MOPT_P2P_EXACT || p->variant == MOPT_P2P_LEFT)) ? 1 : 0;
  void* params[] = {&a, &cv};
  MOPT_CUDA_TRY(cudaLaunchKernel(k.fn, dim3(unsigned(grid)), dim3(unsigned(k.threads)), params, 0, ctx->stream));
  return MOPT_OK;
}

// Per-residual evaluation (mopt_evaluate): evaluate_kernel of the model on set 0 of slot 0 (staged by setup_slot),
// reducing its statistics through the same partials / ticket as the passes.
int launch_eval(mopt_ctx* ctx, const mopt_store* st, const mopt_problem* p, int out_dtype, const EvalArgs& ev) {
  KernelDesc k[2];  // fp32, fp64 outputs
  for (int o = 0; o < 2; ++o)
    MOPT_TRY(p->model >= MOPT_MODEL_USER_BASE
                 ? user_kernel(ctx->device, p->model, KIND_EVAL, st->dtype, p->compute_dtype, o == 1, &k[o])
                 : evaluate_kernel_desc(p->model, st->dtype, p->compute_dtype, o == 1, &k[o]));
  // One grid for both output dtypes (the smaller of their persistent grids), so that the statistics -- whose
  // summation order follows the grid -- do not depend on which outputs are written or in which dtype.
  const PassLaunch L = pass_launch(ctx, p);
  const int64_t groups = ev.count / store_vec(st->dtype) + 1;
  const int g0 = persistent_grid(k[0].occupancy, k[0].threads, L, groups);
  const int g1 = persistent_grid(k[1].occupancy, k[1].threads, L, groups);
  const KernelDesc& kern = k[out_dtype == MOPT_F64 ? 1 : 0];
  PassArgs a = make_args(ctx, st, 0, 0, PASS_COST);
  EvalArgs e = ev;
  void* params[] = {&a, &e};
  MOPT_CUDA_TRY(cudaLaunchKernel(kern.fn, dim3(unsigned(g0 < g1 ? g0 : g1)), dim3(unsigned(kern.threads)), params, 0,
                                 ctx->stream));
  return MOPT_OK;
}

// One radix-select sweep (mopt_residual_quantiles) of the model, on set 0 of slot 0.
int launch_quant_sweep(mopt_ctx* ctx, const mopt_store* st, const mopt_problem* p, const QuantArgs& qa) {
  KernelDesc k;
  MOPT_TRY(p->model >= MOPT_MODEL_USER_BASE
               ? user_kernel(ctx->device, p->model, KIND_QUANT, st->dtype, p->compute_dtype, false, &k)
               : quantile_sweep_kernel_desc(p->model, st->dtype, p->compute_dtype, &k));
  const int grid = persistent_grid(k.occupancy, k.threads, pass_launch(ctx, p), qa.count / store_vec(st->dtype) + 1);
  PassArgs a = make_args(ctx, st, 0, 0, PASS_COST);
  QuantArgs q = qa;
  void* params[] = {&a, &q};
  MOPT_CUDA_TRY(cudaLaunchKernel(k.fn, dim3(unsigned(grid)), dim3(unsigned(k.threads)), params, 0, ctx->stream));
  return MOPT_OK;
}

// Hypothesis scores (mopt_score_hypotheses) of the model, from the sets in h.sets.  The grid follows the elements
// only: the CTA partition of the data, and with it every per-CTA partial, is the same whatever the batch.
int launch_hyp_score(mopt_ctx* ctx, const mopt_store* st, const mopt_problem* p, const HypArgs& h) {
  KernelDesc k;
  MOPT_TRY(p->model >= MOPT_MODEL_USER_BASE
               ? user_kernel(ctx->device, p->model, KIND_HYP, st->dtype, p->compute_dtype, false, &k)
               : hypothesis_score_kernel_desc(p->model, st->dtype, p->compute_dtype, &k));
  const int grid = persistent_grid(k.occupancy, k.threads, pass_launch(ctx, p), h.count / store_vec(st->dtype) + 1);
  PassArgs a = make_args(ctx, st, 0, 0, PASS_COST);
  HypArgs ha = h;
  void* params[] = {&a, &ha};
  MOPT_CUDA_TRY(cudaLaunchKernel(k.fn, dim3(unsigned(grid), unsigned((h.n_hyp + kHypTile - 1) / kHypTile)),
                                 dim3(unsigned(k.threads)), params, 0, ctx->stream));
  return MOPT_OK;
}

// The buffers of mopt_score_hypotheses, on its first call on this context (the partials take 48 MB).
int hyp_alloc(mopt_ctx* ctx) {
  // each buffer on its own: after a failed allocation the next call allocates only what is missing
  constexpr size_t kTiles = MOPT_MAX_HYPOTHESES / kHypTile;
  if (!ctx->h_hyp)
    MOPT_CUDA_TRY(cudaHostAlloc(&ctx->h_hyp, sizeof(double) * MOPT_MAX_HYPOTHESES * kMaxP, cudaHostAllocDefault));
  if (!ctx->d_hyp_x) MOPT_CUDA_TRY(cudaMalloc(&ctx->d_hyp_x, sizeof(double) * MOPT_MAX_HYPOTHESES * kMaxP));
  if (!ctx->d_hyp_sets) MOPT_CUDA_TRY(cudaMalloc(&ctx->d_hyp_sets, sizeof(double) * MOPT_MAX_HYPOTHESES * kSetSize));
  if (!ctx->d_hyp_partials)
    MOPT_CUDA_TRY(cudaMalloc(&ctx->d_hyp_partials, sizeof(double) * kTiles * kHypRows * kMaxGrid));
  if (!ctx->d_hyp_out) MOPT_CUDA_TRY(cudaMalloc(&ctx->d_hyp_out, sizeof(double) * MOPT_MAX_HYPOTHESES * kHypStats));
  if (!ctx->d_hyp_tickets) {
    // zeroed on the context stream, ahead of the first score kernel (the stream does not wait for the default one)
    unsigned int* t = nullptr;
    MOPT_CUDA_TRY(cudaMalloc(&t, sizeof(unsigned int) * kTiles));
    const cudaError_t e = cudaMemsetAsync(t, 0, sizeof(unsigned int) * kTiles, ctx->stream);
    if (e != cudaSuccess) cudaFree(t);
    MOPT_CUDA_TRY(e);
    ctx->d_hyp_tickets = t;
  }
  return MOPT_OK;
}

// An output of mopt_evaluate must be device memory the context's device can write.
int check_device_output(const mopt_ctx* ctx, const void* ptr, const char* what) {
  if (!ptr) return MOPT_OK;
  cudaPointerAttributes attr;
  const cudaError_t e = cudaPointerGetAttributes(&attr, ptr);
  if (e != cudaSuccess) (void)cudaGetLastError();
  MOPT_REQUIRE(e == cudaSuccess && (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged) &&
                   attr.device == ctx->device,
               std::string(what) + " must be device memory on the context's device");
  return MOPT_OK;
}

int allreduce_trial(mopt_ctx* ctx, int P, int mode_override) {
  if (ctx->world <= 1 || !ctx->exchange_enabled) return MOPT_OK;
  if (ctx->peers_open) {
    if (ctx->fused_consumer) return MOPT_OK;  // the pass kernel's last CTA already wrote the totals (peer_push)
    peer_reduce_kernel<<<1, 64, 0, ctx->stream>>>(ctx->d_xbuf, ctx->world, ctx->xseq, ctx->d_trial, packed_size(P),
                                                  &ctx->d_lm->pass_mode, mode_override, ctx->d_xerr, ctx->d_xerr_dev);
    MOPT_CUDA_TRY(cudaGetLastError());
    return MOPT_OK;
  }
  if (!ctx->nccl_comm) {
    set_last_error("sharded context has neither a NCCL communicator nor an open peer exchange");
    return MOPT_ERR_COMM;
  }
  MOPT_NCCL_TRY(nccl().AllReduce(ctx->d_trial, ctx->d_trial, size_t(packed_size(P)), kNcclFloat64, kNcclSum,
                                 static_cast<NcclApi::comm_t>(ctx->nccl_comm), ctx->stream));
  return MOPT_OK;
}

void unpack_result(const PassResult& r, int P, double* H, double* b, double* sum) {
  if (H)
    for (int i = 0; i < P; ++i)
      for (int j = i; j < P; ++j) {
        const double v = r.v[tri_index(P, i, j)];
        H[i + j * P] = v;
        H[j + i * P] = v;
      }
  if (b)
    for (int i = 0; i < P; ++i) b[i] = r.v[P * (P + 1) / 2 + i];
  if (sum) *sum = r.v[packed_size(P) - 1];
}

// After a peer-exchange timeout the sequence numbers of the ranks no longer agree: the context is unusable.
int check_exchange_alive(const mopt_ctx* ctx) {
  if (ctx->h_xerr && *reinterpret_cast<volatile int*>(ctx->h_xerr)) {
    set_last_error("an earlier peer exchange on this context timed out (a rank died); destroy the context");
    return MOPT_ERR_COMM;
  }
  return MOPT_OK;
}

int enqueue_pass(mopt_ctx* ctx, mopt_store* st, const mopt_problem* p, const double* x, int mode) {
  MOPT_TRY(check_exchange_alive(ctx));
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  MOPT_TRY(stage_cost(ctx, 0, p));
  const int P = p->num_parameters;
  XArg xa;
  std::memset(&xa, 0, sizeof(xa));
  if (P > 0) {
    MOPT_REQUIRE(x != nullptr, "null parameter vector");
    for (int i = 0; i < P; ++i) xa.v[i] = x[i];
  }
  if (can_fuse_setup(ctx, p, st)) {
    MOPT_TRY(launch_pass(ctx, st, p, 0, 0, mode, true, &xa));
  } else {
    setup_kernel<<<1, 32, 0, ctx->stream>>>(&ctx->d_slots[0], xa);
    MOPT_CUDA_TRY(cudaGetLastError());
    if (user_model_has_setup(p->model))
      MOPT_TRY(launch_user_setup(ctx->stream, ctx->device, p->model, &ctx->d_slots[0], nullptr, xa.v, P));
    MOPT_TRY(launch_pass(ctx, st, p, 0, 0, mode, true));
  }
  MOPT_TRY(allreduce_trial(ctx, P, mode));
  return MOPT_OK;
}

}  // namespace

namespace mopt {
int setup_slot(mopt_ctx* ctx, int slot, const mopt_problem* problem, const double* x) {
  MOPT_TRY(stage_cost(ctx, slot, problem));
  XArg xa;
  std::memset(&xa, 0, sizeof(xa));
  for (int i = 0; i < problem->num_parameters; ++i) xa.v[i] = x[i];
  setup_kernel<<<1, 32, 0, ctx->stream>>>(&ctx->d_slots[slot], xa);
  MOPT_CUDA_TRY(cudaGetLastError());
  if (user_model_has_setup(problem->model))
    MOPT_TRY(launch_user_setup(ctx->stream, ctx->device, problem->model, &ctx->d_slots[slot], nullptr, xa.v,
                               problem->num_parameters));
  return MOPT_OK;
}
}  // namespace mopt

namespace {

int fetch_result(mopt_ctx* ctx, int P, double* H, double* b, double* sum) {
  MOPT_CUDA_TRY(cudaMemcpyAsync(ctx->h_result, ctx->d_trial, sizeof(double) * packed_size(P), cudaMemcpyDeviceToHost, ctx->stream));
  MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  if (ctx->h_xerr && *reinterpret_cast<volatile int*>(ctx->h_xerr)) {
    set_last_error("peer exchange timed out waiting for another rank");
    return MOPT_ERR_COMM;
  }
  unpack_result(*ctx->h_result, P, H, b, sum);
  return MOPT_OK;
}

// Copies the final optimizer state back: x, status, iteration count and trace (end of mopt_lm_minimize).
// on_host: the kernel wrote the final state and the trace into ctx->h_lm itself (mapped memory; persistent LM kernel)
// and the stream has been synchronised: no copy, no second round trip.
int finish_lm(mopt_ctx* ctx, int P, double* x, mopt_lm_report* report, bool on_host = false) {
  // the state is 57 KB with its 1024-entry trace: fetch the hot part and the first trials, the rest only if used
  LmState* hs = ctx->h_lm;
  constexpr int kFirstTrials = 48;
  const size_t first = offsetof(LmState, trials) + sizeof(mopt_lm_trial) * kFirstTrials;
  if (!on_host) {
    MOPT_CUDA_TRY(cudaMemcpyAsync(hs, ctx->d_lm, first, cudaMemcpyDeviceToHost, ctx->stream));
    MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  }
  if (!on_host && hs->num_trials > kFirstTrials) {
    const int more = (hs->num_trials < MOPT_MAX_TRACE ? hs->num_trials : MOPT_MAX_TRACE) - kFirstTrials;
    MOPT_CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(hs) + first, reinterpret_cast<const char*>(ctx->d_lm) + first,
                                  sizeof(mopt_lm_trial) * size_t(more), cudaMemcpyDeviceToHost, ctx->stream));
    MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  }
  if (ctx->h_xerr && *reinterpret_cast<volatile int*>(ctx->h_xerr)) {
    set_last_error("peer exchange timed out waiting for another rank; this context cannot be used any more");
    return MOPT_ERR_COMM;
  }
  if (!hs->done) {
    set_last_error("internal error: the LM state machine did not terminate within its slot budget");
    return MOPT_ERR_CUDA;
  }
  for (int i = 0; i < P; ++i) x[i] = hs->x[i];
  report->status = hs->status;
  report->executed_iterations = hs->executed;
  report->num_trials = hs->num_trials < MOPT_MAX_TRACE ? hs->num_trials : MOPT_MAX_TRACE;
  report->num_passes = hs->num_passes;
  report->final_cost = hs->cur.v[packed_size(P) - 1];
  std::memcpy(report->trials, hs->trials, sizeof(mopt_lm_trial) * size_t(report->num_trials));
  return MOPT_OK;
}

int ctx_alloc(mopt_ctx* ctx) {
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  cudaDeviceProp prop;
  MOPT_CUDA_TRY(cudaGetDeviceProperties(&prop, ctx->device));
  ctx->num_sms = prop.multiProcessorCount;
  MOPT_CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  MOPT_CUDA_TRY(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  MOPT_CUDA_TRY(cudaMalloc(&ctx->d_partials, sizeof(double) * kMaxRaw * kMaxGrid));
  MOPT_CUDA_TRY(cudaMalloc(&ctx->d_ticket, sizeof(unsigned int)));
  MOPT_CUDA_TRY(cudaMemset(ctx->d_ticket, 0, sizeof(unsigned int)));
  MOPT_CUDA_TRY(cudaMalloc(&ctx->d_trial, sizeof(PassResult)));
  MOPT_CUDA_TRY(cudaMemset(ctx->d_trial, 0, sizeof(PassResult)));
  MOPT_CUDA_TRY(cudaMalloc(&ctx->d_slots, sizeof(CostSlot) * MOPT_MAX_COSTS));
  MOPT_CUDA_TRY(cudaMemset(ctx->d_slots, 0, sizeof(CostSlot) * MOPT_MAX_COSTS));
  MOPT_CUDA_TRY(cudaMalloc(&ctx->d_lm, sizeof(LmState)));
  MOPT_CUDA_TRY(cudaMemset(ctx->d_lm, 0, sizeof(LmState)));
  MOPT_CUDA_TRY(cudaHostAlloc(&ctx->h_result, sizeof(PassResult), cudaHostAllocDefault));
  MOPT_CUDA_TRY(cudaHostAlloc(&ctx->h_lm, sizeof(LmState), cudaHostAllocMapped));
  MOPT_CUDA_TRY(cudaHostGetDevicePointer(reinterpret_cast<void**>(&ctx->d_lm_host), ctx->h_lm, 0));
  MOPT_CUDA_TRY(cudaHostAlloc(&ctx->h_slot, sizeof(CostSlot), cudaHostAllocDefault));
  MOPT_CUDA_TRY(cudaMalloc(&ctx->d_xbuf, sizeof(XSlot) * 2 * kMaxWorld));
  MOPT_CUDA_TRY(cudaMemset(ctx->d_xbuf, 0, sizeof(XSlot) * 2 * kMaxWorld));
  MOPT_CUDA_TRY(cudaHostAlloc(&ctx->h_xerr, sizeof(int), cudaHostAllocMapped));
  *ctx->h_xerr = 0;
  MOPT_CUDA_TRY(cudaHostGetDevicePointer(&ctx->d_xerr, ctx->h_xerr, 0));
  MOPT_CUDA_TRY(cudaMalloc(&ctx->d_gen, 32 * sizeof(unsigned long long)));
  MOPT_CUDA_TRY(cudaMemset(ctx->d_gen, 0, 32 * sizeof(unsigned long long)));
  MOPT_CUDA_TRY(cudaMalloc(&ctx->d_xerr_dev, sizeof(int)));
  MOPT_CUDA_TRY(cudaMemset(ctx->d_xerr_dev, 0, sizeof(int)));
  MOPT_CUDA_TRY(cudaMalloc(&ctx->d_eval_stats, sizeof(double) * (kEvalSums + 1)));
  MOPT_CUDA_TRY(cudaMalloc(&ctx->d_align, sizeof(AlignAcc)));
  MOPT_CUDA_TRY(cudaMalloc(&ctx->d_cov_sums, sizeof(double) * MOPT_MAX_COSTS * kMaxRaw));
  MOPT_CUDA_TRY(cudaHostAlloc(&ctx->h_cov_sums, sizeof(double) * MOPT_MAX_COSTS * kMaxRaw, cudaHostAllocDefault));
  MOPT_CUDA_TRY(cudaMalloc(&ctx->d_quant, sizeof(QuantState)));
  ctx->flags_capacity = 4096;
  if (const char* e = getenv("MOPT_LM_FLAG_RING")) {  // test knob: a small ring makes an ordinary solve wrap it
    const int v = atoi(e);
    if (v >= 8 && v <= 4096) ctx->flags_capacity = v;
  }
  MOPT_CUDA_TRY(cudaHostAlloc(&ctx->h_flags, sizeof(int) * ctx->flags_capacity, cudaHostAllocMapped));
  MOPT_CUDA_TRY(cudaHostGetDevicePointer(&ctx->d_flags, ctx->h_flags, 0));
  for (int i = 0; i < 2; ++i) {
    MOPT_CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_copy[i], cudaEventDisableTiming));
    MOPT_CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_free[i], cudaEventDisableTiming));
    MOPT_CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_batch[i], cudaEventDisableTiming));
  }
  return MOPT_OK;
}

}  // namespace

// ============================================================================== C ABI ====
extern "C" {

const char* mopt_last_error(void) { return g_last_error.c_str(); }
const char* mopt_version(void) { return "moptimizer_0_b200 0.1 (sm_100a)"; }

int mopt_device_count(int* count) try {
  MOPT_REQUIRE(count, "null count");
  MOPT_CUDA_TRY(cudaGetDeviceCount(count));
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_ctx_create(int device, mopt_ctx** out) try {
  MOPT_REQUIRE(out, "null out");
  mopt_ctx* ctx = new mopt_ctx();
  ctx->device = device;
  const int s = ctx_alloc(ctx);
  if (s != MOPT_OK) {
    mopt_ctx_destroy(ctx);  // releases whatever ctx_alloc got before it failed (every member starts null)
    return s;
  }
  *out = ctx;
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_comm_unique_id(void* out_id) try {
  MOPT_REQUIRE(out_id, "null out_id");
  if (!nccl().ok) {
    set_last_error(nccl().why);
    return MOPT_ERR_COMM;
  }
  NcclApi::unique_id id;
  MOPT_NCCL_TRY(nccl().GetUniqueId(&id));
  std::memcpy(out_id, &id, MOPT_NCCL_ID_BYTES);
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_ctx_create_sharded(int device, int rank, int world_size, const void* nccl_unique_id, mopt_ctx** out) try {
  MOPT_REQUIRE(out, "null out");
  MOPT_REQUIRE(world_size >= 1 && rank >= 0 && rank < world_size, "bad rank/world_size");
  MOPT_REQUIRE(world_size <= kMaxWorld, "at most 8 ranks (one box) are supported");
  MOPT_TRY(mopt_ctx_create(device, out));
  mopt_ctx* ctx = *out;
  ctx->rank = rank;
  ctx->world = world_size;
  if (world_size > 1 && nccl_unique_id) {  // without an id the caller must open the NVLink peer exchange instead
    if (!nccl().ok) {
      set_last_error(nccl().why);
      mopt_ctx_destroy(ctx);
      *out = nullptr;
      return MOPT_ERR_COMM;
    }
    NcclApi::unique_id id;
    std::memcpy(&id, nccl_unique_id, MOPT_NCCL_ID_BYTES);
    NcclApi::comm_t comm = nullptr;
    const int r = nccl().CommInitRank(&comm, world_size, id, rank);
    if (r != 0) {
      set_last_error(std::string("ncclCommInitRank failed: ") + nccl().GetErrorString(r));
      mopt_ctx_destroy(ctx);
      *out = nullptr;
      return MOPT_ERR_COMM;
    }
    ctx->nccl_comm = comm;
  }
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_ctx_destroy(mopt_ctx* ctx) try {
  if (!ctx) return MOPT_OK;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->nccl_comm) nccl().CommDestroy(static_cast<NcclApi::comm_t>(ctx->nccl_comm));
  if (ctx->peers_open)
    for (int r = 0; r < ctx->world; ++r)
      if (r != ctx->rank && ctx->peer_base[r]) cudaIpcCloseMemHandle(ctx->peer_base[r]);
  cudaFree(ctx->d_xbuf);
  cudaFree(ctx->d_xerr_dev);
  cudaFree(ctx->d_gen);
  cudaFree(ctx->d_eval_stats);
  cudaFree(ctx->d_align);
  cudaFree(ctx->d_cov_sums);
  cudaFree(ctx->d_quant);
  cudaFree(ctx->d_hyp_x);
  cudaFree(ctx->d_hyp_sets);
  cudaFree(ctx->d_hyp_partials);
  cudaFree(ctx->d_hyp_tickets);
  cudaFree(ctx->d_hyp_out);
  if (ctx->h_hyp) cudaFreeHost(ctx->h_hyp);
  if (ctx->h_cov_sums) cudaFreeHost(ctx->h_cov_sums);
  if (ctx->h_xerr) cudaFreeHost(ctx->h_xerr);
  cudaFree(ctx->d_partials); cudaFree(ctx->d_ticket); cudaFree(ctx->d_trial);
  cudaFree(ctx->d_slots); cudaFree(ctx->d_lm);
  for (int i = 0; i < 2; ++i) {
    if (ctx->d_stage[i]) cudaFree(ctx->d_stage[i]);
    if (ctx->ev_copy[i]) cudaEventDestroy(ctx->ev_copy[i]);
    if (ctx->ev_free[i]) cudaEventDestroy(ctx->ev_free[i]);
    if (ctx->ev_batch[i]) cudaEventDestroy(ctx->ev_batch[i]);
  }
  if (ctx->h_result) cudaFreeHost(ctx->h_result);
  if (ctx->h_lm) cudaFreeHost(ctx->h_lm);
  if (ctx->h_slot) cudaFreeHost(ctx->h_slot);
  if (ctx->h_flags) cudaFreeHost(ctx->h_flags);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  delete ctx;
  (void)cudaGetLastError();  // teardown of a half-built context (bad device id) must not leave an error behind for
                             // the next launch check of another context
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_ctx_peer_handle(mopt_ctx* ctx, void* out_handle) try {
  MOPT_REQUIRE(ctx && out_handle, "null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == MOPT_PEER_HANDLE_BYTES, "cudaIpcMemHandle_t size");
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  MOPT_CUDA_TRY(cudaIpcGetMemHandle(&h, ctx->d_xbuf));
  std::memcpy(out_handle, &h, sizeof(h));
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_ctx_open_peers(mopt_ctx* ctx, const void* handles) try {
  MOPT_REQUIRE(ctx && handles, "null argument");
  MOPT_REQUIRE(ctx->world > 1, "not a sharded context");
  MOPT_REQUIRE(!ctx->peers_open, "peers already open");
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  for (int r = 0; r < ctx->world; ++r) {
    if (r == ctx->rank) {
      ctx->peer_base[r] = ctx->d_xbuf;
      continue;
    }
    cudaIpcMemHandle_t h;
    std::memcpy(&h, static_cast<const char*>(handles) + size_t(r) * sizeof(h), sizeof(h));
    void* p = nullptr;
    MOPT_CUDA_TRY(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->peer_base[r] = static_cast<XSlot*>(p);
  }
  ctx->peers_open = true;
  const char* mode = getenv("MOPT_PEER_CONSUMER");  // "kernel": keep the separate one-warp consumer kernel (A/B)
  ctx->fused_consumer = !(mode && std::string(mode) == "kernel");
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_ctx_set_exchange_enabled(mopt_ctx* ctx, int enabled) try {
  MOPT_REQUIRE(ctx, "null ctx");
  ctx->exchange_enabled = enabled != 0;
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_ctx_synchronize(mopt_ctx* ctx) try {
  MOPT_REQUIRE(ctx, "null ctx");
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_ctx_stream(mopt_ctx* ctx, uint64_t* out_stream) try {
  MOPT_REQUIRE(ctx && out_stream, "null ctx/out");
  *out_stream = reinterpret_cast<uint64_t>(ctx->stream);
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_ctx_set_launch(mopt_ctx* ctx, int ctas_per_sm, int threads) try {
  MOPT_REQUIRE(ctx, "null ctx");
  MOPT_REQUIRE(ctas_per_sm >= 0 && ctas_per_sm <= 8, "ctas_per_sm must be in [0, 8]");
  ctx->ctas_per_sm = ctas_per_sm;
  ctx->threads = threads;
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_linearize(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const double* x, double* H, double* b,
                   double* sum) try {
  MOPT_REQUIRE(ctx && store && store->ctx == ctx, "store does not belong to this context");
  MOPT_TRY(validate_problem(store, problem, true));
  MOPT_TRY(enqueue_pass(ctx, store, problem, x, PASS_LINEARIZE));
  return fetch_result(ctx, problem->num_parameters, H, b, sum);
}
MOPT_ABI_CATCH

int mopt_compute_cost(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const double* x, double* sum) try {
  MOPT_REQUIRE(ctx && store && store->ctx == ctx, "store does not belong to this context");
  MOPT_TRY(validate_problem(store, problem, false));
  MOPT_TRY(enqueue_pass(ctx, store, problem, x, PASS_COST));
  return fetch_result(ctx, problem->num_parameters, nullptr, nullptr, sum);
}
MOPT_ABI_CATCH

int mopt_evaluate(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const double* x, int64_t first,
                  int64_t count, double inlier_threshold, int out_dtype, void* residuals, void* weights,
                  mopt_eval_stats* stats) try {
  MOPT_REQUIRE(ctx && store && store->ctx == ctx, "store does not belong to this context");
  MOPT_TRY(validate_problem(store, problem, false));
  MOPT_REQUIRE(first >= 0 && count >= 0 && first <= store->n && count <= store->n - first,
               "the range [first, first + count) must lie inside the store");
  MOPT_REQUIRE(out_dtype == MOPT_F32 || out_dtype == MOPT_F64, "out_dtype must be MOPT_F32 or MOPT_F64");
  MOPT_REQUIRE(residuals || weights || stats, "residuals, weights and stats are all NULL: nothing to evaluate");
  MOPT_REQUIRE(count > 0 || (!residuals && !weights), "residuals or weights requested for an empty range");
  MOPT_REQUIRE(problem->num_parameters == 0 || x, "null parameter vector");
  MOPT_REQUIRE(!(inlier_threshold < 0.0), "inlier_threshold must not be negative");
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  MOPT_TRY(check_device_output(ctx, residuals, "residuals"));
  MOPT_TRY(check_device_output(ctx, weights, "weights"));
  if (count == 0) {
    std::memset(stats, 0, sizeof(*stats));
    return MOPT_OK;
  }
  MOPT_TRY(setup_slot(ctx, 0, problem, x));
  EvalArgs ev;
  ev.first = first;
  ev.count = count;
  ev.r = residuals;
  ev.w = weights;
  ev.thr2 = inlier_threshold * inlier_threshold;
  ev.stats = ctx->d_eval_stats;
  MOPT_TRY(launch_eval(ctx, store, problem, out_dtype, ev));
  double* h = ctx->h_result->v;  // pinned bounce buffer (idle between calls)
  MOPT_CUDA_TRY(cudaMemcpyAsync(h, ctx->d_eval_stats, sizeof(double) * (kEvalSums + 1), cudaMemcpyDeviceToHost,
                                ctx->stream));
  MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  if (stats) {
    std::memset(stats, 0, sizeof(*stats));
    stats->n_valid = int64_t(h[0]);
    stats->n_inliers = int64_t(h[1]);
    stats->sum_sq = h[2];
    stats->inlier_sum_sq = h[3];
    stats->max_sq = h[4];
  }
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_score_hypotheses(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, int n_hyp, const double* xs,
                          int64_t first, int64_t count, double inlier_threshold, mopt_eval_stats* out) try {
  MOPT_REQUIRE(ctx && store && store->ctx == ctx, "store does not belong to this context");
  MOPT_TRY(validate_problem(store, problem, false));
  MOPT_REQUIRE(problem->num_parameters > 0, "a model without parameters has no hypotheses to score");
  MOPT_REQUIRE(n_hyp >= 1 && n_hyp <= MOPT_MAX_HYPOTHESES, "n_hyp must lie in [1, MOPT_MAX_HYPOTHESES]");
  MOPT_REQUIRE(xs && out, "null xs or out");
  MOPT_REQUIRE(first >= 0 && count >= 0 && first <= store->n && count <= store->n - first,
               "the range [first, first + count) must lie inside the store");
  MOPT_REQUIRE(!(inlier_threshold < 0.0), "inlier_threshold must not be negative");
  if (count == 0) {
    std::memset(out, 0, sizeof(*out) * size_t(n_hyp));
    return MOPT_OK;
  }
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  MOPT_TRY(hyp_alloc(ctx));
  MOPT_TRY(stage_cost(ctx, 0, problem));
  const int P = problem->num_parameters;
  double* h = ctx->h_hyp;  // pinned; idle between calls (each call returns after synchronising)
  std::memset(h, 0, sizeof(double) * size_t(n_hyp) * kMaxP);
  for (int k = 0; k < n_hyp; ++k)
    for (int i = 0; i < P; ++i) h[size_t(k) * kMaxP + i] = xs[size_t(k) * P + i];
  MOPT_CUDA_TRY(cudaMemcpyAsync(ctx->d_hyp_x, h, sizeof(double) * size_t(n_hyp) * kMaxP, cudaMemcpyHostToDevice,
                                ctx->stream));
  const CostDev* cost = &ctx->d_slots[0].cost;
  if (user_model_has_setup(problem->model))
    MOPT_TRY(launch_user_hypothesis_setup(ctx->stream, ctx->device, problem->model, cost, ctx->d_hyp_x, n_hyp,
                                          ctx->d_hyp_sets));
  else
    MOPT_TRY(launch_hypothesis_setup(ctx->stream, cost, ctx->d_hyp_x, n_hyp, ctx->d_hyp_sets));
  HypArgs ha;
  ha.first = first;
  ha.count = count;
  ha.n_hyp = n_hyp;
  ha.thr2 = inlier_threshold * inlier_threshold;  // as mopt_evaluate forms it
  ha.thr2f = largest_float_le(ha.thr2);
  ha.sets = ctx->d_hyp_sets;
  ha.partials = ctx->d_hyp_partials;
  ha.tickets = ctx->d_hyp_tickets;
  ha.out = ctx->d_hyp_out;
  MOPT_TRY(launch_hyp_score(ctx, store, problem, ha));
  MOPT_CUDA_TRY(cudaMemcpyAsync(h, ctx->d_hyp_out, sizeof(double) * size_t(n_hyp) * kHypStats, cudaMemcpyDeviceToHost,
                                ctx->stream));
  MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  for (int k = 0; k < n_hyp; ++k) {
    const double* v = h + size_t(k) * kHypStats;
    mopt_eval_stats& o = out[k];
    std::memset(&o, 0, sizeof(o));
    o.n_valid = int64_t(v[0]);
    o.n_inliers = int64_t(v[1]);
    o.sum_sq = v[2];
    o.inlier_sum_sq = v[3];
    o.max_sq = v[4];
  }
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_residual_quantiles(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const double* x,
                            int64_t first, int64_t count, int n_q, const double* q, mopt_quantiles* out) try {
  MOPT_REQUIRE(ctx && store && store->ctx == ctx, "store does not belong to this context");
  MOPT_TRY(validate_problem(store, problem, false));
  MOPT_REQUIRE(first >= 0 && count >= 0 && first <= store->n && count <= store->n - first,
               "the range [first, first + count) must lie inside the store");
  MOPT_REQUIRE(n_q >= 0 && n_q <= MOPT_MAX_QUANTILES, "n_q must lie in [0, MOPT_MAX_QUANTILES]");
  MOPT_REQUIRE(n_q == 0 || q, "null q");
  for (int k = 0; k < n_q; ++k) MOPT_REQUIRE(q[k] >= 0.0 && q[k] <= 1.0, "every q must lie in [0, 1]");
  MOPT_REQUIRE(out, "null out");
  MOPT_REQUIRE(problem->num_parameters == 0 || x, "null parameter vector");
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  QuantLevels lv;
  for (int k = 0; k < n_q; ++k) lv.q[k] = q[k];
  lv.q[n_q] = 0.5;  // the median
  // the head of the state: counts, target ranks and their keys (the histogram is zeroed by the steps)
  constexpr size_t kHead = offsetof(QuantState, rem);
  static_assert(kHead <= sizeof(PassResult), "the quantile result must fit the pinned bounce buffer");
  unsigned char* h = reinterpret_cast<unsigned char*>(ctx->h_result->v);
  if (count > 0) {
    MOPT_TRY(setup_slot(ctx, 0, problem, x));
    MOPT_CUDA_TRY(cudaMemsetAsync(ctx->d_quant, 0, sizeof(QuantState), ctx->stream));
    const int sweeps = problem->compute_dtype == MOPT_F32 ? 4 : 8;
    QuantArgs qa;
    qa.first = first;
    qa.count = count;
    qa.st = ctx->d_quant;
    for (int d = 0; d < sweeps; ++d) {
      qa.sweep = d;
      MOPT_TRY(launch_quant_sweep(ctx, store, problem, qa));
      MOPT_TRY(launch_quantile_step(ctx->stream, ctx->d_quant, d, n_q + 1, lv));
    }
    MOPT_CUDA_TRY(cudaMemcpyAsync(h, ctx->d_quant, kHead, cudaMemcpyDeviceToHost, ctx->stream));
    MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  } else {
    std::memset(h, 0, kHead);
  }
  QuantState head;
  std::memcpy(&head, h, kHead);
  mopt_quantiles r;
  std::memset(&r, 0, sizeof(r));
  r.n_ranked = int64_t(head.n_ranked);
  r.n_nan = int64_t(head.n_nan);
  // the selected key of rank j, as the fp64 value numpy ranks (the fp32 keys widen exactly)
  auto value_of = [&](int64_t j) -> double {
    for (int k = 0; k < head.n_rank; ++k)
      if (head.rank[k] == j) {
        if (problem->compute_dtype == MOPT_F32) {
          const uint32_t b = uint32_t(head.key[k]);
          float f;
          std::memcpy(&f, &b, sizeof(f));
          return double(f);
        }
        double v;
        std::memcpy(&v, &head.key[k], sizeof(v));
        return v;
      }
    return NAN;
  };
  for (int k = 0; k <= n_q; ++k) {
    double lo = NAN, hi = NAN, v = NAN;
    if (r.n_ranked > 0) {
      const QuantRank qr = quantile_rank(r.n_ranked, lv.q[k]);
      lo = value_of(qr.j);
      hi = value_of(qr.j1);
      MOPT_REQUIRE(!std::isnan(lo) && !std::isnan(hi), "internal error: a quantile rank was not selected");
      v = quantile_lerp(lo, hi, qr.t);
    }
    if (k < n_q) {
      r.lo[k] = lo;
      r.hi[k] = hi;
      r.value[k] = v;
    } else {
      r.median = v;
    }
  }
  for (int k = n_q; k < MOPT_MAX_QUANTILES; ++k) r.lo[k] = r.hi[k] = r.value[k] = NAN;
  r.robust_sigma = std::sqrt(r.median / chi2_median(problem->num_outputs));
  *out = r;
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_covariance_terms(mopt_ctx* ctx, int n_costs, mopt_store* const* stores, const mopt_problem* problems,
                          const double* x, mopt_cov_terms* out) try {
  MOPT_REQUIRE(ctx && stores && problems && out, "null argument");
  MOPT_REQUIRE(x, "null parameter vector");
  MOPT_REQUIRE(n_costs >= 1 && n_costs <= MOPT_MAX_COSTS, "n_costs must lie in [1, MOPT_MAX_COSTS]");
  const int P = problems[0].num_parameters;
  for (int c = 0; c < n_costs; ++c) {
    MOPT_REQUIRE(stores[c] && stores[c]->ctx == ctx, "store does not belong to this context");
    MOPT_REQUIRE(problems[c].num_parameters == P, "all cost terms must share the parameter vector");
    MOPT_REQUIRE(problems[c].manifold == problems[0].manifold, "all cost terms must use the same manifold");
    MOPT_TRY(validate_problem(stores[c], &problems[c], true));  // also: a model without parameters
  }
  MOPT_TRY(check_exchange_alive(ctx));
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  XArg xa;
  std::memset(&xa, 0, sizeof(xa));
  for (int i = 0; i < P; ++i) xa.v[i] = x[i];
  for (int c = 0; c < n_costs; ++c) {
    const mopt_problem* p = &problems[c];
    // the ParamBlock of slot c (sets, steps, point2point affine Jacobian pieces): read by the score Gram kernel
    // even where the linearization pass derives them itself (fused set-up)
    MOPT_TRY(setup_slot(ctx, c, p, x));
    // H, b, sum r^T r: the pass mopt_linearize (one cost) / mopt_lm_minimize (several) runs, rank-local
    if (can_fuse_setup(ctx, p, stores[c])) MOPT_TRY(launch_pass(ctx, stores[c], p, c, c > 0 ? 1 : 0, PASS_LINEARIZE, false, &xa));
    else MOPT_TRY(launch_pass(ctx, stores[c], p, c, c > 0 ? 1 : 0, PASS_LINEARIZE, false));
    MOPT_TRY(launch_cov_pass(ctx, stores[c], p, c, ctx->d_cov_sums + size_t(c) * kMaxRaw));
  }
  MOPT_CUDA_TRY(cudaMemcpyAsync(ctx->h_result, ctx->d_trial, sizeof(double) * packed_size(P), cudaMemcpyDeviceToHost,
                                ctx->stream));
  MOPT_CUDA_TRY(cudaMemcpyAsync(ctx->h_cov_sums, ctx->d_cov_sums, sizeof(double) * size_t(n_costs) * kMaxRaw,
                                cudaMemcpyDeviceToHost, ctx->stream));
  MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  mopt_cov_terms t;
  std::memset(&t, 0, sizeof(t));
  t.num_parameters = P;
  unpack_result(*ctx->h_result, P, t.H, t.b, &t.sum_sq);
  const int nh = P * (P + 1) / 2;
  double Gp[kMaxP * (kMaxP + 1) / 2] = {0.0};
  for (int c = 0; c < n_costs; ++c) {  // cost terms in order, as the passes accumulate H
    const double* v = ctx->h_cov_sums + size_t(c) * kMaxRaw;
    for (int k = 0; k < nh; ++k) Gp[k] += v[k];
    t.wsse += v[nh];
    const int64_t nv = int64_t(v[nh + 1]);
    t.n_valid += nv;
    t.m += nv * problems[c].num_outputs;
  }
  for (int i = 0; i < P; ++i)
    for (int j = i; j < P; ++j) t.G[i + j * P] = t.G[j + i * P] = Gp[tri_index(P, i, j)];
  *out = t;
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_linearize_async(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const double* x) try {
  MOPT_REQUIRE(ctx && store && store->ctx == ctx, "store does not belong to this context");
  MOPT_TRY(validate_problem(store, problem, true));
  return enqueue_pass(ctx, store, problem, x, PASS_LINEARIZE);
}
MOPT_ABI_CATCH

int mopt_ctx_result(mopt_ctx* ctx, int num_parameters, double* H, double* b, double* sum) try {
  MOPT_REQUIRE(ctx, "null ctx");
  MOPT_REQUIRE(num_parameters >= 0 && num_parameters <= kMaxP, "bad num_parameters");
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  return fetch_result(ctx, num_parameters, H, b, sum);
}
MOPT_ABI_CATCH

int mopt_upload_and_linearize(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const void* host_a,
                              const void* host_b, int host_dtype, int64_t count, const double* x, double* H, double* b,
                              double* sum) try {
  MOPT_REQUIRE(ctx && store && store->ctx == ctx, "store does not belong to this context");
  MOPT_TRY(validate_problem(store, problem, true));
  MOPT_REQUIRE(count == store->n, "count must equal the store size");
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  MOPT_TRY(store_upload_async(store, 0, host_a, host_dtype, 0, 0, count));
  MOPT_TRY(store_upload_async(store, 1, host_b, host_dtype, 0, 0, count));
  MOPT_TRY(enqueue_pass(ctx, store, problem, x, PASS_LINEARIZE));
  return fetch_result(ctx, problem->num_parameters, H, b, sum);
}
MOPT_ABI_CATCH

void mopt_lm_default_options(mopt_lm_options* o) {
  if (!o) return;
  o->max_iterations = 15;       // optimizer.h:19
  o->lm_max_iterations = 3;     // levenberg_marquadt_dyn.cpp:9
  o->lambda_factor = 1e-9;      // levenberg_marquadt_dyn.cpp:16
  o->scalar_dtype = MOPT_F64;
  o->speculative = 1;
  o->flags = MOPT_LM_STAGNATION_STOP;
}

int mopt_lm_minimize(mopt_ctx* ctx, int n_costs, mopt_store* const* stores, const mopt_problem* problems,
                     const mopt_lm_options* options, double* x, mopt_lm_report* report) try {
  MOPT_REQUIRE(ctx && stores && problems && x && report, "null argument");
  if (n_costs <= 0) {
    // Optimizer::checkCosts, optimizer.h:48-54
    set_last_error("No cost function added!");
    return MOPT_ERR_INVALID_ARGUMENT;
  }
  MOPT_REQUIRE(n_costs <= MOPT_MAX_COSTS, "too many cost terms");
  mopt_lm_options opt;
  if (options) opt = *options; else mopt_lm_default_options(&opt);
  MOPT_REQUIRE(opt.max_iterations >= 0, "Optimization::max_iterations cannot be less than 0.");  // optimizer.h:34-35
  MOPT_REQUIRE(opt.lm_max_iterations >= 0, "lm_max_iterations cannot be negative");
  const int P = problems[0].num_parameters;
  MOPT_REQUIRE(P > 0 && P <= kMaxP, "bad num_parameters");
  for (int c = 0; c < n_costs; ++c) {
    MOPT_REQUIRE(stores[c] && stores[c]->ctx == ctx, "store does not belong to this context");
    MOPT_TRY(validate_problem(stores[c], &problems[c], true));
    MOPT_REQUIRE(problems[c].num_parameters == P, "all cost terms must share the parameter vector");
    MOPT_REQUIRE(problems[c].manifold == problems[0].manifold, "all cost terms must use the same manifold");
  }
  MOPT_TRY(check_exchange_alive(ctx));
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  std::memset(report, 0, offsetof(mopt_lm_report, trials));  // the trace entries are valid up to num_trials
  if (opt.max_iterations == 0) {
    report->status = MOPT_MAXIMUM_ITERATIONS_REACHED;
    return MOPT_OK;
  }
  for (int c = 0; c < n_costs; ++c) MOPT_TRY(stage_cost(ctx, c, &problems[c]));

  LmInit in;
  std::memset(&in, 0, sizeof(in));
  in.P = P; in.n_costs = n_costs; in.max_it = opt.max_iterations; in.lm_max_it = opt.lm_max_iterations;
  in.speculative = opt.speculative ? 1 : 0; in.scalar_f32 = (opt.scalar_dtype == MOPT_F32) ? 1 : 0;
  // model->update(x) (levenberg_marquadt_dyn.cpp:54) changes the residual set at every outer iteration, so the
  // H, b evaluated speculatively at a trial point are not those of the next linearization: reference pass order.
  bool has_update = false;
  for (int c = 0; c < n_costs; ++c) has_update = has_update || (stores[c]->index != nullptr);
  if (has_update) in.speculative = 0;
  in.lambda_factor = opt.lambda_factor;
  in.flags = opt.flags;
  for (int i = 0; i < P; ++i) in.x0[i] = x[i];
  bool init_launched = false;
  auto launch_init = [&]() -> int {
    if (init_launched) return MOPT_OK;
    lm_init_kernel<<<1, 32, 0, ctx->stream>>>(ctx->d_lm, ctx->d_slots, in);
    MOPT_CUDA_TRY(cudaGetLastError());
    init_launched = true;
    return MOPT_OK;
  };
  // user models with their own setup(x): the run-time compiled setup kernel re-derives their parameter sets from
  // the state's evaluation point after every optimizer transition (idempotent when x_eval did not move)
  bool any_user_setup = false;
  for (int c = 0; c < n_costs; ++c) any_user_setup = any_user_setup || user_model_has_setup(problems[c].model);
  auto user_setups = [&]() -> int {
    if (!any_user_setup) return MOPT_OK;
    for (int c = 0; c < n_costs; ++c)
      if (user_model_has_setup(problems[c].model))
        MOPT_TRY(launch_user_setup(ctx->stream, ctx->device, problems[c].model, &ctx->d_slots[c], ctx->d_lm->x_eval,
                                   nullptr, P));
    return MOPT_OK;
  };
  if (any_user_setup) {
    MOPT_TRY(launch_init());
    MOPT_TRY(user_setups());
  }

  // Small single-cost point2point problems on one GPU: the whole loop in ONE cooperative launch (mopt_lm_mono.cuh);
  // up to 2^22 residuals.  MOPT_LM_MONO=0 in the environment keeps the launch-per-trial path (A/B).
  {
    static const int64_t mono_max = [] {
      const char* e = getenv("MOPT_LM_MONO");
      return (e && e[0] == '0') ? int64_t(0) : int64_t(1) << 22;
    }();
    const mopt_problem& p0 = problems[0];
    const bool moment_path = p0.model == MOPT_MODEL_POINT2POINT &&
                             (p0.jacobian == MOPT_JAC_ANALYTICAL || !(p0.flags & MOPT_FLAG_GENERIC_KERNEL));
    if (n_costs == 1 && ctx->world == 1 && !has_update && !any_user_setup && moment_path && stores[0]->n <= mono_max) {
      PassArgs a = make_args(ctx, stores[0], 0, 0, -1);
      PassLaunch L{ctx->stream, ctx->num_sms, ctx->ctas_per_sm, ctx->threads};
      MonoArgs m;
      m.st = ctx->d_lm;
      m.host_st = ctx->d_lm_host;
      m.host_flag = ctx->d_flags;  // word 0 of the mapped flag ring (idle: this path and the launch-per-trial path exclude each other)
      reinterpret_cast<volatile int*>(ctx->h_flags)[0] = 0;
      ctx->h_lm->done = 0;
      m.slots = ctx->d_slots;
      m.rt_words = ctx->d_gen;
      const int64_t slots64 = int64_t(opt.max_iterations) * (int64_t(opt.lm_max_iterations) + 1) + 2;
      m.max_slots = int(slots64 < INT32_MAX ? slots64 : INT32_MAX);
      m.init = in;  // prepare() + the first setup(x0) run inside the kernel too (CTA 0, before the first pass)
      m.gen_base = ctx->mono_gen;
      ctx->mono_gen += (unsigned long long)(m.max_slots) + 2ull;
      const bool qrot = p0.jacobian == MOPT_JAC_ANALYTICAL && (p0.variant == MOPT_P2P_EXACT || p0.variant == MOPT_P2P_LEFT);
      MOPT_TRY(launch_p2p_lm_mono(L, stores[0]->dtype, p0.compute_dtype, p0.loss, qrot, a, m));
      // The kernel's last act is to set the mapped flag (after a system-scope fence behind the state and the trace):
      // spinning on it sees the end ~5 us before cudaStreamSynchronize would return (kernel teardown + driver
      // wake-up).  The stream is queried now and then so that a failed launch cannot hang the caller.
      for (int spins = 0;; ++spins) {
        if (reinterpret_cast<volatile int*>(ctx->h_flags)[0] != 0) break;
        if ((spins & 4095) == 4095) {
          const cudaError_t q = cudaStreamQuery(ctx->stream);
          if (q == cudaSuccess) break;  // finished (the flag is set by now, or the state says why not)
          if (q != cudaErrorNotReady) MOPT_CUDA_TRY(q);
        }
      }
      std::atomic_thread_fence(std::memory_order_acquire);
      return finish_lm(ctx, P, x, report, /*on_host=*/true);
    }
  }

  MOPT_TRY(launch_init());
  // Passes are enqueued in batches, always one batch ahead of the one whose done flag is being
  // awaited, so the device never idles on the host; every rank reads the flag of the same slot,
  // so all ranks stop after the same number of (collective-bearing) slots.
  // The per-slot done flags live in a ring of flags_capacity mapped words: at most two batches are ever in flight
  // and a slot's word is free again once its batch event has completed, so any slot budget fits.
  const int64_t max_slots = int64_t(opt.max_iterations) * (int64_t(opt.lm_max_iterations) + 1) + 2;
  const int kBatch = 2;
  int64_t enq = 0;
  auto slot_index = [&](int64_t slot) { return int(slot % ctx->flags_capacity); };
  auto enqueue_batch = [&](int par, int64_t* last_slot) -> int {
    *last_slot = -1;
    for (int s = 0; s < kBatch && enq < max_slots; ++s, ++enq) {
      ctx->h_flags[slot_index(enq)] = 0;
      // cost->update(x0): re-associate correspondences; the kernel gates itself on "start of an outer iteration"
      for (int c = 0; c < n_costs; ++c) MOPT_TRY(enqueue_reassociate(stores[c], &ctx->d_slots[c].pb, ctx->d_lm));
      for (int c = 0; c < n_costs; ++c)
        MOPT_TRY(launch_pass(ctx, stores[c], &problems[c], c, c > 0 ? 1 : 0, -1, c == n_costs - 1));
      MOPT_TRY(allreduce_trial(ctx, P, -1));
      lm_step_kernel<<<1, 32, 0, ctx->stream>>>(ctx->d_lm, ctx->d_trial, ctx->d_slots, ctx->d_flags + slot_index(enq),
                                                ctx->d_xerr_dev, in.P, in.scalar_f32);
      MOPT_CUDA_TRY(cudaGetLastError());
      MOPT_TRY(user_setups());
      *last_slot = enq;
    }
    if (*last_slot >= 0) MOPT_CUDA_TRY(cudaEventRecord(ctx->ev_batch[par], ctx->stream));
    return MOPT_OK;
  };
  int par = 0;
  int64_t cur_last = -1, next_last = -1;
  MOPT_TRY(enqueue_batch(par, &cur_last));
  while (cur_last >= 0) {
    MOPT_TRY(enqueue_batch(par ^ 1, &next_last));  // keep one batch in flight behind the awaited one
    MOPT_CUDA_TRY(cudaEventSynchronize(ctx->ev_batch[par]));
    if (reinterpret_cast<volatile int*>(ctx->h_flags)[slot_index(cur_last)] != 0) break;
    if (ctx->h_xerr && *reinterpret_cast<volatile int*>(ctx->h_xerr)) break;  // a peer died: stop enqueuing
    par ^= 1;
    cur_last = next_last;
  }
  MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));

  return finish_lm(ctx, P, x, report);
}
MOPT_ABI_CATCH

int mopt_so3_convert6dof(const double* x, double* T) try {
  MOPT_REQUIRE(x && T, "null argument");
  // src/so3.cpp:7-19,43-57 (host-side helper kept for API parity; the device copy is so3_exp_dev)
  const double w[3] = {x[3], x[4], x[5]};
  const double n = std::sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
  double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  if (n > 10.0 * 2.220446049250313e-16) {
    const double a[3] = {w[0] / n, w[1] / n, w[2] / n};
    const double K[9] = {0, -a[2], a[1], a[2], 0, -a[0], -a[1], a[0], 0};
    const double s = std::sin(n), c = std::cos(n);
    for (int r = 0; r < 3; ++r)
      for (int col = 0; col < 3; ++col) {
        double kk = 0;
        for (int k = 0; k < 3; ++k) kk += K[r * 3 + k] * K[k * 3 + col];
        R[r * 3 + col] += s * K[r * 3 + col] + (1.0 - c) * kk;
      }
  }
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) T[r * 4 + c] = R[r * 3 + c];
    T[r * 4 + 3] = x[r];
  }
  T[12] = T[13] = T[14] = 0.0;
  T[15] = 1.0;
  return MOPT_OK;
}
MOPT_ABI_CATCH

// Runs the DEVICE LDL^T (the one the LM step kernel uses) on one thread; for tests.
int mopt_ldlt_solve(int n, const double* A, const double* rhs, double* out) try {
  MOPT_REQUIRE(n >= 1 && n <= kMaxP && A && rhs && out, "bad argument");
  double *dA = nullptr, *dr = nullptr, *dout = nullptr;
  MOPT_CUDA_TRY(cudaMalloc(&dA, sizeof(double) * n * n));
  MOPT_CUDA_TRY(cudaMalloc(&dr, sizeof(double) * n));
  MOPT_CUDA_TRY(cudaMalloc(&dout, sizeof(double) * n));
  MOPT_CUDA_TRY(cudaMemcpy(dA, A, sizeof(double) * n * n, cudaMemcpyHostToDevice));
  MOPT_CUDA_TRY(cudaMemcpy(dr, rhs, sizeof(double) * n, cudaMemcpyHostToDevice));
  // the warp-cooperative factorization the LM step kernel uses, then the serial restatement on a scratch copy:
  // the two must agree to the last bit (same summation order per row)
  double out_warp[kMaxP], *dA2 = nullptr;
  ldlt_warp_test_kernel<<<1, 32>>>(n, dA, dr, dout);
  MOPT_CUDA_TRY(cudaGetLastError());
  MOPT_CUDA_TRY(cudaMemcpy(out_warp, dout, sizeof(double) * n, cudaMemcpyDeviceToHost));
  MOPT_CUDA_TRY(cudaMalloc(&dA2, sizeof(double) * n * n));
  MOPT_CUDA_TRY(cudaMemcpy(dA2, A, sizeof(double) * n * n, cudaMemcpyHostToDevice));
  ldlt_test_kernel<<<1, 1>>>(n, dA2, dr, dout);
  MOPT_CUDA_TRY(cudaGetLastError());
  MOPT_CUDA_TRY(cudaMemcpy(out, dout, sizeof(double) * n, cudaMemcpyDeviceToHost));
  cudaFree(dA); cudaFree(dA2); cudaFree(dr); cudaFree(dout);
  if (std::memcmp(out, out_warp, sizeof(double) * n) != 0) {
    set_last_error("internal error: warp-cooperative and serial LDL^T disagree");
    return MOPT_ERR_CUDA;
  }
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_host_alloc(void** ptr, uint64_t bytes) try {
  MOPT_REQUIRE(ptr, "null ptr");
  MOPT_CUDA_TRY(cudaHostAlloc(ptr, bytes, cudaHostAllocDefault));
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_host_free(void* ptr) try {
  if (ptr) MOPT_CUDA_TRY(cudaFreeHost(ptr));
  return MOPT_OK;
}
MOPT_ABI_CATCH

}  // extern "C"
