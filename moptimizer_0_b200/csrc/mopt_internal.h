// Host-side internals shared by the translation units of libmopt_b200.so.
#pragma once

#include <cuda_runtime.h>

#include "mopt_align.cuh"
#include "mopt_common.cuh"
#include "mopt_cov.cuh"
#include "mopt_eval.cuh"
#include "mopt_hyp.cuh"
#include "mopt_lm.cuh"
#include "mopt_lm_mono.cuh"
#include "mopt_models.cuh"
#include "mopt_pass.cuh"
#include "mopt_quant.cuh"

struct mopt_ctx {
  int device = 0;
  int num_sms = 148;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;
  // pass plumbing
  double* d_partials = nullptr;      // [kPackedMaxRaw][kMaxGrid]
  unsigned int* d_ticket = nullptr;
  mopt::PassResult* d_trial = nullptr;
  mopt::CostSlot* d_slots = nullptr; // [MOPT_MAX_COSTS]
  mopt::LmState* d_lm = nullptr;
  // pinned host mirrors
  mopt::PassResult* h_result = nullptr;
  mopt::LmState* h_lm = nullptr;
  mopt::LmState* d_lm_host = nullptr;  // device address of h_lm (mapped): the persistent LM kernel reports through it
  mopt::CostSlot* h_slot = nullptr;  // staging for cost constants
  int* h_flags = nullptr;            // per-slot done flags written by lm_step_kernel (mapped)
  int* d_flags = nullptr;            // device alias of h_flags
  int flags_capacity = 0;
  mopt::CostDev cached_cost[MOPT_MAX_COSTS];
  bool cached_valid[MOPT_MAX_COSTS] = {false};
  // upload staging (device, double buffered) + events
  void* d_stage[2] = {nullptr, nullptr};
  size_t stage_bytes = 0;
  cudaEvent_t ev_copy[2] = {nullptr, nullptr};
  cudaEvent_t ev_free[2] = {nullptr, nullptr};
  cudaEvent_t ev_batch[2] = {nullptr, nullptr};
  // launch tuning
  int ctas_per_sm = 0;
  int threads = 0;
  // sharding
  void* nccl_comm = nullptr;
  int rank = 0, world = 1;
  // NVLink peer exchange (mopt_ctx_open_peers): replaces the NCCL all-reduce of the packed result
  mopt::XSlot* d_xbuf = nullptr;                 // this rank's slots[2][kMaxWorld]
  mopt::XSlot* peer_base[mopt::kMaxWorld] = {nullptr};
  bool peers_open = false;
  bool exchange_enabled = true;                  // diagnostics: false = rank-local results, no collective
  bool fused_consumer = true;                    // the pushing warp also consumes (MOPT_PEER_CONSUMER=kernel: separate kernel)
  unsigned long long xseq = 0;
  int* h_xerr = nullptr;                         // mapped: set by the consumer kernel on a wait timeout
  int* d_xerr = nullptr;
  unsigned long long* d_gen = nullptr;           // persistent LM kernel: the 24 tagged words that carry (R, t) and act as its grid barrier (publish_rt)
  unsigned long long mono_gen = 0;               // barrier targets handed out so far (monotonic over the context's life)
  int* d_xerr_dev = nullptr;                     // device-resident copy, read by the kernels that follow a failed exchange
  double* d_eval_stats = nullptr;                // mopt_evaluate: the statistics written by the evaluation kernel's last CTA
  double* d_align = nullptr;                     // mopt_align_terms: the terms (an AlignAcc) written by its last CTA
  double* d_cov_sums = nullptr;                  // mopt_covariance_terms: [MOPT_MAX_COSTS][kMaxRaw] score Gram totals
  double* h_cov_sums = nullptr;                  // pinned host copy of the same
  mopt::QuantState* d_quant = nullptr;           // mopt_residual_quantiles: histogram, prefixes and selected keys
  // mopt_score_hypotheses, allocated on first use: the hypotheses ([MOPT_MAX_HYPOTHESES][kMaxP], uploaded through the
  // pinned h_hyp, which also takes the results back), their sets, the per-CTA partials of every tile, the tickets
  // and the per-hypothesis statistics
  double* h_hyp = nullptr;
  double* d_hyp_x = nullptr;
  double* d_hyp_sets = nullptr;
  double* d_hyp_partials = nullptr;
  unsigned int* d_hyp_tickets = nullptr;
  double* d_hyp_out = nullptr;
};

struct mopt_store {
  mopt_ctx* ctx = nullptr;
  int model = 0;
  int dtype = 0;
  int64_t n = 0;
  int nstreams = 0;
  void* streams[mopt::kMaxStreams] = {nullptr};
  struct mopt_nn_index* index = nullptr;  // target cloud for model->update(x) (mopt_icp.cu), not owned
  bool may_have_invalid = false;          // target streams may hold the NaN "no correspondence" marker
};

namespace mopt {

struct PassLaunch {
  cudaStream_t stream;
  int num_sms;
  int ctas_per_sm;  // 0 = occupancy-derived default
  int threads;      // 0 = default launch shape
  bool affine_fd = true;  // finite differences over a common denominator where the model allows it
                          // (dense_pass_kernel AFFINE_FD); false with MOPT_FLAG_GENERIC_KERNEL
  bool identity_cov = false;  // the problem has no setCovariance matrix (C = I): the tensor-core Gram kernel applies
};

// A streaming kernel ready to launch: a builtin instantiation, or the run-time compiled kernel of a user model.
struct KernelDesc {
  const void* fn = nullptr;
  int threads = 0;
  size_t smem = 0;    // dynamic shared memory
  int occupancy = 1;  // resident CTAs per SM
};

// The kinds of run-time compiled kernels of a user model (mopt_rtc.cu); the last four are the analysis kernels.
enum KernelKind : int { KIND_PASS = 0, KIND_SETUP = 1, KIND_EVAL = 2, KIND_COV = 3, KIND_QUANT = 4, KIND_HYP = 5 };

// Elements of a store of this dtype per 16-byte load (VecOf): the work-item granularity of the streaming kernels.
inline int store_vec(int store_dtype) { return store_dtype == MOPT_F32 ? VecOf<float>::N : VecOf<double>::N; }

// A model with more than 32 packed sums (H upper, b, sum) takes the wide pass kernel: the dense pass reduces them in
// one transposing-reduce chunk.
constexpr bool is_wide(int P) { return P * (P + 1) / 2 + P + 1 > 32; }

// Does model M declare an affine first stage (NAFF / affine / finish / finish_diff)?
template <class M, class = void>
struct HasAffineStage { static constexpr bool value = false; };
template <class M>
struct HasAffineStage<M, decltype(void(M::NAFF))> { static constexpr bool value = true; };

// f(M{}) with the struct of builtin model `model`: the one place a model id becomes a kernel instantiation.
template <class F>
int with_builtin_model(int model, F&& f) {
  switch (model) {
    case MOPT_MODEL_POINT2POINT: return f(P2PModel{});
    case MOPT_MODEL_EXP_CURVE: return f(ExpCurveModel{});
    case MOPT_MODEL_MICHAELIS_MENTEN: return f(MichaelisMentenModel{});
    case MOPT_MODEL_PINHOLE: return f(PinholeModel{});
    case MOPT_MODEL_POWELL: return f(PowellModel{});
    case MOPT_MODEL_POINT_DIST: return f(PointDistModel{});
    case MOPT_MODEL_PINHOLE_DISTORT: return f(PinholeDistortModel{});
    default:
      set_last_error("unknown model kind");
      return MOPT_ERR_INVALID_ARGUMENT;
  }
}

// f(ST{}, CT{}) for the (store, compute) dtype pair.  validate_problem (mopt_capi.cu) rejects f64 store + f32 compute.
template <class F>
int with_dtypes(int store_dtype, int compute_dtype, F&& f) {
  if (store_dtype == MOPT_F32 && compute_dtype == MOPT_F32) return f(float{}, float{});
  if (store_dtype == MOPT_F32 && compute_dtype == MOPT_F64) return f(float{}, double{});
  if (store_dtype == MOPT_F64 && compute_dtype == MOPT_F64) return f(double{}, double{});
  set_last_error("internal error: no kernel for this (store, compute) dtype pair");
  return MOPT_ERR_CUDA;
}

// Resident CTAs per SM of a kernel at this launch shape (1 if the query fails).
inline int occupancy_of(const void* kernel, int threads, size_t dyn_smem = 0) {
  int occ = 1;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, dyn_smem) != cudaSuccess || occ < 1) occ = 1;
  return occ;
}

inline KernelDesc builtin_kernel(const void* kernel, int threads) {
  return {kernel, threads, 0, occupancy_of(kernel, threads)};
}

// Persistent grid of a streaming kernel with `occupancy` resident CTAs per SM: that many CTAs per SM (at most
// L.ctas_per_sm when that is set) times the SMs, capped at kMaxGrid and at one CTA per `threads` work items, never
// below 1.  The summation order of a pass follows the grid, so every launcher of a streaming kernel, builtin or run-time
// compiled, sizes it here.
inline int persistent_grid(int occupancy, int threads, const PassLaunch& L, int64_t work_items) {
  int per_sm = (L.ctas_per_sm > 0) ? (L.ctas_per_sm < occupancy ? L.ctas_per_sm : occupancy) : occupancy;
  int64_t g = int64_t(per_sm) * L.num_sms;
  if (g > kMaxGrid) g = kMaxGrid;
  const int64_t need = (work_items + threads - 1) / threads;
  if (need < g) g = need;
  if (g < 1) g = 1;
  return int(g);
}

inline int pick_grid(const void* kernel, int threads, const PassLaunch& L, int64_t work_items, size_t dyn_smem = 0) {
  return persistent_grid(occupancy_of(kernel, threads, dyn_smem), threads, L, work_items);
}

// mopt_pass_p2p.cu
int launch_p2p_moment(const PassLaunch& L, int store_dtype, int compute_dtype, int loss, bool qrot, const PassArgs& a);
// mopt_pass_p2p2.cu: second generation, fp32 store + fp32 compute
int launch_p2p_moment_gen2(const PassLaunch& L, int loss, bool qrot, const PassArgs& a);
// mopt_lm_mono.cu: the whole LM loop of a small single-cost point2point problem in one cooperative launch
int launch_p2p_lm_mono(const PassLaunch& L, int store_dtype, int compute_dtype, int loss, bool qrot, const PassArgs& a,
                       const MonoArgs& m);
// mopt_pass_dense.cu
int launch_dense(const PassLaunch& L, int model, bool numeric, int store_dtype, int compute_dtype, const PassArgs& a);

// mopt_capi.cu: copy the cost constants of `problem` into slot `slot` and run model setup at x on the device
int setup_slot(mopt_ctx* ctx, int slot, const mopt_problem* problem, const double* x);
// mopt_capi.cu: does `st` accept `p` (and, with need_linearize, can it be linearized)?  Sets the last error if not.
int validate_problem(const mopt_store* st, const mopt_problem* p, bool need_linearize);
// mopt_capi.cu: the kernel arguments of a pass over `st` with the constants of cost slot `slot`
PassArgs make_args(mopt_ctx* ctx, const mopt_store* st, int slot, int accumulate, int mode_override);
// mopt_capi.cu: the launch settings of the context for problem `p`
PassLaunch pass_launch(const mopt_ctx* ctx, const mopt_problem* p);
// mopt_icp.cu: enqueue model->update(x) for a store with a target index (no-op without one)
int enqueue_reassociate(mopt_store* st, const ParamBlock* pb, const LmState* gate);

// mopt_pass_wide.cu
int launch_wide(const PassLaunch& L, int model, int store_dtype, int compute_dtype, const PassArgs& a);

// The analysis kernels of the builtin models; mopt_capi.cu launches them, and the run-time compiled ones (user_kernel).
// mopt_eval.cu: per-residual evaluation (mopt_evaluate), with fp32 or fp64 outputs
int evaluate_kernel_desc(int model, int store_dtype, int compute_dtype, bool f64_out, KernelDesc* k);
// mopt_cov.cu: score Gram sums (mopt_covariance_terms); `form` is a CovJac, `affine_fd` as PassLaunch::affine_fd
int score_gram_kernel_desc(int model, int form, bool affine_fd, int store_dtype, int compute_dtype, KernelDesc* k);
// mopt_quant.cu: one radix-select sweep, and the step between sweeps (mopt_residual_quantiles)
int quantile_sweep_kernel_desc(int model, int store_dtype, int compute_dtype, KernelDesc* k);
int launch_quantile_step(cudaStream_t stream, QuantState* st, int sweep, int n_q, const QuantLevels& lv);
// mopt_hyp.cu: set 0 of n hypotheses (xs [n][kMaxP] -> sets [n][kSetSize]) and their scores (mopt_score_hypotheses)
int launch_hypothesis_setup(cudaStream_t stream, const CostDev* c, const double* xs, int n, double* sets);
int hypothesis_score_kernel_desc(int model, int store_dtype, int compute_dtype, KernelDesc* k);
// mopt_align.cu: the moments of a point2point store (mopt_align_terms); no other model has them
int align_kernel_desc(int store_dtype, int compute_dtype, KernelDesc* k);

// mopt_cov.cu: cyclic Jacobi eigendecomposition of the symmetric n x n column-major A (overwritten): on return the
// diagonal of A holds the eigenvalues (unsorted) and the columns of V the eigenvectors
void jacobi_eigen(int n, double* A, double* V);

// mopt_rtc.cu: run-time compiled user models (ids >= MOPT_MODEL_USER_BASE)
int launch_user(const PassLaunch& L, int device, int model, bool numeric, int store_dtype, int compute_dtype,
                const PassArgs& a);
// The kernel of `kind` of a user model, compiled and configured for `device`.  `numeric`: for KIND_EVAL fp64 outputs,
// for KIND_COV and KIND_PASS finite differences.
int user_kernel(int device, int model, KernelKind kind, int store_dtype, int compute_dtype, bool numeric,
                KernelDesc* k);
int launch_user_hypothesis_setup(cudaStream_t stream, int device, int model, const CostDev* c, const double* xs, int n,
                                 double* sets);
int launch_user_setup(cudaStream_t stream, int device, int model, CostSlot* slot, const double* x_dev,
                      const double* x_host, int P);
int user_model_rot_offset(int model);
bool user_model_has_setup(int model);

// Opt kernel K in to `bytes` of dynamic shared memory.  Function attributes are per device, so this runs once on each.
template <auto K>
int allow_dyn_smem(size_t bytes) {
  static bool configured[64] = {false};
  int dev = 0;
  MOPT_CUDA_TRY(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    MOPT_CUDA_TRY(cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes)));
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  return MOPT_OK;
}

}  // namespace mopt
