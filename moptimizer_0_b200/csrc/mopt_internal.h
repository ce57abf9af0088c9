// Host-side internals shared by the translation units of libmopt_b200.so.
#pragma once

#include <cuda_runtime.h>

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
// mopt_icp.cu: enqueue model->update(x) for a store with a target index (no-op without one)
int enqueue_reassociate(mopt_store* st, const ParamBlock* pb, const LmState* gate);

// mopt_pass_wide.cu
int launch_wide(const PassLaunch& L, int model, int store_dtype, int compute_dtype, const PassArgs& a);

// mopt_eval.cu: per-residual evaluation of a builtin model (mopt_evaluate)
int launch_evaluate(const PassLaunch& L, int model, int store_dtype, int compute_dtype, int out_dtype,
                    const PassArgs& a, const EvalArgs& ev);

// mopt_cov.cu: score Gram sums of a builtin model (mopt_covariance_terms); `form` is a CovJac
int launch_cov(const PassLaunch& L, int model, int form, int store_dtype, int compute_dtype, const PassArgs& a,
               const CovArgs& cv);

// mopt_quant.cu: one radix-select sweep of a builtin model, and the step between sweeps (mopt_residual_quantiles)
int launch_quantile_sweep(const PassLaunch& L, int model, int store_dtype, int compute_dtype, const PassArgs& a,
                          const QuantArgs& qa);
int launch_quantile_step(cudaStream_t stream, QuantState* st, int sweep, int n_q, const QuantLevels& lv);

// mopt_hyp.cu: set 0 of n hypotheses (xs [n][kMaxP] -> sets [n][kSetSize]) and their scores (mopt_score_hypotheses)
int launch_hypothesis_setup(cudaStream_t stream, const CostDev* c, const double* xs, int n, double* sets);
int launch_hypothesis_score(const PassLaunch& L, int model, int store_dtype, int compute_dtype, const PassArgs& a,
                            const HypArgs& h);

// mopt_rtc.cu: run-time compiled user models (ids >= MOPT_MODEL_USER_BASE)
int launch_user(const PassLaunch& L, int device, int model, bool numeric, int store_dtype, int compute_dtype,
                const PassArgs& a);
int launch_user_evaluate(const PassLaunch& L, int device, int model, int store_dtype, int compute_dtype, int out_dtype,
                         const PassArgs& a, const EvalArgs& ev);
int launch_user_cov(const PassLaunch& L, int device, int model, bool numeric, int store_dtype, int compute_dtype,
                    const PassArgs& a, const CovArgs& cv);
int launch_user_quantile_sweep(const PassLaunch& L, int device, int model, int store_dtype, int compute_dtype,
                               const PassArgs& a, const QuantArgs& qa);
int launch_user_hypothesis_score(const PassLaunch& L, int device, int model, int store_dtype, int compute_dtype,
                                 const PassArgs& a, const HypArgs& h);
int launch_user_hypothesis_setup(cudaStream_t stream, int device, int model, const CostDev* c, const double* xs, int n,
                                 double* sets);
int launch_user_setup(cudaStream_t stream, int device, int model, CostSlot* slot, const double* x_dev,
                      const double* x_host, int P);
int user_model_rot_offset(int model);
bool user_model_has_setup(int model);

// Persistent grid of a streaming kernel: resident CTAs per SM (at most L.ctas_per_sm when that is set) times the SMs,
// capped at kMaxGrid and at one CTA per `threads` work items, never below 1.  The summation order of a pass follows
// the grid, so every launcher of a pass kernel sizes it here.
inline int pick_grid(const void* kernel, int threads, const PassLaunch& L, int64_t work_items, size_t dyn_smem = 0) {
  int occ = 1;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, dyn_smem) != cudaSuccess || occ < 1) occ = 1;
  int per_sm = (L.ctas_per_sm > 0) ? (L.ctas_per_sm < occ ? L.ctas_per_sm : occ) : occ;
  int64_t g = int64_t(per_sm) * L.num_sms;
  if (g > kMaxGrid) g = kMaxGrid;
  const int64_t need = (work_items + threads - 1) / threads;
  if (need < g) g = need;
  if (g < 1) g = 1;
  return int(g);
}

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
