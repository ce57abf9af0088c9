/*
 * mopt_capi.h — C ABI of the B200-native linearization / Levenberg-Marquardt hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, `extern "C"`, int status returns,
 * no exceptions and no C++/torch types cross it.  The reference (Marcus-Forte/moptimizer_0)
 * has no FFI of its own; its boundary for this path is the C++ operator API
 *     CostFunctionBase<Scalar>::{update, computeCost, linearize}      include/moptimizer/cost_function.h:37-50
 *     CostFunction{Analytical,Numerical}Dynamic                         src/cost_function_*_dyn.cpp:19-30
 *     CostComputation::{computeHessian, computeHessianNumerical,
 *                       computeCost, parallelComputeCost}               include/moptimizer/linearization.h:36-158
 *     LevenbergMarquadtDynamic<Scalar>::minimize                        src/levenberg_marquadt_dyn.cpp:34-119
 * and every entry point below names the reference function it replaces.  The C++ classes in
 * include/moptimizer/ (same names and signatures as the reference) call these functions;
 * INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * All `file:line` citations are relative to the reference repository root.
 *
 * Threading: one host thread per context.  All device work of a context is issued on the
 * context's own CUDA stream; calls that return results to host memory synchronise that stream.
 */
#ifndef MOPT_CAPI_H
#define MOPT_CAPI_H

#ifndef __CUDACC_RTC__ /* NVRTC (user-defined device models) has no host headers; the kernel prologue typedefs these */
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define MOPT_MAX_PARAMETERS 16 /* P: parameters per problem (n x n device solve)              */
#define MOPT_MAX_OUTPUTS 4     /* O: residual dimension                                       */
#define MOPT_MAX_COSTS 8       /* cost terms summed by one LM problem (optimizer.h:58 addCost) */
#define MOPT_MAX_TRACE 1024    /* LM trial records kept in a report                           */
#define MOPT_NCCL_ID_BYTES 128

#if defined(__GNUC__)
#define MOPT_API __attribute__((visibility("default")))
#else
#define MOPT_API
#endif

typedef struct mopt_ctx mopt_ctx;     /* one GPU (+ optional communicator rank)            */
typedef struct mopt_store mopt_store; /* device-buffer residual store: planar data streams */

typedef enum mopt_status {
  MOPT_OK = 0,
  MOPT_ERR_INVALID_ARGUMENT = 1,
  MOPT_ERR_CUDA = 2,
  MOPT_ERR_COMM = 3,
  MOPT_ERR_UNSUPPORTED = 4,
  MOPT_ERR_OUT_OF_MEMORY = 5
} mopt_status;

/* include/moptimizer/types.h:6-12 — same numeric values. */
typedef enum mopt_optimization_status {
  MOPT_CONVERGED = 0,
  MOPT_MAXIMUM_ITERATIONS_REACHED = 1,
  MOPT_SMALL_DELTA = 2,
  MOPT_NUMERIC_ERROR = 3,
  MOPT_FATAL_ERROR = 4
} mopt_optimization_status;

typedef enum mopt_dtype { MOPT_F32 = 0, MOPT_F64 = 1 } mopt_dtype;

/* Builtin device models.  IBaseModel's virtual f / f_df (include/moptimizer/model.h:33,42) cannot
 * be called from a kernel, so the workloads the reference defines in its tests are compiled in. */
typedef enum mopt_model {
  /* r = T(x) p - q, x = [t, omega]; P=6, O=3.  tst/point2point.cpp:24-84.  data A = src xyz, B = tgt xyz */
  MOPT_MODEL_POINT2POINT = 0,
  /* r = y - exp(x0 t + x1); P=2, O=1.  tst/curve_fitting.cpp:81-98.  A = t, B = y */
  MOPT_MODEL_EXP_CURVE = 1,
  /* r = y - x0 t / (x1 + t); P=2, O=1.  tst/test_models.h:8-19, tst/differentiation.cpp:16-41.  A = t, B = y */
  MOPT_MODEL_MICHAELIS_MENTEN = 2,
  /* r = pix - proj(K T(x) C P); P=6, O=2.  tst/camera_calibration.cpp:12-57.  A = XYZ, B = uv;
   * consts = K (3x4 row-major, 12) then C (4x4 row-major, 16) */
  MOPT_MODEL_PINHOLE = 3,
  /* Powell's singular function; P=4, O=4, no data.  tst/powell.cpp:22-59 */
  MOPT_MODEL_POWELL = 4,
  /* r = p - q, no parameters; P=0, O=3, cost only.  tst/parallel.cpp:12-32 */
  MOPT_MODEL_POINT_DIST = 5,
  /* Pinhole with OpenCV-style distortion and free intrinsics (NOT in the reference; BASELINE.json configs[4]):
   * x = [t(3), omega(3), fx, fy, cx, cy, k1, k2, p1, p2, k3]; P=15, O=2.  A = XYZ, B = uv;
   * consts = C (4x4 row-major, 16), the fixed frame conversion applied before the extrinsics */
  MOPT_MODEL_PINHOLE_DISTORT = 6,
  MOPT_MODEL_COUNT_
} mopt_model;
/* Ids >= MOPT_MODEL_USER_BASE name run-time compiled user models (mopt_user_model_compile below). */
#define MOPT_MODEL_USER_BASE 1000

/* Which Jacobian the linearization uses. */
typedef enum mopt_jacobian {
  MOPT_JAC_ANALYTICAL = 0, /* computeHessian,          linearization.h:126-158 (model f_df) */
  MOPT_JAC_FORWARD = 1,    /* computeHessianNumerical, linearization.h:65-124 (reference: forward difference) */
  MOPT_JAC_CENTRAL = 2     /* same steps h_j, (r(x+h)-r(x-h))/2h — north-star addition */
} mopt_jacobian;

/* Analytical Jacobian form of MOPT_MODEL_POINT2POINT (ignored by other models). */
typedef enum mopt_p2p_variant {
  MOPT_P2P_EXACT = 0,           /* [I | -[R p]x J_l(omega)] — exact for the additive update of levenberg_marquadt_dyn.cpp:83 */
  MOPT_P2P_REFTEST = 1,         /* [I | -[p]x], row-major as linearization.h:17-18 requires (tst/point2point.cpp:72-75) */
  MOPT_P2P_REFTEST_COLMAJOR = 2, /* same values written column-major, bit-faithful to tst/point2point.cpp:18,71 */
  MOPT_P2P_LEFT = 3 /* [I | -[R p]x]: derivative w.r.t. a left SO(3) perturbation, for manifold = MOPT_MANIFOLD_SO3_LEFT */
} mopt_p2p_variant;

/* Parameter update rule.  The reference adds delta to x (levenberg_marquadt_dyn.cpp:82-83, "TODO Manifold
 * operation"); MOPT_MANIFOLD_SO3_LEFT finishes that TODO as an opt-in (SURVEY.md §8f-3) for models whose
 * x[3..5] is a rotation vector: omega <- Log(Exp(delta_omega) Exp(omega)) with so3::Exp / so3::Log
 * (src/so3.cpp:43-57,96-105), every other component additive.  Jacobians are then taken with respect to the
 * tangent perturbation at 0 (finite-difference steps sqrt(eps) on the rotation block). */
typedef enum mopt_manifold { MOPT_MANIFOLD_ADDITIVE = 0, MOPT_MANIFOLD_SO3_LEFT = 1 } mopt_manifold;

/* loss_function/loss_function.h:20-23, loss_function/geman_mcclure.h:7-19; Huber is new. */
typedef enum mopt_loss {
  MOPT_LOSS_NONE = 0,
  MOPT_LOSS_GEMAN_MCCLURE = 1, /* w = th^2 / (e2 + th)^2,            loss_param = th */
  MOPT_LOSS_HUBER = 2          /* w = 1 if e2 <= k^2 else k/sqrt(e2), loss_param = k  */
} mopt_loss;

/* One cost term: what CostFunction{Analytical,Numerical}Dynamic holds besides the data
 * (cost_function.h:52-58, cost_function_*_dyn.h:28-31). */
typedef struct mopt_problem {
  int32_t model;          /* mopt_model */
  int32_t variant;        /* mopt_p2p_variant */
  int32_t num_parameters; /* P */
  int32_t num_outputs;    /* O */
  int32_t jacobian;       /* mopt_jacobian */
  int32_t compute_dtype;  /* mopt_dtype: arithmetic of residual/Jacobian evaluation (the reference's Scalar);
                             accumulation across residuals is always fp64 */
  int32_t loss;           /* mopt_loss */
  int32_t has_covariance; /* 0: identity (src/cost_function_*_dyn.cpp:14-15) */
  double loss_param;
  double covariance[MOPT_MAX_OUTPUTS * MOPT_MAX_OUTPUTS]; /* O x O column-major, symmetric (setCovariance, cost_function.h:38-40) */
  double consts[32];                                       /* model constants, see mopt_model */
  int32_t manifold; /* mopt_manifold: how x + delta is formed and what the Jacobian differentiates */
  int32_t flags;    /* mopt_problem_flags, 0 by default */
} mopt_problem;
/* MOPT_FLAG_GENERIC_KERNEL: evaluate with the generic per-residual kernel even where a specialised one applies.
 * Point2point finite differences normally run on the moment kernel: r is affine in the source point, so
 * (r(x + h e_j) - r(x)) / h = ((R_j - R) p + (t_j - t)) / h exactly; the generic kernel forms the difference per
 * residual in floating point as linearization.h:97-111 does (same Jacobian up to that subtraction's rounding).
 * The camera models (pinhole, pinhole + distortion) with fp32 compute likewise form the same quotient
 * (f(x + h e_j) - f_ref) / H over a common denominator / from the parameter-wise affine structure of the residual
 * instead of subtracting two float-rounded ~1e3-pixel projections; with this flag they use the per-residual form. */
/* MOPT_FLAG_STABLE_FD: opt the fp64-compute finite differences of the camera models into the same common-denominator
 * form (by default fp64 compute is the literal per-residual restatement of linearization.h:97-111, the path compared
 * with the reference at 1e-10 / 1e-6).  Same quotient without the eps/h rounding of the subtraction, and 26 IEEE
 * divisions per observation fewer.  Ignored where no such form exists. */
/* MOPT_FLAG_REFERENCE_FLOAT_GUARD: with compute_dtype MOPT_F32, so3::Exp returns the identity below |omega| = 10 eps_f32
 * (1.2e-6) exactly as the reference's float instantiation does (src/so3.cpp:47).  By default the device derives the
 * rotation in fp64 for either Scalar and uses the fp64 threshold: inside that ball every finite-difference column of
 * the rotation block is exactly zero, and an LM run started at omega = 0 with a heavily damped first step can land in
 * it and never leave (DESIGN.md §3.2). */
typedef enum mopt_problem_flags {
  MOPT_FLAG_GENERIC_KERNEL = 1,
  MOPT_FLAG_STABLE_FD = 2,
  MOPT_FLAG_REFERENCE_FLOAT_GUARD = 4
} mopt_problem_flags;

/* Optimizer knobs: optimizer.h:19,33-37, levenberg_marquadt_dyn.cpp:9,16, levenberg_marquadt_dyn.h:22-24. */
typedef struct mopt_lm_options {
  int32_t max_iterations;    /* default 15 */
  int32_t lm_max_iterations; /* default 3  */
  double lambda_factor;      /* default 1e-9 */
  int32_t scalar_dtype;      /* mopt_dtype of the LM arithmetic (lambda, rho, solve): the reference's Scalar */
  int32_t speculative;       /* 1: every trial pass evaluates cost AND H,b at x+delta so an accepted step needs
                                no second pass (valid while model->update(x) is a no-op); 0: reference pass order */
  int32_t flags;             /* mopt_lm_flags; mopt_lm_default_options sets MOPT_LM_STAGNATION_STOP */
  int32_t reserved;
} mopt_lm_options;
/* MOPT_LM_STAGNATION_STOP: end with SMALL_DELTA (CONVERGED if the cost is small) when an accepted step is below
 * isDeltaSmall's threshold (delta.h:11-16) AND left sum r^T r bit-for-bit unchanged.  The reference accepts such a
 * step (rho = 0 is not < 0, levenberg_marquadt_dyn.cpp:97), doubles lambda (:113) and carries on; it leaves that
 * state only because its y0 (serial loop, linearization.h:142-154) and y_i (TBB parallel_reduce, :52-62) are summed
 * in different orders, so that the sign of rho is rounding noise and the next negative one returns SMALL_DELTA
 * (:98-101).  On the device both sums come from the same deterministic kernel and the noise never arrives: without
 * this flag such a run spends every remaining iteration on rho = 0 steps (DESIGN.md "LM tail").  0 = literal. */
typedef enum mopt_lm_flags { MOPT_LM_STAGNATION_STOP = 1 } mopt_lm_flags;

typedef struct mopt_lm_trial {
  int32_t outer_iteration, k, accepted, reserved;
  double y0, yi, rho, lambda, nu;
} mopt_lm_trial;

typedef struct mopt_lm_report {
  int32_t status;              /* mopt_optimization_status */
  int32_t executed_iterations; /* Optimizer::getExecutedIterations, optimizer.h:44 */
  int32_t num_trials;
  int32_t num_passes;          /* full passes over the residuals executed on the device */
  double final_cost;           /* last accepted sum r^T r */
  mopt_lm_trial trials[MOPT_MAX_TRACE];
} mopt_lm_report;

/* Synthetic workloads generated on the device by a counter-based hash of (seed, global index) — the value of
 * element i does not depend on how the set is sharded (csrc/mopt_store.cu); read it back with
 * mopt_store_download to run a host implementation on identical data. */
typedef struct mopt_synth {
  uint64_t seed;
  int64_t first_index; /* global index of this store's element 0 (rank offset when sharded) */
  double gt[MOPT_MAX_PARAMETERS]; /* ground-truth parameters */
  double lo[3], hi[3]; /* p2p: source box; curve: t range lo[0]..hi[0] over n_total; pinhole: frustum box */
  int64_t n_total;     /* curve: t_i = lo + (hi-lo) * i / n_total */
  double noise_sigma;  /* approx. Gaussian (Irwin-Hall 4) noise added to B */
  double outlier_fraction, outlier_range; /* fraction of elements whose B gets U(-range, range) added */
  double consts[32];   /* model constants (same meaning as mopt_problem.consts), e.g. the pinhole frame conversion */
} mopt_synth;

/* ---- library ------------------------------------------------------------------------------- */
MOPT_API const char* mopt_last_error(void);        /* text of the calling thread's last failure */
MOPT_API const char* mopt_version(void);
MOPT_API int mopt_device_count(int* count);

/* ---- context ------------------------------------------------------------------------------- */
MOPT_API int mopt_ctx_create(int device, mopt_ctx** out);
/* Sharded operation: one context per process/GPU.  `nccl_unique_id` is MOPT_NCCL_ID_BYTES bytes obtained
 * from mopt_comm_unique_id() on rank 0 and broadcast by the host (e.g. torch.distributed).  After this,
 * linearize / compute_cost / lm_minimize return the sum over all ranks' stores (one fp64 all-reduce of
 * P(P+1)/2 + P + 1 values per pass), identical on every rank. */
MOPT_API int mopt_ctx_create_sharded(int device, int rank, int world_size, const void* nccl_unique_id, mopt_ctx** out);
MOPT_API int mopt_comm_unique_id(void* out_id);
/* NVLink peer exchange instead of NCCL: the last CTA of every pass stores the packed result straight into every
 * rank's exchange buffer (P2P stores through NVSwitch), then waits for every rank's slot in its own buffer and sums
 * the slots in rank order — pass and collective are one kernel (MOPT_PEER_CONSUMER=kernel in the environment keeps
 * the consumer as a separate one-warp kernel, for A/B).
 * Each rank publishes mopt_ctx_peer_handle (MOPT_PEER_HANDLE_BYTES bytes, a CUDA IPC handle), the host gathers
 * them in rank order and every rank calls mopt_ctx_open_peers.  With this open, `nccl_unique_id` of
 * mopt_ctx_create_sharded may be NULL. */
#define MOPT_PEER_HANDLE_BYTES 64
MOPT_API int mopt_ctx_peer_handle(mopt_ctx* ctx, void* out_handle);
MOPT_API int mopt_ctx_open_peers(mopt_ctx* ctx, const void* handles_in_rank_order);
/* Diagnostics: 0 makes every call return this rank's local sums only (no collective), e.g. to time each shard's
 * pass without the lock-step coupling of the exchange.  Must be switched identically on every rank. */
MOPT_API int mopt_ctx_set_exchange_enabled(mopt_ctx* ctx, int enabled);
MOPT_API int mopt_ctx_destroy(mopt_ctx* ctx);
MOPT_API int mopt_ctx_synchronize(mopt_ctx* ctx);
/* cudaStream_t of the context as an integer (for CUDA-event timing by the caller). */
MOPT_API int mopt_ctx_stream(mopt_ctx* ctx, uint64_t* out_stream);
/* Tuning: CTAs per SM / threads per CTA of the pass kernels (0 = default). */
MOPT_API int mopt_ctx_set_launch(mopt_ctx* ctx, int ctas_per_sm, int threads);

/* ---- device-buffer residual store ---------------------------------------------------------- */
/* Replaces the caller-owned std::vector data the reference models point into
 * (tst/point2point.cpp:82-83, tst/curve_fitting.cpp:95, tst/camera_calibration.cpp:46-47). */
MOPT_API int mopt_store_create(mopt_ctx* ctx, int model, int dtype, int64_t n, mopt_store** out);
MOPT_API int mopt_store_destroy(mopt_store* store);
MOPT_API int mopt_store_size(const mopt_store* store, int64_t* n);
/* Copy `count` elements of data group `group` (0 = A, 1 = B, see mopt_model) from a host AoS array into
 * elements [first, first+count).  Element i's components are host[(i*host_stride) + c], c < ncomp(group);
 * host_stride = 0 means packed (= ncomp).  Converts host_dtype -> store dtype on the device. */
MOPT_API int mopt_store_upload(mopt_store* store, int group, const void* host, int host_dtype, int64_t host_stride,
                      int64_t first, int64_t count);
MOPT_API int mopt_store_download(mopt_store* store, int group, void* host, int host_dtype, int64_t first, int64_t count);
MOPT_API int mopt_store_generate(mopt_store* store, const mopt_synth* desc);

/* ---- the hot path -------------------------------------------------------------------------- */
/* CostFunction*Dynamic::linearize (src/cost_function_*_dyn.cpp:25-30) -> computeHessian /
 * computeHessianNumerical (linearization.h:65-158).  H is P x P full symmetric (column-major ==
 * row-major), b is P, *sum = sum r^T r (unweighted).  x, H, b, sum are host pointers. */
MOPT_API int mopt_linearize(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const double* x, double* H,
                   double* b, double* sum);
/* CostFunction*Dynamic::computeCost (src/cost_function_*_dyn.cpp:19-22) -> parallelComputeCost
 * (linearization.h:49-63). */
MOPT_API int mopt_compute_cost(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const double* x, double* sum);
/* Same as mopt_linearize but asynchronous and device-resident: x is read from / (H upper-packed, b, sum)
 * written to device memory owned by the context (`mopt_ctx_result` fetches them).  Used for timing the
 * kernel without host round trips. */
MOPT_API int mopt_linearize_async(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const double* x);
MOPT_API int mopt_ctx_result(mopt_ctx* ctx, int num_parameters, double* H, double* b, double* sum);

/* ---- per-residual evaluation ------------------------------------------------------------------ */
/* Fit statistics of one cost term over a range of its store (mopt_evaluate).  Counts and sums add across the
 * ranks of a sharded problem and max_sq combines by maximum: each rank evaluates its own store only. */
typedef struct mopt_eval_stats {
  int64_t n_valid;        /* elements of the range whose residual exists (not masked, see mopt_evaluate) */
  int64_t n_inliers;      /* valid elements with r^T r <= inlier_threshold^2 */
  double sum_sq;          /* sum of r^T r over valid elements: mopt_compute_cost's value over the same range */
  double inlier_sum_sq;   /* sum of r^T r over inliers */
  double max_sq;          /* max r^T r over valid elements (0 if none) */
  double reserved[3];
} mopt_eval_stats;

/* CostComputation::computeCost's loop body (linearization.h:36-47) with each element's result kept:
 * for the elements [first, first + count) of `store` at x, optionally write the residual r_i (count x O,
 * row-major: element i's O components are contiguous) and the loss weight w_i = loss(r_i^T r_i), both in
 * `out_dtype`, to DEVICE memory on the context's device.  `residuals`, `weights` and `stats` may each be NULL,
 * but not all three.  Returns after the context stream is synchronised.
 *   - r_i is the model residual in problem.compute_dtype arithmetic at setup(x); w_i is the IRLS weight the pass
 *     kernels apply.  The covariance, jacobian, variant and manifold fields have no effect.
 *   - Elements without a correspondence (point2point stores with an attached target index, see
 *     mopt_store_reassociate) get NaN in every residual component and weight 0, and enter no statistic.
 *   - Evaluation never re-associates: a store with a target index is evaluated with the correspondences it holds
 *     now.  Call mopt_store_reassociate(store, x) first to evaluate at fresh correspondences.
 *   - Statistics are accumulated in fp64 and reduced in a fixed order: identical bits from run to run, whichever
 *     outputs are written.  inlier_threshold = +inf counts every valid element as an inlier.
 *   - Sharded contexts: this rank's store only, no collective (see mopt_eval_stats).
 * MOPT_ERR_INVALID_ARGUMENT, with nothing written, for a range outside the store, out_dtype not MOPT_F32 /
 * MOPT_F64, residuals or weights with count 0, or all three outputs NULL. */
MOPT_API int mopt_evaluate(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const double* x,
                           int64_t first, int64_t count, double inlier_threshold, int out_dtype,
                           void* residuals, void* weights, mopt_eval_stats* stats);

/* ---- hypothesis scoring ----------------------------------------------------------------------- */
#define MOPT_MAX_HYPOTHESES 1024
/* mopt_evaluate's statistics (no per-element outputs) at n_hyp parameter vectors in one call: out[k] is what
 * mopt_evaluate(ctx, store, problem, xs + k * P, first, count, inlier_threshold, ..., &stats) returns.  The store is
 * read once per 32 hypotheses instead of once per hypothesis, so from 32 hypotheses on a call costs arithmetic rather
 * than memory traffic: the scoring step of RANSAC (minimal-sample hypotheses against all putative correspondences)
 * and of multi-start fits.  Returns after the context stream is synchronised.
 *   - Exact parts.  n_valid, n_inliers and max_sq of out[k] equal mopt_evaluate's at xs[k] bit for bit, for every
 *     builtin and user model and dtype pair: the same set-up (x rounded to the compute Scalar, then model setup),
 *     the same residual, the same key e2 = sum fma(r_o, r_o) in the compute dtype and the same test
 *     double(e2) <= inlier_threshold^2.  They do not depend on n_hyp, on k's place in the batch or on
 *     mopt_ctx_set_launch, so a caller with more than MOPT_MAX_HYPOTHESES hypotheses splits them over calls.
 *   - Sums.  sum_sq and inlier_sum_sq accumulate double(e2) in fp64 like mopt_evaluate's, in another order: they
 *     agree with its sums to rounding, and are identical from run to run for the same inputs and launch settings.
 *   - As mopt_evaluate: masked elements (no correspondence) enter no statistic, correspondences are never
 *     re-associated, count = 0 gives all-zero statistics, and the covariance, loss, jacobian, variant and manifold
 *     fields have no effect.  A non-finite hypothesis gets what mopt_evaluate gives at that x and does not affect
 *     the others.
 *   - Sharded contexts: this rank's store only, no collective (see mopt_eval_stats).
 * MOPT_ERR_INVALID_ARGUMENT, with nothing written, for n_hyp outside [1, MOPT_MAX_HYPOTHESES], a null xs or out, a
 * model without parameters, a store of another context, a problem the store does not accept, a range outside the
 * store or a negative inlier_threshold. */
MOPT_API int mopt_score_hypotheses(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, int n_hyp,
                                   const double* xs /* n_hyp x P, row-major, host */, int64_t first, int64_t count,
                                   double inlier_threshold, mopt_eval_stats* out /* n_hyp, host */);

/* ---- residual quantiles ----------------------------------------------------------------------- */
#define MOPT_MAX_QUANTILES 8
/* Exact order statistics of the keys e_i = r_i^T r_i of one cost term over a range of its store
 * (mopt_residual_quantiles).  Unlike the counts and sums of mopt_eval_stats, quantiles do NOT combine across the
 * ranks of a sharded problem: each rank gets the quantiles of its own store. */
typedef struct mopt_quantiles {
  int64_t n_ranked;                 /* valid elements of the range whose e_i is not NaN: the sample */
  int64_t n_nan;                    /* valid elements whose e_i is NaN (not ranked) */
  double lo[MOPT_MAX_QUANTILES];    /* e_(j),   j = floor(h), h = (n_ranked - 1) * q  (0-based order statistics) */
  double hi[MOPT_MAX_QUANTILES];    /* e_(j+1), clamped to e_(n_ranked - 1) */
  double value[MOPT_MAX_QUANTILES]; /* numpy's method="linear" interpolation of lo, hi */
  double median;                    /* value at q = 0.5, always computed */
  double robust_sigma;              /* sqrt(median / chi2_median(O)) */
  double reserved[4];
} mopt_quantiles;

/* Quantiles of e_i = r_i^T r_i over the elements [first, first + count) of `store` at x, for n_q levels q[0..n_q)
 * (host arrays), plus the median and the median-based robust scale.  Exact: every lo / hi is one element's e_i.
 * Returns after the context stream is synchronised.
 *   - The key.  r_i is the residual mopt_evaluate computes (the model residual in problem.compute_dtype at
 *     setup(x)).  e_i is summed in the compute dtype in component order, every product and sum rounded separately
 *     (no fused multiply-add): e = r_0 r_0, then e = e + r_o r_o for o = 1 .. O-1.  mopt_evaluate's residuals written
 *     with out_dtype = compute_dtype reproduce it exactly; it can differ in the last bit from the FMA-formed r^T r
 *     behind mopt_eval_stats and the loss weight.  The covariance, loss, jacobian, variant and manifold fields
 *     have no effect.
 *   - The sample.  Elements without a correspondence (as in mopt_evaluate) are excluded.  A valid element whose
 *     e_i is NaN (NaN data) is counted in n_nan and not ranked; +inf is ranked and sorts last.  Never
 *     re-associates correspondences.
 *   - Quantiles (q in [0, 1]).  lo, hi and value are what np.quantile(e.astype(np.float64), q) (method "linear")
 *     takes and returns: h = (n_ranked - 1) q in fp64, j = floor(h), t = h - j, value = lo + (hi - lo) t, or
 *     hi - (hi - lo)(1 - t) when t >= 0.5.  One difference: value = lo when t = 0 (numpy gives NaN for a finite lo
 *     next to hi = +inf).
 *   - robust_sigma = sqrt(median / m_O), m_O the median of the chi-square distribution with O degrees of freedom
 *     (O = problem.num_outputs): 1.4826 median|r| for O = 1, and a consistent estimate of the per-component sigma
 *     for isotropic Gaussian noise.
 *   - An empty sample (n_ranked = 0) returns MOPT_OK with the counts set and every value NaN.
 *   - Results are exact element values: identical from run to run, whatever the grid or mopt_ctx_set_launch.
 *   - Sharded contexts: this rank's store only, no collective (see mopt_quantiles).
 * MOPT_ERR_INVALID_ARGUMENT, with nothing written, for a store of another context, a problem the store does not
 * accept, a range outside the store, n_q outside [0, MOPT_MAX_QUANTILES], a q that is NaN or outside [0, 1], a
 * null q with n_q > 0, a null out, or a null x for a model with parameters. */
MOPT_API int mopt_residual_quantiles(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const double* x,
                                     int64_t first, int64_t count, int n_q, const double* q, mopt_quantiles* out);

/* ---- parameter covariance at a solution ------------------------------------------------------- */
/* How certain is x?  Two calls: mopt_covariance_terms streams the stores on the device and returns ADDITIVE terms;
 * mopt_covariance_from_terms (host only) turns terms into a P x P covariance.  The caller of a sharded problem sums
 * the terms of its ranks between the two calls (every field but num_parameters adds), as it does with
 * mopt_eval_stats: the device part is rank-local and runs no collective. */
typedef enum mopt_cov_estimator {
  MOPT_COV_UNSCALED = 0, /* H^+: the cost terms' covariance matrices (setCovariance) already are the inverse noise covariances */
  MOPT_COV_SCALED = 1,   /* s^2 H^+, s^2 = wsse / (m - rank): noise level estimated from the fit (scipy curve_fit's pcov) */
  MOPT_COV_SANDWICH = 2  /* H^+ G H^+ (HC0): robust to a mis-specified noise model, heteroscedasticity and IRLS weights */
} mopt_cov_estimator;

typedef struct mopt_cov_terms { /* every field adds across cost terms and across the ranks of a sharded problem */
  int32_t num_parameters;       /* P (not added: must agree) */
  int32_t reserved0;
  int64_t n_valid;              /* elements that have a residual (ICP elements without a correspondence excluded) */
  int64_t m;                    /* residual components: sum over cost terms of n_valid * O */
  double H[MOPT_MAX_PARAMETERS * MOPT_MAX_PARAMETERS]; /* sum w J^T C J, P x P column-major: what mopt_linearize returns */
  double G[MOPT_MAX_PARAMETERS * MOPT_MAX_PARAMETERS]; /* sum g g^T, g = w J^T C r, P x P column-major */
  double b[MOPT_MAX_PARAMETERS]; /* sum g: mopt_linearize's b */
  double wsse;                  /* sum w r^T C r */
  double sum_sq;                /* sum r^T r: mopt_linearize's sum */
  double reserved[4];
} mopt_cov_terms;               /* H and G fill their first P*P entries (leading dimension P); the rest is 0 */

typedef struct mopt_cov_report {
  int32_t rank;                 /* eigenvalues of the scaled H kept (see mopt_covariance_from_terms) */
  int32_t reserved0;
  int64_t dof;                  /* m - rank */
  double sigma2;                /* s^2 = wsse / dof (computed for every estimator, used by MOPT_COV_SCALED) */
  double eig_min, eig_max;      /* smallest kept / largest eigenvalue of the Jacobi-scaled H */
  double reserved[3];
} mopt_cov_report;

/* Terms at x of n_costs cost terms sharing x (same P), on the device.  x is a host pointer.
 *   - H, b, sum_sq come from the linearization pass kernels, accumulated over the cost terms in order as
 *     mopt_lm_minimize does; for one cost term on an unsharded context they are bit-identical to mopt_linearize's.
 *   - G, wsse and n_valid come from one more streaming sweep per cost term (score_gram_kernel).  Its Jacobian of
 *     each residual is the one the linearization of the same problem and flags uses (the affine point2point form, the
 *     common-denominator finite differences of the camera models and of the exp curve where those are selected, the
 *     per-residual differences or the model's f_df otherwise), so that G and H describe the same linearization.
 *     Sums in fp64 (fp32 compute: fp32 partials folded into fp64 as the passes do), reduced in a fixed order:
 *     identical bits from run to run.
 *   - Never re-associates (as mopt_evaluate): a store with a target index is taken with the correspondences it holds.
 *   - Sharded contexts: this rank's stores only, no collective.  Returns after the context stream is synchronised.
 * MOPT_ERR_INVALID_ARGUMENT, with nothing written, for n_costs outside [1, MOPT_MAX_COSTS], a store of another
 * context, a null x, a model without parameters or cost terms whose P differ. */
MOPT_API int mopt_covariance_terms(mopt_ctx* ctx, int n_costs, mopt_store* const* stores, const mopt_problem* problems,
                                   const double* x, mopt_cov_terms* out);
/* Host only, needs no GPU: the P x P column-major covariance of x (in the tangent space at x for
 * MOPT_MANIFOLD_SO3_LEFT) from terms.
 *   - Pseudo-inverse: D = diag(H)^(-1/2) (0 for a zero diagonal entry: that parameter is unobservable), S = D H D,
 *     symmetric eigendecomposition of S by cyclic Jacobi in fp64, eigenvalues lambda > rcond * lambda_max kept,
 *     H^+ = D S^+ D with S^+ the truncated inverse.  For a full-rank H this is H^-1 up to rounding.  rcond = 0
 *     selects 1e-10; problems with fp32 compute and a near-null direction want about 1e-6.
 *   - MOPT_COV_UNSCALED returns H^+, MOPT_COV_SCALED sigma2 H^+ (sigma2 = wsse / dof, dof = m - rank),
 *     MOPT_COV_SANDWICH H^+ G H^+ with no small-sample factor.  The bread is the Gauss-Newton H the LM iterates with;
 *     for robust losses that is the usual IRLS approximation of the M-estimator's sandwich.
 *   - `report` may be NULL.
 * MOPT_ERR_INVALID_ARGUMENT, with nothing written, for num_parameters outside [1, MOPT_MAX_PARAMETERS], an unknown
 * estimator, a negative rcond, non-finite terms or dof <= 0. */
MOPT_API int mopt_covariance_from_terms(const mopt_cov_terms* terms, int estimator, double rcond, double* cov,
                                        mopt_cov_report* report);

/* ---- closed-form rigid alignment -------------------------------------------------------------- */
/* The best rigid transform for the correspondences a point2point store holds: the weighted Kabsch / Horn solution.
 * Two calls, as for the covariance: mopt_align_terms streams the store once on the device and returns the weighted
 * first and second moments of the pairs it uses; mopt_align_from_terms (host only) solves for x = [t, omega].  Terms
 * of several ranges or of the ranks of a sharded problem combine with mopt_align_terms_merge, not field by field. */
typedef struct mopt_align_moments { /* the terms: combine with mopt_align_terms_merge, NOT by adding fields */
  int64_t n_valid;     /* elements of the range with a correspondence: mopt_evaluate's n_valid */
  int64_t n_used;      /* valid elements with double(e2(x)) <= thr^2: mopt_evaluate's n_inliers; they enter the moments */
  double w;            /* sum of w_i over used elements */
  double mean_src[3];  /* weighted mean of p (group A) */
  double mean_tgt[3];  /* weighted mean of q (group B) */
  double cross[9];     /* cross[3a+b] = sum w (p_a - mean_src_a)(q_b - mean_tgt_b) */
  double var_src;      /* sum w |p - mean_src|^2 */
  double var_tgt;      /* sum w |q - mean_tgt|^2 */
  double reserved[4];
} mopt_align_moments;

typedef struct mopt_align_report {
  double cost;         /* sum w |R p + t - q|^2 at the solution = max(0, var_src + var_tgt - 2 eig[0]) */
  double rms;          /* sqrt(cost / w) */
  double eig[4];       /* eigenvalues of Horn's 4x4 matrix N, descending */
  int32_t degenerate;  /* eig[0] - eig[1] <= 1e-12 * |eig[0]|: rotation not unique (collinear / < 3 distinct points) */
  int32_t reserved0;
  double reserved[3];
} mopt_align_report;

/* Alignment terms of the elements [first, first + count) of a MOPT_MODEL_POINT2POINT store at x (host pointer), on
 * the device.  Returns after the context stream is synchronised.
 *   - Which elements enter.  Element i is used when it has a correspondence and double(e2_i) <= inlier_threshold^2,
 *     e2_i = sum fma(r_o, r_o) of the residual on set 0 in problem.compute_dtype at x: mopt_evaluate's inlier test,
 *     so n_valid and n_used equal mopt_evaluate's n_valid and n_inliers bit for bit.  NaN data and NaN keys never
 *     enter.  inlier_threshold = +inf takes every valid element.
 *   - Weights.  w_i is the loss weight of e2_i in the compute dtype (what mopt_evaluate writes to `weights` with
 *     out_dtype = compute_dtype), converted to fp64; MOPT_LOSS_NONE gives w = 1.  With a robust loss one call and one
 *     solve are one IRLS step of the robust closed-form fit.
 *   - Moments of the store values p_i, q_i (converted exactly to fp64), not of T(x) p_i, accumulated in fp64 in
 *     centred form and combined in a fixed order: identical bits from run to run for the same launch settings, equal
 *     to rounding under another mopt_ctx_set_launch.  They stay accurate on clouds far from the origin.
 *   - The covariance, jacobian, variant and manifold fields have no effect.  Correspondences are never re-associated:
 *     call mopt_store_reassociate(store, x) first for fresh ones.
 *   - Sharded contexts: this rank's store only, no collective (merge the ranks' terms with mopt_align_terms_merge).
 *   - count = 0 gives all-zero terms.
 * MOPT_ERR_INVALID_ARGUMENT, with nothing written, for a store whose model is not point2point, a store of another
 * context, a problem the store does not accept, a range outside the store, a NaN or negative inlier_threshold, or a
 * null x or out. */
MOPT_API int mopt_align_terms(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const double* x,
                              int64_t first, int64_t count, double inlier_threshold, mopt_align_moments* out);
/* Host only: the terms of the union of two disjoint sets of pairs (Chan's pairwise rule: counts and w add, means
 * combine by weight, cross and var gain Wa Wb / W d_src d_tgt^T with d the difference of the means).  merge(a, b) and
 * merge(b, a) are identical bits; an operand with w = 0 leaves the other's moments unchanged (its counts still add).
 * `out` may alias `a` or `b`.  Accuracy: each mean of the struct is one double, so far from the origin it carries up to
 * half an ulp of rounding (6e-11 at 1e6), which the merge takes into cross and var at first order.  For a cloud 1e6 from
 * the origin with unit spread, merged terms agree with one-shot moments to about 1e-12 of the largest moment after one
 * merge and 8e-12 after 63 (1e-15 near the origin), so fold few terms, such as one per rank.  mopt_align_terms itself
 * carries each mean's rounding error through its device reduction and does not have this loss.
 * MOPT_ERR_INVALID_ARGUMENT for a null argument. */
MOPT_API int mopt_align_terms_merge(const mopt_align_moments* a, const mopt_align_moments* b,
                                   mopt_align_moments* out);
/* Host only, needs no GPU: Horn's quaternion solution of min sum w |R p + t - q|^2 from terms.  N (4x4 symmetric) is
 * built from `cross`, the eigenvector of its largest eigenvalue (cyclic Jacobi in fp64) is the rotation as a unit
 * quaternion (w >= 0), t = mean_tgt - R mean_src and omega = 2 atan2(|v|, w) v / |v| (|omega| <= pi).  x_out = [t, omega]
 * (6 doubles) is the point2point parameter vector: a start for mopt_lm_minimize or a hypothesis for
 * mopt_score_hypotheses.  R is always a proper rotation.  `report` may be NULL.  A degenerate configuration returns
 * MOPT_OK with one of the minimisers and report->degenerate = 1.
 * MOPT_ERR_INVALID_ARGUMENT, with nothing written, for a null terms or x_out, w <= 0 or non-finite terms. */
MOPT_API int mopt_align_from_terms(const mopt_align_moments* terms, double* x_out, mopt_align_report* report);

/* End-to-end convenience: upload host AoS data (group A and B) into `store` and linearize, with the
 * host->device copies chunked and overlapped with the device work. */
MOPT_API int mopt_upload_and_linearize(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const void* host_a,
                              const void* host_b, int host_dtype, int64_t count, const double* x, double* H,
                              double* b, double* sum);

/* LevenbergMarquadtDynamic<Scalar>::minimize (src/levenberg_marquadt_dyn.cpp:34-119) over `n_costs` cost
 * terms (addCost, optimizer.h:58), entirely on the device: linearization passes, the damped P x P LDL^T
 * solve, gain ratio and accept/reject never round-trip through the host.  x is in/out (host pointer). */
MOPT_API int mopt_lm_minimize(mopt_ctx* ctx, int n_costs, mopt_store* const* stores, const mopt_problem* problems,
                     const mopt_lm_options* options, double* x, mopt_lm_report* report);
MOPT_API void mopt_lm_default_options(mopt_lm_options* options);

/* ---- small host-side math kept for API parity (src/so3.cpp:7-19,43-57; delta.h:11-16) -------- */
MOPT_API int mopt_so3_convert6dof(const double* x, double* T16_rowmajor);
MOPT_API int mopt_ldlt_solve(int n, const double* A_colmajor, const double* rhs, double* out);

/* ---- correspondence re-association: model->update(x) (SURVEY.md §8f-1) ------------------------------ */
/* The reference calls cost->update(x0) -> model->update(x) before every linearization
 * (src/levenberg_marquadt_dyn.cpp:54; include/moptimizer/model.h:24-26 "i.e registration correspondences") but
 * ships no implementation.  A mopt_nn_index holds a fixed TARGET cloud in a device uniform grid; attached to a
 * point2point store it makes update(x) mean: tgt_i <- nearest target point of T(x) src_i within `max_distance`,
 * source points without one being skipped by later passes (model f returning false, linearization.h:102,144).
 * The match is the brute-force nearest neighbour:
 *   - ties go to the lowest original index of the target cloud;
 *   - the radius is inclusive: a target at exactly max_distance matches;
 *   - an fp32 index (index_dtype = MOPT_F32) forms the query and the distances in fp32 from fp32-rounded data and
 *     writes fp32-rounded target coordinates;
 *   - a target point with a non-finite coordinate is kept but never matches (it does not size the grid either).
 * max_distance must be positive and finite. */
typedef struct mopt_nn_index mopt_nn_index;
MOPT_API int mopt_nn_index_create(mopt_ctx* ctx, const void* host_xyz, int host_dtype, int index_dtype, int64_t m,
                                  double max_distance, mopt_nn_index** out);
MOPT_API int mopt_nn_index_destroy(mopt_nn_index* index);
/* Attach (or detach with NULL) the target cloud.  With one attached, mopt_lm_minimize re-associates at the start
 * of every outer iteration, exactly where the reference calls cost->update(x0), and uses the reference pass order. */
MOPT_API int mopt_store_set_target(mopt_store* store, mopt_nn_index* index);
/* CostFunctionBase::update(x) (cost_function.h:44): re-associate now; *matched = correspondences found. */
MOPT_API int mopt_store_reassociate(mopt_store* store, const double* x, int64_t* matched);

/* ---- point-cloud ingest (input side of the path) ---------------------------------------------------- */
/* tst/point2point.cpp:125-138 `txt_cloud_loader`: whitespace-separated records of `columns` numbers (the
 * fixture tst/data/fachada.txt has 6: x y z r g b); the first `keep` of each record are stored, AoS, in
 * `host_dtype`.  Parsing stops at the first malformed record, as the reference's stream extraction does.
 * `pinned` != 0 allocates page-locked memory (needs a CUDA device) so mopt_store_upload runs at full speed.
 * Free with mopt_cloud_free(ptr, pinned). */
MOPT_API int mopt_cloud_read_text(const char* path, int columns, int keep, int host_dtype, int pinned, void** out,
                                  int64_t* n);
/* Raw binary cache of a parsed cloud: 24-byte header {"MOPTCLD1", int64 n, int32 dtype, int32 keep} + AoS data. */
MOPT_API int mopt_cloud_write_binary(const char* path, const void* data, int host_dtype, int keep, int64_t n);
MOPT_API int mopt_cloud_read_binary(const char* path, int pinned, int* host_dtype, int* keep, void** out, int64_t* n);
MOPT_API int mopt_cloud_free(void* ptr, int pinned);

/* ---- user-defined device models (SURVEY.md §8f-4) --------------------------------------------------- */
/* IBaseModel's virtual f / f_df / setup (include/moptimizer/model.h:19-42) are host functions and cannot run in a
 * kernel.  A user model is therefore given as CUDA C++ SOURCE and compiled at run time (NVRTC, sm_100a) INTO the
 * same pass kernels the builtin models use: residual + analytical or finite-difference Jacobian + loss weighting +
 * packed H / b accumulation + the three-level reduction, with the user's functions inlined.  The source defines
 *
 *   template <typename T>   // T = float or double: mopt_problem.compute_dtype, the reference's Scalar
 *   __device__ void mopt_f(const T* s, const T* a, const T* b, T* r);             // model.h:33  f(x, r, index)
 *   template <typename T>
 *   __device__ void mopt_f_df(const T* s, const T* a, const T* b, T* r, T* J);    // model.h:42  f_df, J row-major O x P
 *   __device__ void mopt_setup(const double* x, const double* consts, double* s); // model.h:19  setup(x), optional
 *
 * `a` / `b` are the ncomp_a / ncomp_b data components of ONE residual (what the reference models fetch from their
 * caller-owned vectors with `index`), `s` is x itself or, when set_size > 0, the set_size values mopt_setup derived
 * from x (and from mopt_problem.consts) — evaluated once per pass on the device, also for every finite-difference
 * perturbation of x, exactly where linearization.h:84-93 calls setup on the cloned models.  mopt_f_df is only
 * required with has_jacobian.  Helpers of csrc/mopt_setup.cuh (mopt::so3_exp_dev, ...) are visible to the source. */
typedef struct mopt_user_model_desc {
  int32_t num_parameters; /* P in [1, MOPT_MAX_PARAMETERS] */
  int32_t num_outputs;    /* O in [1, MOPT_MAX_OUTPUTS] */
  int32_t ncomp_a;        /* components of data group A (>= 1) */
  int32_t ncomp_b;        /* components of data group B; ncomp_a + ncomp_b <= 6 planar streams */
  int32_t has_jacobian;   /* the source defines mopt_f_df (MOPT_JAC_ANALYTICAL allowed) */
  int32_t set_size;       /* 0: s = x;  1..24: the source defines mopt_setup writing this many values */
  int32_t rot_offset;     /* index of a rotation-vector block in x for MOPT_MANIFOLD_SO3_LEFT, or -1 */
  int32_t reserved;
} mopt_user_model_desc;
/* Compiles the model (the fp64 finite-difference variant immediately, so source errors surface here with the
 * compiler log in mopt_last_error(); other dtype / Jacobian variants on first use) and returns its model id
 * (>= MOPT_MODEL_USER_BASE) for mopt_store_create and mopt_problem.model.  Needs no GPU; launching does. */
MOPT_API int mopt_user_model_compile(const char* cuda_source, const mopt_user_model_desc* desc, int* model_id);
MOPT_API int mopt_user_model_release(int model_id);
/* Compiler log of the most recent NVRTC compilation of this model (warnings included), "" if none. */
MOPT_API const char* mopt_user_model_log(int model_id);

/* ---- measured ceilings of this box (roofline denominators; SURVEY.md §8d) --------------------------- */
/* MEASURED_PEAKS.json holds an HBM copy and a bf16 GEMM figure only.  The ALU-bound paths (finite differences of
 * the curve and camera models, computeHessianNumerical, linearization.h:65-124) are judged against an fp32 rate
 * measured here with committed micro-kernels (csrc/mopt_peaks.cu). */
typedef struct mopt_peaks {
  double fp32_fma_tflops;         /* scalar FFMA, 8 independent chains per thread, 2048 threads per SM */
  double fp32_fma2_tflops;        /* packed FFMA2 (fma.rn.f32x2), same shape */
  double issue_gwarp_inst_per_s;  /* warp instructions issued per second, in 1e9: the FFMA-only rate (1 per clock per scheduler) */
  double hbm_read_gbs;            /* read-only stream of 2 GiB, 16-byte loads */
  double reserved[4];
} mopt_peaks;
MOPT_API int mopt_measure_peaks(mopt_ctx* ctx, mopt_peaks* out);
/* Pinned host -> device copy rate of this process over at least `seconds` (concurrent callers on other GPUs
 * overlap): the ceiling of the end-to-end path that starts from host buffers (mopt_upload_and_linearize). */
MOPT_API int mopt_measure_h2d(mopt_ctx* ctx, uint64_t bytes, double seconds, double* gbs);

/* Pinned host memory for callers that want full-speed uploads. */
MOPT_API int mopt_host_alloc(void** ptr, uint64_t bytes);
MOPT_API int mopt_host_free(void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* MOPT_CAPI_H */
