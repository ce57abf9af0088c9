// Mirrors include/moptimizer/cost_function.h:15-59 (same operator API, ownership and defaults).  New: a
// device hook so the optimizer can run every pass and its own state machine on the GPU.
#pragma once

#include <cstring>
#include <memory>
#include <vector>

#include "mopt_capi.h"
#include "moptimizer/covariance/covariance.h"
#include "moptimizer/device/models.h"
#include "moptimizer/loss_function/geman_mcclure.h"
#include "moptimizer/loss_function/huber.h"
#include "moptimizer/loss_function/loss_function.h"
#include "moptimizer/model.h"
#include "moptimizer/types.h"

namespace moptimizer {

template <class Scalar = double>
class CostFunctionBase {
 public:
  using Model = IBaseModel<Scalar>;
  using ModelPtr = typename Model::Ptr;
  using ModelConstPtr = typename Model::ConstPtr;
  using LossFunctionPtr = typename loss::ILossFunction<Scalar>::Ptr;

  CostFunctionBase(ModelPtr model, int num_residuals) : num_residuals_(num_residuals), model_(model) {
    loss_function_.reset(new loss::NoLoss<Scalar>());
    covariance_.reset(new covariance::Matrix<Scalar>());
  }
  CostFunctionBase() = delete;
  CostFunctionBase(const CostFunctionBase&) = delete;
  CostFunctionBase& operator=(const CostFunctionBase&) = delete;
  virtual ~CostFunctionBase() = default;

  inline void setLossFunction(LossFunctionPtr loss_function) { loss_function_ = loss_function; }
  inline void setCovariance(const covariance::MatrixPtr<Scalar> covariance) { covariance_ = covariance; }
  /// New (opt-in, SURVEY.md §8f-3): MOPT_MANIFOLD_SO3_LEFT makes the optimizer update the rotation block of x
  /// with so3::Exp/Log instead of adding delta (the reference's "TODO Manifold operation"); Jacobians are then
  /// taken in the tangent space (use the MOPT_P2P_LEFT variant for analytical point2point).
  inline void setManifold(int manifold) { manifold_ = manifold; }
  /// New (opt-in): mopt_problem_flags for the device pass, e.g. MOPT_FLAG_STABLE_FD (double: finite differences of
  /// the camera models over a common denominator) or MOPT_FLAG_GENERIC_KERNEL (always the per-residual quotient of
  /// linearization.h:97-111).  0 by default.
  inline void setKernelFlags(int flags) { kernel_flags_ = flags; }

  virtual void update(const Scalar* x) { model_->update(x); }
  virtual Scalar computeCost(const Scalar* x) = 0;
  virtual Scalar linearize(const Scalar* x, Scalar* hessian, Scalar* b) = 0;

  /// Device description of this cost term (C-ABI problem + store).  Throws moptimizer::Exception if the model
  /// is not a builtin device model or the loss is not one the kernels implement: there is no host fallback.
  virtual void deviceProblem(mopt_problem* problem, device::Store::Ptr* store) const = 0;

  /// New: fit statistics of this cost term at x over all its residuals (mopt_evaluate without per-element outputs):
  /// valid residuals, inliers (r^T r <= inlier_threshold^2), sum r^T r, its inlier part and max r^T r.  Fitness is
  /// n_inliers / residual count, inlier RMSE sqrt(inlier_sum_sq / n_inliers).  Correspondences are not re-associated:
  /// call update(x) first for fresh ones.  Per-element residuals and weights live in device memory only, so they
  /// are read through the C ABI (mopt_evaluate on deviceProblem()'s store) by a caller that owns device buffers.
  mopt_eval_stats evaluateStatistics(const Scalar* x, double inlier_threshold) const {
    mopt_problem p;
    device::Store::Ptr st;
    deviceProblem(&p, &st);
    double xd[MOPT_MAX_PARAMETERS] = {0};
    for (int i = 0; i < p.num_parameters && x; ++i) xd[i] = double(x[i]);
    mopt_eval_stats stats;
    device::check(mopt_evaluate(st->context()->get(), st->get(), &p, xd, 0, st->size(), inlier_threshold, MOPT_F64,
                                nullptr, nullptr, &stats),
                  "mopt_evaluate");
    return stats;
  }

  /// New: evaluateStatistics at n_hyp parameter vectors xs (n_hyp x P, row-major) in one pass over the data
  /// (mopt_score_hypotheses, at most MOPT_MAX_HYPOTHESES per call): the scoring step of RANSAC and of multi-start
  /// fits.  Counts and max_sq equal evaluateStatistics' at each row exactly.  Correspondences are not re-associated.
  std::vector<mopt_eval_stats> scoreHypotheses(const Scalar* xs, int n_hyp, double inlier_threshold) const {
    mopt_problem p;
    device::Store::Ptr st;
    deviceProblem(&p, &st);
    std::vector<double> xd(size_t(n_hyp > 0 ? n_hyp : 0) * size_t(p.num_parameters));
    for (size_t i = 0; i < xd.size(); ++i) xd[i] = double(xs[i]);
    std::vector<mopt_eval_stats> out(size_t(n_hyp > 0 ? n_hyp : 0));
    device::check(mopt_score_hypotheses(st->context()->get(), st->get(), &p, n_hyp, xd.data(), 0, st->size(),
                                        inlier_threshold, out.data()),
                  "mopt_score_hypotheses");
    return out;
  }

  /// New: exact quantiles of e = r^T r over all residuals of this cost term at x (mopt_residual_quantiles) for the
  /// levels qs (at most MOPT_MAX_QUANTILES), plus the median and the robust scale sqrt(median / chi2_median(O)).
  /// sqrt of a value is the quantile of the residual norm |r|.  Correspondences are not re-associated: call
  /// update(x) first for fresh ones.
  mopt_quantiles residualQuantiles(const Scalar* x, const std::vector<double>& qs) const {
    mopt_problem p;
    device::Store::Ptr st;
    deviceProblem(&p, &st);
    double xd[MOPT_MAX_PARAMETERS] = {0};
    for (int i = 0; i < p.num_parameters && x; ++i) xd[i] = double(x[i]);
    mopt_quantiles out;
    device::check(mopt_residual_quantiles(st->context()->get(), st->get(), &p, xd, 0, st->size(), int(qs.size()),
                                          qs.empty() ? nullptr : qs.data(), &out),
                  "mopt_residual_quantiles");
    return out;
  }

  /// New: additive covariance terms of this cost at x (mopt_covariance_terms): H, b, sum r^T r of the linearization,
  /// the score Gram matrix G, wsse and the counts.  Terms of several costs, or of the ranks of a sharded problem,
  /// add field by field before mopt_covariance_from_terms.  Correspondences are not re-associated.
  mopt_cov_terms covarianceTerms(const Scalar* x) const {
    mopt_problem p;
    device::Store::Ptr st;
    deviceProblem(&p, &st);
    double xd[MOPT_MAX_PARAMETERS] = {0};
    for (int i = 0; i < p.num_parameters && x; ++i) xd[i] = double(x[i]);
    mopt_store* raw = st->get();
    mopt_cov_terms terms;
    device::check(mopt_covariance_terms(st->context()->get(), 1, &raw, &p, xd, &terms), "mopt_covariance_terms");
    return terms;
  }

  /// New: closed-form rigid alignment terms of this point2point cost at x (mopt_align_terms): the weighted moments of
  /// the source and target points of every residual with r^T r <= inlier_threshold^2, weighted by the loss weight at
  /// x.  Fold terms with mopt_align_terms_merge and solve with mopt_align_from_terms, which returns x = [t, omega].
  /// Correspondences are not re-associated: call update(x) first for fresh ones.
  mopt_align_moments alignmentTerms(const Scalar* x, double inlier_threshold) const {
    mopt_problem p;
    device::Store::Ptr st;
    deviceProblem(&p, &st);
    double xd[MOPT_MAX_PARAMETERS] = {0};
    for (int i = 0; i < p.num_parameters && x; ++i) xd[i] = double(x[i]);
    mopt_align_moments terms;
    device::check(mopt_align_terms(st->context()->get(), st->get(), &p, xd, 0, st->size(), inlier_threshold, &terms),
                  "mopt_align_terms");
    return terms;
  }

 protected:
  void fillDeviceProblem(int num_parameters, int num_outputs, int jacobian, mopt_problem* p,
                         device::Store::Ptr* store) const {
    const auto* dm = dynamic_cast<const device::IDeviceModel*>(model_.get());
    if (!dm)
      throw Exception("cost function: the model is not a device model (moptimizer/device/models.h); user-defined "
                      "host models cannot run on the GPU path and there is no CPU fallback");
    std::memset(p, 0, sizeof(*p));
    p->model = dm->kind();
    p->variant = dm->variant();
    p->num_parameters = num_parameters;
    p->num_outputs = num_outputs;
    p->jacobian = jacobian;
    p->compute_dtype = device::dtypeOf<Scalar>();
    p->manifold = manifold_;
    p->flags = kernel_flags_;
    int loss_kind = MOPT_LOSS_NONE;
    double loss_parameter = 0.0;
    if (!loss_function_ || !loss_function_->deviceLoss(&loss_kind, &loss_parameter))
      throw Exception("cost function: this loss has no device implementation (ILossFunction::deviceLoss); NoLoss, "
                      "GemmanMCClure and Huber are implemented by the kernels");
    p->loss = loss_kind;
    p->loss_param = loss_parameter;
    const int O = num_outputs;
    if (covariance_ && covariance_->rows() == O && covariance_->cols() == O) {
      bool identity = true;
      for (int r = 0; r < O; ++r)
        for (int c = 0; c < O; ++c) {
          const double v = double((*covariance_)(r, c));
          p->covariance[r + c * O] = v;
          if (v != (r == c ? 1.0 : 0.0)) identity = false;
        }
      p->has_covariance = identity ? 0 : 1;
    } else if (covariance_ && covariance_->size() != 0) {
      throw Exception("cost function: covariance must be num_outputs x num_outputs");
    }
    dm->fillConsts(p->consts);
    *store = dm->store();
  }

  int num_residuals_;
  int manifold_ = MOPT_MANIFOLD_ADDITIVE;
  int kernel_flags_ = 0;
  ModelPtr model_;
  LossFunctionPtr loss_function_;
  covariance::MatrixPtr<Scalar> covariance_;
};

namespace detail {
// Shared body of the four cost-function classes: one device pass through the C ABI.
template <class Scalar>
inline Scalar deviceLinearize(const mopt_problem& p, const device::Store::Ptr& st, const Scalar* x, Scalar* hessian,
                              Scalar* b) {
  const int P = p.num_parameters;
  double xd[MOPT_MAX_PARAMETERS] = {0}, Hd[MOPT_MAX_PARAMETERS * MOPT_MAX_PARAMETERS], bd[MOPT_MAX_PARAMETERS], sum = 0;
  for (int i = 0; i < P; ++i) xd[i] = double(x[i]);
  device::check(mopt_linearize(st->context()->get(), st->get(), &p, xd, Hd, bd, &sum), "mopt_linearize");
  for (int i = 0; i < P * P; ++i) hessian[i] = Scalar(Hd[i]);
  for (int i = 0; i < P; ++i) b[i] = Scalar(bd[i]);
  return Scalar(sum);
}
template <class Scalar>
inline Scalar deviceCost(const mopt_problem& p, const device::Store::Ptr& st, const Scalar* x) {
  double xd[MOPT_MAX_PARAMETERS] = {0}, sum = 0;
  for (int i = 0; i < p.num_parameters && x; ++i) xd[i] = double(x[i]);
  device::check(mopt_compute_cost(st->context()->get(), st->get(), &p, xd, &sum), "mopt_compute_cost");
  return Scalar(sum);
}
}  // namespace detail

}  // namespace moptimizer
