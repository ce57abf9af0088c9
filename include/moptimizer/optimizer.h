// Optimizer base of the reference API (include/moptimizer/optimizer.h:12-89): a list of non-owning cost functions, an
// iteration budget (default 15) and the minimize / step contract.  Same public members, defaults, exceptions and
// ownership rules; the device path adds gatherDeviceProblems(), which turns the cost list into what one
// mopt_lm_minimize call needs.
#pragma once

#include <cmath>
#include <iostream>
#include <limits>
#include <memory>
#include <stdexcept>
#include <vector>

#include "moptimizer/cost_function.h"
#include "moptimizer/logger.h"

namespace moptimizer {

template <class Scalar = double>
class Optimizer {
 public:
  using Ptr = std::shared_ptr<Optimizer>;
  using ConstPtr = std::shared_ptr<const Optimizer>;
  using CostFunctionType = CostFunctionBase<Scalar>;

  Optimizer() : logger_(std::make_shared<duna::Logger>(std::cout, duna::Logger::L_ERROR, "Optimizer")) {}
  Optimizer(const Optimizer&) = delete;
  Optimizer& operator=(const Optimizer&) = delete;
  virtual ~Optimizer() = default;

  // ---- iteration budget (optimizer.h:19,33-44) -------------------------------------------------------------
  void setMaximumIterations(int max_iterations) {
    if (max_iterations < 0) throw std::invalid_argument("Optimization::max_iterations cannot be less than 0.");
    maximum_iterations_ = static_cast<unsigned int>(max_iterations);
  }
  unsigned int getMaximumIterations() const { return maximum_iterations_; }
  unsigned int getExecutedIterations() const { return executed_iterations_; }

  // ---- cost list: raw, non-owning pointers unless clearCosts(true) (optimizer.h:46-66) ----------------------
  void addCost(CostFunctionType* cost) { costs_.push_back(cost); }
  void clearCosts(bool delete_costs = false) {
    if (delete_costs)
      for (CostFunctionType* c : costs_) delete c;
    costs_.clear();
  }
  bool checkCosts() const {
    if (!costs_.empty()) return true;
    std::cerr << "No cost function added!\n";
    throw std::runtime_error("No cost function added!");
  }

  /// |cost| < 8 eps of Scalar (optimizer.h:26-29); the device state machine applies the same test (csrc/mopt_lm.cuh).
  bool isCostSmall(Scalar cost_sum) { return std::abs(cost_sum) < Scalar(8) * std::numeric_limits<Scalar>::epsilon(); }

  virtual OptimizationStatus step(Scalar* x0) = 0;
  virtual OptimizationStatus minimize(Scalar* x0) = 0;

  /// New: the P x P covariance of x (column-major; tangent space at x for MOPT_MANIFOLD_SO3_LEFT) from every cost
  /// added, with `estimator` a mopt_cov_estimator (MOPT_COV_SCALED: s^2 H^-1 as scipy's curve_fit reports it).
  /// Built from the same device problems minimize() gathers, but without cost->update(x): the correspondences the
  /// stores hold now are used.  Rank-deficient problems get the truncated pseudo-inverse (report->rank).
  void computeCovariance(const Scalar* x, int estimator, Scalar* cov, mopt_cov_report* report = nullptr) const {
    checkCosts();
    std::vector<mopt_problem> problems;
    std::vector<device::Store::Ptr> stores;
    std::vector<mopt_store*> raw;
    gatherDeviceProblems(x, &problems, &stores, &raw, /*update=*/false);
    const int P = problems[0].num_parameters;
    double xd[MOPT_MAX_PARAMETERS] = {0};
    for (int i = 0; i < P; ++i) xd[i] = double(x[i]);
    mopt_cov_terms terms;
    device::check(mopt_covariance_terms(stores[0]->context()->get(), int(raw.size()), raw.data(), problems.data(), xd,
                                        &terms),
                  "mopt_covariance_terms");
    double out[MOPT_MAX_PARAMETERS * MOPT_MAX_PARAMETERS];
    device::check(mopt_covariance_from_terms(&terms, estimator, 0.0, out, report), "mopt_covariance_from_terms");
    for (int i = 0; i < P * P; ++i) cov[i] = Scalar(out[i]);
  }

 protected:
  virtual bool hasConverged() = 0;
  virtual void prepare(Scalar* x0) = 0;

  /// cost->update(x0) for every cost (levenberg_marquadt_dyn.cpp:54; skipped with update = false), then their device
  /// descriptions.  Throws if a cost is not device-backed, if there are more than MOPT_MAX_COSTS, or if they live on
  /// different contexts.
  void gatherDeviceProblems(const Scalar* x0, std::vector<mopt_problem>* problems, std::vector<device::Store::Ptr>* stores,
                            std::vector<mopt_store*>* raw, bool update = true) const {
    const size_t n = costs_.size();
    if (n > size_t(MOPT_MAX_COSTS)) throw Exception("Optimizer: too many cost functions for the device path");
    problems->resize(n);
    stores->resize(n);
    raw->resize(n);
    for (size_t i = 0; i < n; ++i) {
      if (update) costs_[i]->update(x0);
      costs_[i]->deviceProblem(&(*problems)[i], &(*stores)[i]);
      (*raw)[i] = (*stores)[i]->get();
      if ((*stores)[i]->context() != (*stores)[0]->context())
        throw Exception("Optimizer: all cost functions must live on the same device context");
    }
  }

  std::vector<CostFunctionType*> costs_;
  unsigned int maximum_iterations_ = 15;
  unsigned int executed_iterations_ = 0;
  std::shared_ptr<duna::Logger> logger_;
};

}  // namespace moptimizer
