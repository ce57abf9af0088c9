// TEST INFRASTRUCTURE ONLY: the per-element reference loop that mopt_evaluate is checked against.
// CostComputation::computeCost (include/moptimizer/linearization.h:36-47) with each element's result kept instead of
// summed, over the oracle's restated models and losses (oracle/moptimizer_oracle.hpp).  The oracle's C interface is
// compiled into this library unchanged so that the cost description (orc_cost, build, run_update) is the very one the
// other oracle entry points use; tests/oracle_evaluate.py loads it privately next to oracle/liboracle.so.
#include "oracle_capi.cpp"

namespace {

// r_i (O values), the loss weight w_i = loss(r_i^T r_i) and whether f returned true; elements where it returned
// false get NaN and weight 0.
template <class S>
int evaluate_t(const orc_cost* c, const double* x, int first, int count, double* r, double* w, int* valid) {
  auto h = build<S>(*c);
  if (!h || first < 0 || count < 0 || first + count > c->n) return 1;
  const int O = c->O;
  std::vector<S> xs(c->P > 0 ? c->P : 1), ri(O);
  for (int i = 0; i < c->P; ++i) xs[i] = S(x[i]);
  run_update<S>(c, h->cost, xs);
  IModel<S>& m = *h->cost.model;
  m.setup(xs.data());
  for (int k = 0; k < count; ++k) {
    const bool ok = m.f(xs.data(), ri.data(), unsigned(first + k));
    valid[k] = ok ? 1 : 0;
    S e2 = 0;  // CostComputation::dot
    for (int o = 0; o < O; ++o) e2 += ri[o] * ri[o];
    for (int o = 0; o < O; ++o) r[size_t(k) * O + o] = ok ? double(ri[o]) : std::nan("");
    w[k] = ok ? double(h->cost.loss->weight(e2)) : 0.0;
  }
  return 0;
}

}  // namespace

extern "C" {

// Per-element residuals (count x O, row-major), loss weights and validity of elements [first, first + count).
// scalar: 0 = float, 1 = double (the reference's two instantiations).
int orc_evaluate(const orc_cost* c, int scalar, const double* x, int first, int count, double* r, double* w,
                 int* valid) {
  return scalar ? evaluate_t<double>(c, x, first, count, r, w, valid)
                : evaluate_t<float>(c, x, first, count, r, w, valid);
}

}  // extern "C"
