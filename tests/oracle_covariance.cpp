// TEST INFRASTRUCTURE ONLY: the reference loops that mopt_covariance_terms' score Gram sums are checked against.
// CostComputation::computeHessian / computeHessianNumerical (include/moptimizer/linearization.h:65-158, restated in
// oracle/moptimizer_oracle.hpp) with the accumulation replaced by that of the score g = w J^T C r of each element:
// G = sum g g^T, wsse = sum w r^T C r and the count of elements whose model f returned true.  Each element's r, J, w
// and g are formed in the reference's Scalar exactly as accumulate() forms its b term; the three sums are kept in
// fp64.  The oracle's C interface is compiled into this library unchanged so that the cost description (orc_cost,
// build, run_update) is the very one the other oracle entry points use.
#include "oracle_capi.cpp"

namespace {

template <class S>
int score_gram_t(const orc_cost* c, const double* x, double* G, double* wsse, int64_t* n_valid) {
  auto h = build<S>(*c);
  if (!h || c->P < 1) return 1;
  const int P = c->P, O = c->O;
  std::vector<S> xs(P);
  for (int i = 0; i < P; ++i) xs[i] = S(x[i]);
  run_update<S>(c, h->cost, xs);
  IModel<S>& m = *h->cost.model;
  ILoss<S>& loss = *h->cost.loss;
  const S* C = h->cost.C.data();
  CostComputation<S> cc(P, O);
  cc.manifold_ = c->manifold;
  std::vector<double> Gd(size_t(P) * P, 0.0);
  double q = 0.0;
  int64_t count = 0;
  auto accumulate = [&]() {  // accumulate()'s b term of one element, kept as the score g
    S e2 = 0;
    for (int o = 0; o < O; ++o) e2 += cc.r_[o] * cc.r_[o];
    const S w = loss.weight(e2);
    S Cr[CostComputation<S>::kMaxO], g[CostComputation<S>::kMaxP];
    for (int o = 0; o < O; ++o) {
      S s = 0;
      for (int k = 0; k < O; ++k) s += C[o + size_t(k) * O] * cc.r_[k];
      Cr[o] = s;
    }
    S rc = 0;
    for (int o = 0; o < O; ++o) rc += cc.r_[o] * Cr[o];
    for (int a = 0; a < P; ++a) {
      S s = 0;
      for (int o = 0; o < O; ++o) s += cc.J_[size_t(o) * P + a] * Cr[o];
      g[a] = w * s;
    }
    for (int a = 0; a < P; ++a)
      for (int b = 0; b < P; ++b) Gd[a + size_t(b) * P] += double(g[a]) * double(g[b]);
    q += double(w * rc);
    ++count;
  };
  if (c->jac_mode == JAC_ANALYTICAL) {  // computeHessian
    m.setup(xs.data());
    for (int i = 0; i < c->n; ++i)
      if (m.f_df(xs.data(), cc.r_.data(), cc.J_.data(), unsigned(i))) accumulate();
  } else {  // computeHessianNumerical: same steps and perturbed models
    const bool central = c->jac_mode == JAC_CENTRAL;
    std::vector<S> hs(P), rm(O);
    std::vector<std::vector<S>> xp(P, xs), xm(P, xs);
    std::vector<std::shared_ptr<IModel<S>>> mp(P), mm(P);
    for (int j = 0; j < P; ++j) {
      cc.perturbed(xs.data(), j, hs[j], xp[j], central ? &xm[j] : nullptr);
      mp[j] = m.clone();
      mp[j]->setup(xp[j].data());
      if (central) {
        mm[j] = m.clone();
        mm[j]->setup(xm[j].data());
      }
    }
    m.setup(xs.data());
    for (int i = 0; i < c->n; ++i) {
      if (!m.f(xs.data(), cc.r_.data(), unsigned(i))) continue;
      for (int j = 0; j < P; ++j) {
        mp[j]->f(xp[j].data(), cc.rp_.data(), unsigned(i));
        if (central) {
          mm[j]->f(xm[j].data(), rm.data(), unsigned(i));
          for (int o = 0; o < O; ++o) cc.J_[size_t(o) * P + j] = (cc.rp_[o] - rm[o]) / (S(2) * hs[j]);
        } else {
          for (int o = 0; o < O; ++o) cc.J_[size_t(o) * P + j] = (cc.rp_[o] - cc.r_[o]) / hs[j];
        }
      }
      accumulate();
    }
  }
  for (size_t k = 0; k < Gd.size(); ++k) G[k] = Gd[k];
  *wsse = q;
  *n_valid = count;
  return 0;
}

}  // namespace

extern "C" {

// G (P x P column-major), wsse and the valid count at x.  scalar: 0 = float, 1 = double.
int orc_score_gram(const orc_cost* c, int scalar, const double* x, double* G, double* wsse, int64_t* n_valid) {
  return scalar ? score_gram_t<double>(c, x, G, wsse, n_valid) : score_gram_t<float>(c, x, G, wsse, n_valid);
}

}  // extern "C"
