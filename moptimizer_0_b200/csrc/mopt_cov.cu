// Parameter covariance: instantiations of the score Gram kernel (mopt_cov.cuh) for the builtin models, and
// mopt_covariance_from_terms, the host-only fp64 finish (Jacobi eigensolver, truncated pseudo-inverse, estimators).
// mopt_covariance_terms itself lives in mopt_capi.cu next to the pass launcher it mirrors.
#include <cmath>
#include <cstring>
#include <type_traits>

#include "mopt_cov.cuh"
#include "mopt_internal.h"

namespace mopt {
namespace {

template <class M, typename ST, typename CT, int JAC>
int gram_kernel(KernelDesc* k) {
  *k = builtin_kernel(reinterpret_cast<const void*>(score_gram_kernel<M, ST, CT, JAC>), kCovThreads);
  return MOPT_OK;
}

// The Jacobian form of the linearization pass of the same problem (launch_pass, launch_dense, launch_wide).
template <class M, typename ST, typename CT>
int gram_form(int form, bool affine_fd, KernelDesc* k) {
  if constexpr (std::is_same_v<M, P2PModel>) {
    if (form == COV_JAC_P2P_AFFINE) return gram_kernel<M, ST, CT, COV_JAC_P2P_AFFINE>(k);
  }
  if (form == COV_JAC_ANALYTICAL) {
    if constexpr (M::HAS_JAC) return gram_kernel<M, ST, CT, COV_JAC_ANALYTICAL>(k);
    set_last_error("this model has no analytical Jacobian");
    return MOPT_ERR_UNSUPPORTED;
  }
  if constexpr (HasAffineStage<M>::value) {
    if (affine_fd) return gram_kernel<M, ST, CT, COV_JAC_AFFINE_FD>(k);
  }
  return gram_kernel<M, ST, CT, COV_JAC_FD>(k);
}

}  // namespace

int score_gram_kernel_desc(int model, int form, bool affine_fd, int store_dtype, int compute_dtype, KernelDesc* k) {
  return with_builtin_model(model, [&](auto m) {
    using M = decltype(m);
    if constexpr (M::P == 0) {
      set_last_error("internal error: no covariance for a model without parameters");
      return MOPT_ERR_CUDA;
    } else {
      return with_dtypes(store_dtype, compute_dtype, [&](auto st, auto ct) {
        return gram_form<M, decltype(st), decltype(ct)>(form, affine_fd, k);
      });
    }
  });
}

// Cyclic Jacobi eigendecomposition of the symmetric n x n matrix A (column-major, overwritten): on return the
// diagonal of A holds the eigenvalues and the columns of V the eigenvectors.  Sweeps until the off-diagonal mass is
// below 1e-30 of the total (fp64 rounding level), at most 100 sweeps.  Also Horn's solve (mopt_align.cu).
void jacobi_eigen(int n, double* A, double* V) {
  auto a = [&](int r, int c) -> double& { return A[r + c * n]; };
  for (int i = 0; i < n * n; ++i) V[i] = (i % (n + 1) == 0) ? 1.0 : 0.0;
  double total = 0.0;
  for (int i = 0; i < n * n; ++i) total += A[i] * A[i];
  for (int sweep = 0; sweep < 100; ++sweep) {
    double off = 0.0;
    for (int c = 0; c < n; ++c)
      for (int r = 0; r < c; ++r) off += a(r, c) * a(r, c);
    if (off <= 1e-30 * total) break;
    for (int p = 0; p < n - 1; ++p)
      for (int q = p + 1; q < n; ++q) {
        const double apq = a(p, q);
        if (apq == 0.0) continue;
        const double theta = (a(q, q) - a(p, p)) / (2.0 * apq);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < n; ++k) {  // A <- A J (columns p, q)
          const double akp = a(k, p), akq = a(k, q);
          a(k, p) = c * akp - s * akq;
          a(k, q) = s * akp + c * akq;
        }
        for (int k = 0; k < n; ++k) {  // A <- J^T A (rows p, q)
          const double apk = a(p, k), aqk = a(q, k);
          a(p, k) = c * apk - s * aqk;
          a(q, k) = s * apk + c * aqk;
        }
        a(p, q) = a(q, p) = 0.0;
        for (int k = 0; k < n; ++k) {
          const double vkp = V[k + p * n], vkq = V[k + q * n];
          V[k + p * n] = c * vkp - s * vkq;
          V[k + q * n] = s * vkp + c * vkq;
        }
      }
  }
}

}  // namespace mopt

extern "C" {

int mopt_covariance_from_terms(const mopt_cov_terms* terms, int estimator, double rcond, double* cov,
                               mopt_cov_report* report) try {
  MOPT_REQUIRE(terms && cov, "null terms or cov");
  const int P = terms->num_parameters;
  MOPT_REQUIRE(P >= 1 && P <= mopt::kMaxP, "num_parameters out of range");
  MOPT_REQUIRE(estimator == MOPT_COV_UNSCALED || estimator == MOPT_COV_SCALED || estimator == MOPT_COV_SANDWICH,
               "unknown estimator");
  MOPT_REQUIRE(rcond >= 0.0, "rcond must not be negative");  // NaN fails too
  MOPT_REQUIRE(terms->n_valid >= 0 && terms->m >= terms->n_valid, "inconsistent element counts");
  bool finite = std::isfinite(terms->wsse) && std::isfinite(terms->sum_sq);
  for (int i = 0; i < P * P; ++i) finite = finite && std::isfinite(terms->H[i]) && std::isfinite(terms->G[i]);
  for (int i = 0; i < P; ++i) finite = finite && std::isfinite(terms->b[i]);
  MOPT_REQUIRE(finite, "the terms are not finite");
  if (rcond == 0.0) rcond = 1e-10;

  // S = D H D with D = diag(H)^(-1/2) (a zero diagonal entry: an unobservable parameter, D = 0)
  double d[mopt::kMaxP], S[mopt::kMaxP * mopt::kMaxP], V[mopt::kMaxP * mopt::kMaxP];
  for (int i = 0; i < P; ++i) {
    const double h = terms->H[i + i * P];
    MOPT_REQUIRE(h >= 0.0, "H has a negative diagonal entry");
    d[i] = h > 0.0 ? 1.0 / std::sqrt(h) : 0.0;
  }
  for (int c = 0; c < P; ++c)
    for (int r = 0; r < P; ++r) S[r + c * P] = d[r] * (0.5 * (terms->H[r + c * P] + terms->H[c + r * P])) * d[c];
  mopt::jacobi_eigen(P, S, V);
  double lmax = 0.0;
  for (int i = 0; i < P; ++i) lmax = std::fmax(lmax, S[i + i * P]);
  int rank = 0;
  double lmin_kept = 0.0, inv[mopt::kMaxP];
  for (int i = 0; i < P; ++i) {
    const double l = S[i + i * P];
    const bool keep = lmax > 0.0 && l > rcond * lmax;
    inv[i] = keep ? 1.0 / l : 0.0;
    if (keep) {
      lmin_kept = (rank == 0) ? l : std::fmin(lmin_kept, l);
      ++rank;
    }
  }
  const int64_t dof = terms->m - rank;
  MOPT_REQUIRE(dof > 0, "no degrees of freedom left (m <= rank)");
  const double sigma2 = terms->wsse / double(dof);

  // H^+ = D V diag(inv) V^T D
  double Hp[mopt::kMaxP * mopt::kMaxP], out[mopt::kMaxP * mopt::kMaxP];
  for (int c = 0; c < P; ++c)
    for (int r = 0; r < P; ++r) {
      double s = 0.0;
      for (int k = 0; k < P; ++k) s += V[r + k * P] * inv[k] * V[c + k * P];
      Hp[r + c * P] = d[r] * s * d[c];
    }
  if (estimator == MOPT_COV_SANDWICH) {
    double T[mopt::kMaxP * mopt::kMaxP];  // T = G H^+
    for (int c = 0; c < P; ++c)
      for (int r = 0; r < P; ++r) {
        double s = 0.0;
        for (int k = 0; k < P; ++k) s += terms->G[r + k * P] * Hp[k + c * P];
        T[r + c * P] = s;
      }
    for (int c = 0; c < P; ++c)
      for (int r = 0; r < P; ++r) {
        double s = 0.0;
        for (int k = 0; k < P; ++k) s += Hp[r + k * P] * T[k + c * P];
        out[r + c * P] = s;
      }
    for (int c = 0; c < P; ++c)  // symmetric up to rounding: make it exactly so
      for (int r = 0; r < c; ++r) out[r + c * P] = out[c + r * P] = 0.5 * (out[r + c * P] + out[c + r * P]);
  } else {
    const double f = (estimator == MOPT_COV_SCALED) ? sigma2 : 1.0;
    for (int i = 0; i < P * P; ++i) out[i] = f * Hp[i];
  }
  std::memcpy(cov, out, sizeof(double) * size_t(P) * P);
  if (report) {
    std::memset(report, 0, sizeof(*report));
    report->rank = rank;
    report->dof = dof;
    report->sigma2 = sigma2;
    report->eig_min = lmin_kept;
    report->eig_max = lmax;
  }
  return MOPT_OK;
}
MOPT_ABI_CATCH

}  // extern "C"
