// The order statistics a quantile level selects and numpy's method="linear" interpolation between them
// (mopt_residual_quantiles).  Shared by the device step of the radix select (which ranks to select) and the host
// (which ranks belong to which q, and the interpolated value), so that both agree bit for bit.  Plain C++: the CPU
// tests compile it with the host compiler alone.
#pragma once

#include <stdint.h>

#include <cmath>

#if defined(__CUDACC__)
#define MOPT_QUANT_HD __host__ __device__
#else
#define MOPT_QUANT_HD
#endif

namespace mopt {

// numpy's virtual index for method="linear": h = (n - 1) q in fp64, j = floor(h), hi index j + 1 clamped to n - 1.
struct QuantRank {
  int64_t j, j1;
  double t;  // h - j: the interpolation weight
};

MOPT_QUANT_HD inline QuantRank quantile_rank(int64_t n, double q) {
  const double h = double(n - 1) * q;  // one rounded product, as numpy forms it
  QuantRank r;
  r.j = int64_t(floor(h));
  r.t = h - double(r.j);
  r.j1 = r.j + 1 < n ? r.j + 1 : n - 1;
  return r;
}

// numpy's _lerp(a, b, t) with every product and sum rounded separately (volatile: no contraction into an FMA on
// hosts that have one); value = lo at t = 0, where numpy gives NaN for a finite lo next to hi = +inf.
inline double quantile_lerp(double lo, double hi, double t) {
  if (t == 0.0) return lo;
  const volatile double diff = hi - lo;
  if (t >= 0.5) {
    const volatile double p = diff * (1.0 - t);
    return hi - p;
  }
  const volatile double p = diff * t;
  return lo + p;
}

// Median of the chi-square distribution with `dof` degrees of freedom (scipy.stats.chi2.median), dof = 1 .. 4.
inline double chi2_median(int dof) {
  static const double m[4] = {0.454936423119572, 1.386294361119891, 2.3659738843753377, 3.3566939800333224};
  return (dof >= 1 && dof <= 4) ? m[dof - 1] : NAN;
}

}  // namespace mopt
