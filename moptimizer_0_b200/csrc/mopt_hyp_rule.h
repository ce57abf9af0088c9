// The fp32 form of mopt_evaluate's inlier test (mopt_score_hypotheses).  For a float e2, double(e2) <= thr2 holds
// exactly when e2 <= f, f the largest float not above thr2: the test then needs no conversion of e2.  That holds for
// every thr2 the host forms, 0, subnormal, above FLT_MAX (f = FLT_MAX) and +inf (f = +inf), and for NaN (f = NaN:
// both tests are false).  Plain C++: the CPU tests compile it with the host compiler alone.
#pragma once

#include <cfloat>
#include <cmath>

namespace mopt {

inline float largest_float_le(double thr2) {
  if (thr2 > static_cast<double>(FLT_MAX)) return thr2 == INFINITY ? INFINITY : FLT_MAX;
  float f = static_cast<float>(thr2);  // round to nearest: at most one float above thr2
  if (static_cast<double>(f) > thr2) f = std::nextafter(f, -INFINITY);
  return f;
}

}  // namespace mopt
