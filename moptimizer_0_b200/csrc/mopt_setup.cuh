// Device-side `model->setup(x)` (include/moptimizer/model.h:19-22) for the builtin models and
// for every finite-difference perturbation of x (linearization.h:78-95): turns the parameter
// vector into the small constant block the pass kernels consume.  Runs on one warp, in fp64,
// either as its own tiny kernel (host-driven linearize) or inside the LM step kernel.
#pragma once

#include "mopt_common.cuh"

namespace mopt {

// src/so3.cpp:43-57 — Rodrigues, guard `norm > 10 eps`.  R row-major.  S names the cost's compute Scalar.
// The arithmetic here is fp64 for either S, so the guard is the fp64 one for both: the float threshold (1.2e-6)
// makes R = I on a whole ball of rotation vectors, where every finite-difference column of the rotation block is
// exactly zero — LM started at omega = 0 with a heavily damped first step (lambda_0 grows with N,
// levenberg_marquadt_dyn.cpp:9,62-66) lands inside that ball and can never leave it (observed: camera, 50 M
// observations, fp32 compute).  Inside the ball R differs from I by < 1.2e-6, i.e. below float resolution, so
// values computed with a float Scalar are unaffected.
// MOPT_FLAG_REFERENCE_FLOAT_GUARD restores the reference's float threshold (CostDev::so3_guard = 10 eps_f32) for
// callers that need the literal behaviour of the float instantiation.
constexpr double kSo3GuardF64 = 10.0 * 2.220446049250313e-16;
constexpr double kSo3GuardF32 = 10.0 * 1.1920928955078125e-07;
// The roundings of so3::Exp and of the left Jacobian are spelled out (intrinsics, no compiler-chosen contraction):
// the same values come out of the serial forms below (fused into the pass kernels, finite-difference set-ups) and of
// the warp-parallel form of the optimizer step (so3_exp_jl_warp), wherever they are inlined.
__device__ inline double so3_norm2_dev(const double w[3]) {
  return __fma_rn(w[2], w[2], __fma_rn(w[1], w[1], __dmul_rn(w[0], w[0])));
}
// hat(v)(i, j): [[0, -v2, v1], [v2, 0, -v0], [-v1, v0, 0]], for run-time or compile-time (i, j)
__device__ inline double so3_hat_entry(const double v[3], int i, int j) {
  if (i == j) return 0.0;
  const int k = 3 - i - j;
  const double x = k == 0 ? v[0] : (k == 1 ? v[1] : v[2]);
  return ((j - i + 3) % 3 == 1) ? -x : x;
}
// (K^2)(r, c) for K = hat(v)
__device__ inline double so3_hat2_entry(const double v[3], int r, int c) {
  return __fma_rn(so3_hat_entry(v, r, 2), so3_hat_entry(v, 2, c),
                  __fma_rn(so3_hat_entry(v, r, 1), so3_hat_entry(v, 1, c),
                           __dmul_rn(so3_hat_entry(v, r, 0), so3_hat_entry(v, 0, c))));
}
// R = I + sin(n) K + (1 - cos(n)) K^2, K = hat(axis): entry (r, c)
__device__ inline double so3_exp_entry(const double a[3], double sn, double cs, int r, int c) {
  const double omc = __dsub_rn(1.0, cs);
  return __dadd_rn(r == c ? 1.0 : 0.0, __fma_rn(sn, so3_hat_entry(a, r, c), __dmul_rn(omc, so3_hat2_entry(a, r, c))));
}
// J = I + A [w]x + B [w]x^2: entry (r, c)
__device__ inline double so3_left_jacobian_entry(const double w[3], double A, double B, int r, int c) {
  return __fma_rn(B, so3_hat2_entry(w, r, c), __fma_rn(A, so3_hat_entry(w, r, c), r == c ? 1.0 : 0.0));
}
__device__ inline void so3_exp_entries(const double a[3], double sn, double cs, double R[9]) {
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) R[r * 3 + c] = so3_exp_entry(a, sn, cs, r, c);
}
__device__ inline void so3_left_jacobian_entries(const double w[3], double A, double B, double J[9]) {
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) J[r * 3 + c] = so3_left_jacobian_entry(w, A, B, r, c);
}

template <typename S>
__device__ inline void so3_exp_dev(const double w[3], double R[9], double guard = kSo3GuardF64) {
  const double n = sqrt(so3_norm2_dev(w));
#pragma unroll
  for (int i = 0; i < 9; ++i) R[i] = (i % 4 == 0) ? 1.0 : 0.0;
  if (n > guard) {
    const double a[3] = {w[0] / n, w[1] / n, w[2] / n};
    double sn, cs;
    sincos(n, &sn, &cs);
    so3_exp_entries(a, sn, cs, R);
  }
}

// Closed-form left Jacobian of SO(3): I + (1-cos)/th^2 [w]x + (th-sin)/th^3 [w]x^2.
__device__ inline void so3_left_jacobian_dev(const double w[3], double J[9]) {
  const double th2 = so3_norm2_dev(w);
  const double th = sqrt(th2);
  double A, B;
  if (th2 < 1e-8) {
    A = __dsub_rn(0.5, th2 / 24.0);
    B = __dsub_rn(1.0 / 6.0, th2 / 120.0);
  } else {
    double sn, cs;
    sincos(th, &sn, &cs);
    A = __dsub_rn(1.0, cs) / th2;
    B = __dsub_rn(th, sn) / __dmul_rn(th2, th);
  }
  so3_left_jacobian_entries(w, A, B, J);
}

// so3::Exp(w) and, if want_jl, J_l(wj) together, by one full warp: the two square roots are ONE instruction sequence
// (lane 0: |w|, lane 1: |wj|), likewise the two sincos and the five divisions (lanes 0-2: the axis, lanes 3-4: the
// two Jacobian coefficients); the entries every lane forms for itself (one entry per lane with run-time indices was
// measured slower: 5 200 against 3 700 cycles to the point where R is complete).  Same operations on the same values
// as so3_exp_dev / so3_left_jacobian_dev (bit-identical results); the dependent chain is sqrt -> sincos -> division
// instead of sqrt -> 3 divisions -> sincos -> sqrt -> sincos -> 2 divisions.
// R is complete on return; the Jacobian is left as its two coefficients (so3_left_jacobian_entries(wj, A, B, J) forms it)
// so that a caller with someone waiting for R can hand it over first.
__device__ inline void so3_exp_jl_warp(const double w[3], const double wj[3], double guard, int lane, double R[9],
                                       double& A, double& B) {
  const unsigned full = 0xffffffffu;
  const double n2 = so3_norm2_dev(w), th2 = so3_norm2_dev(wj);
  const double rt = sqrt(lane == 1 ? th2 : n2);
  const double n = __shfl_sync(full, rt, 0), th = __shfl_sync(full, rt, 1);
  double s_, c_;
  sincos(lane == 1 ? th : n, &s_, &c_);
  const double sn = __shfl_sync(full, s_, 0), cs = __shfl_sync(full, c_, 0);
  const double snj = __shfl_sync(full, s_, 1), csj = __shfl_sync(full, c_, 1);
  const bool small = th2 < 1e-8;
  double num = 1.0, den = 1.0;
  if (lane < 3) { num = lane == 0 ? w[0] : (lane == 1 ? w[1] : w[2]); den = n; }
  else if (lane == 3) { num = small ? th2 : __dsub_rn(1.0, csj); den = small ? 24.0 : th2; }
  else if (lane == 4) { num = small ? th2 : __dsub_rn(th, snj); den = small ? 120.0 : __dmul_rn(th2, th); }
  const double q = num / den;
  const double a[3] = {__shfl_sync(full, q, 0), __shfl_sync(full, q, 1), __shfl_sync(full, q, 2)};
  const double q3 = __shfl_sync(full, q, 3), q4 = __shfl_sync(full, q, 4);
#pragma unroll
  for (int i = 0; i < 9; ++i) R[i] = (i % 4 == 0) ? 1.0 : 0.0;
  if (n > guard) so3_exp_entries(a, sn, cs, R);
  A = small ? __dsub_rn(0.5, q3) : q3;
  B = small ? __dsub_rn(1.0 / 6.0, q4) : q4;
}

// Persistent LM kernel: (R, t) of the next pass travels to the data CTAs in 24 self-validating 8-byte words — word
// 2 i carries the low half and word 2 i + 1 the high half of value i (R row-major, then t) in its upper 32 bits, and
// every word carries the same tag in its lower 32 bits: ((barrier target) << 2 | PassMode) truncated to 32 bits.
// An 8-byte store is single-copy atomic, so a reader that finds the expected tag in a word has that word of THIS
// publication: no fence on either side, and the wait for the optimizer and the load of (R, t) are one L2 round trip.
__device__ inline void publish_rt(unsigned long long* words, unsigned long long value, double v, int lane) {
  if (lane < 24) {
    const unsigned half = (lane & 1) ? unsigned(__double2hiint(v)) : unsigned(__double2loint(v));
    const unsigned long long wv = ((unsigned long long)(half) << 32) | (value & 0xffffffffull);
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(words + lane), "l"(wv) : "memory");
  }
}

// src/so3.cpp:96-105 — so3::Log as the reference defines it (first-order branch below theta = 1e-3).
__device__ inline void so3_log_dev(const double R[9], double w[3]) {
  const double tr = R[0] + R[4] + R[8];
  const double theta = (tr > 3.0 - 1e-6) ? 0.0 : acos(0.5 * (tr - 1.0));
  const double K[3] = {R[7] - R[5], R[2] - R[6], R[3] - R[1]};
  const double f = (fabs(theta) < 0.001) ? 0.5 : 0.5 * theta / sin(theta);
  for (int i = 0; i < 3; ++i) w[i] = f * K[i];
}

// x (+) delta.  Additive everywhere (levenberg_marquadt_dyn.cpp:83) except, with MOPT_MANIFOLD_SO3_LEFT, on
// the rotation-vector block: omega <- Log(Exp(delta_omega) Exp(omega)).  `f32` rounds like the float Scalar.
__device__ inline void retract_dev(const CostDev& c, const double* x, const double* delta, double* out, bool f32) {
  for (int i = 0; i < c.P; ++i) out[i] = f32 ? double(float(x[i]) + float(delta[i])) : x[i] + delta[i];
  if (c.manifold == MOPT_MANIFOLD_SO3_LEFT && c.rot_offset >= 0) {
    const int o = c.rot_offset;
    double Rx[9], Rd[9], Rn[9];
    if (f32) { so3_exp_dev<float>(x + o, Rx, c.so3_guard); so3_exp_dev<float>(delta + o, Rd, c.so3_guard); }
    else { so3_exp_dev<double>(x + o, Rx, c.so3_guard); so3_exp_dev<double>(delta + o, Rd, c.so3_guard); }
    for (int r = 0; r < 3; ++r)
      for (int col = 0; col < 3; ++col) {
        double s = 0.0;
        for (int k = 0; k < 3; ++k) s += Rd[r * 3 + k] * Rx[k * 3 + col];
        Rn[r * 3 + col] = s;
      }
    double w[3];
    so3_log_dev(Rn, w);
    for (int i = 0; i < 3; ++i) out[o + i] = f32 ? double(float(w[i])) : w[i];
  }
}

// One parameter set for model `c.model` at parameters xs[0..P).
__device__ inline void setup_one_set(const CostDev& c, const double* xs, double* set) {
  for (int i = 0; i < kSetSize; ++i) set[i] = 0.0;
  switch (c.model) {
    case MOPT_MODEL_POINT2POINT: {
      // so3::convert6DOFParameterToMatrix, src/so3.cpp:7-19: x = [t, omega]
      const double w[3] = {xs[3], xs[4], xs[5]};
      if (c.compute_dtype == MOPT_F32) so3_exp_dev<float>(w, set, c.so3_guard); else so3_exp_dev<double>(w, set, c.so3_guard);
      set[9] = xs[0]; set[10] = xs[1]; set[11] = xs[2];
      break;
    }
    case MOPT_MODEL_PINHOLE: {
      // tst/camera_calibration.cpp:33,37: M = (K * T(x)) * C, 3x4 row-major
      double R[9];
      const double w[3] = {xs[3], xs[4], xs[5]};
      if (c.compute_dtype == MOPT_F32) so3_exp_dev<float>(w, R, c.so3_guard); else so3_exp_dev<double>(w, R, c.so3_guard);
      double T[16];
      for (int r = 0; r < 3; ++r) {
        for (int k = 0; k < 3; ++k) T[r * 4 + k] = R[r * 3 + k];
        T[r * 4 + 3] = xs[r];
      }
      T[12] = T[13] = T[14] = 0.0; T[15] = 1.0;
      const double* K = c.consts;
      const double* C = c.consts + 12;
      double KT[12];
      for (int r = 0; r < 3; ++r)
        for (int col = 0; col < 4; ++col) {
          double s = 0.0;
          for (int k = 0; k < 4; ++k) s += K[r * 4 + k] * T[k * 4 + col];
          KT[r * 4 + col] = s;
        }
      for (int r = 0; r < 3; ++r)
        for (int col = 0; col < 4; ++col) {
          double s = 0.0;
          for (int k = 0; k < 4; ++k) s += KT[r * 4 + k] * C[k * 4 + col];
          set[r * 4 + col] = s;
        }
      break;
    }
    case MOPT_MODEL_PINHOLE_DISTORT: {
      // set = (T(x) C)(3x4 row-major, 12), fx, fy, cx, cy, k1, k2, p1, p2, k3
      double R[9];
      const double w[3] = {xs[3], xs[4], xs[5]};
      if (c.compute_dtype == MOPT_F32) so3_exp_dev<float>(w, R, c.so3_guard); else so3_exp_dev<double>(w, R, c.so3_guard);
      const double* C = c.consts;
      for (int r = 0; r < 3; ++r)
        for (int col = 0; col < 4; ++col) {
          double s = 0.0;
          for (int k = 0; k < 3; ++k) s += R[r * 3 + k] * C[k * 4 + col];
          s += xs[r] * C[12 + col];
          set[r * 4 + col] = s;
        }
      for (int i = 0; i < 9; ++i) set[12 + i] = xs[6 + i];
      break;
    }
    default:  // parameter-only models: the set is x itself
#ifdef MOPT_USER_SETUP
      // run-time compiled user model with its own setup(x) (mopt_rtc.cu; model.h:19-22)
      if (c.model >= MOPT_MODEL_USER_BASE) {
        ::mopt_setup(xs, c.consts, set);
        break;
      }
#endif
      for (int i = 0; i < c.P; ++i) set[i] = xs[i];
      break;
  }
}

// x as the compute Scalar holds it (linearization.h:78-89 with a float Scalar rounds every coordinate).
__device__ inline void scalar_x(const CostDev& c, const double* x, double* xs) {
  const bool f32 = (c.compute_dtype == MOPT_F32);
  for (int i = 0; i < c.P; ++i) xs[i] = f32 ? double(float(x[i])) : x[i];
}

// Set 0 of setup_cost at x: the set every residual of a cost evaluation (mopt_evaluate) is formed from.
__device__ inline void setup_base_set(const CostDev& c, const double* x, double* set) {
  double xs[kMaxP];
  scalar_x(c, x, xs);
  setup_one_set(c, xs, set);
}

// Set 0 of n parameter vectors (mopt_score_hypotheses), one thread each: xs is [n][kMaxP], sets is [n][kSetSize].
__device__ inline void setup_hypotheses(const CostDev& c, const double* xs, int n, double* sets) {
  const int k = int(blockIdx.x * blockDim.x + threadIdx.x);
  if (k < n) setup_base_set(c, xs + size_t(k) * kMaxP, sets + size_t(k) * kSetSize);
}

// Affine decomposition of the point2point analytical Jacobian, J(q) = J0 + q_x J1 + q_y J2 + q_z J3
// (each 3x6 row-major), for the three variants of mopt_p2p_variant.
__device__ inline void setup_p2p_affine(const CostDev& c, const double* x, double jaff[4][18]) {
  double Jl[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  if (c.variant == MOPT_P2P_EXACT) {
    const double w[3] = {x[3], x[4], x[5]};
    so3_left_jacobian_dev(w, Jl);
  }
  // -[q]x = q_x E1 + q_y E2 + q_z E3
  const double E[3][9] = {{0, 0, 0, 0, 0, 1, 0, -1, 0}, {0, 0, -1, 0, 0, 0, 1, 0, 0}, {0, 1, 0, -1, 0, 0, 0, 0, 0}};
  double tru[4][18];
  for (int k = 0; k < 4; ++k)
    for (int i = 0; i < 18; ++i) tru[k][i] = 0.0;
  for (int r = 0; r < 3; ++r) tru[0][r * 6 + r] = 1.0;
  for (int k = 0; k < 3; ++k)
    for (int r = 0; r < 3; ++r)
      for (int col = 0; col < 3; ++col) {
        double s = 0.0;
        for (int m = 0; m < 3; ++m) s += E[k][r * 3 + m] * Jl[m * 3 + col];
        tru[k + 1][r * 6 + 3 + col] = s;
      }
  for (int k = 0; k < 4; ++k)
    for (int idx = 0; idx < 18; ++idx) {
      if (c.variant == MOPT_P2P_REFTEST_COLMAJOR) {
        // tst/point2point.cpp:18,71: Map<Matrix<S,3,6>> is column-major, so true element (r,c) was
        // written at buffer[c*3+r]; linearization.h:17-18 then reads buffer[r'*6+c'] as J(r',c').
        const int cc = idx / 3, rr = idx % 3;
        jaff[k][idx] = tru[k][rr * 6 + cc];
      } else {
        jaff[k][idx] = tru[k][idx];
      }
    }
}

// Whole ParamBlock for one cost at x.  Call with at least one full warp; lane j builds set j.
// Emulates the reference's Scalar for the step: with compute_dtype F32 x_j, h_j and x_j +- h_j are
// rounded to float exactly as `float` arithmetic would (linearization.h:78-89).
// `scratch` (optional, >= 9 doubles of shared memory): enables the warp-parallel fast path of the analytical
// point2point model below.
// Persistent LM kernel: where the next pass's (R, t) is published (publish_rt) and the tag that releases the CTAs
// waiting for it.  A set-up that can tell when the pass's own inputs are complete publishes there (and sets *opened);
// otherwise the caller does after the set-up.
struct SetupEarlyOpen {
  unsigned long long* rt_words;
  unsigned long long value;  // (barrier target << 2) | PassMode
  int* opened;  // shared memory
};
__device__ inline void setup_p2p_analytical_warp(const CostDev& c, const double* x, ParamBlock* pb, int lane, double* Jl,
                                                 const SetupEarlyOpen* early);
__device__ inline void setup_cost(const CostDev& c, const double* x, ParamBlock* pb, int lane, int nlanes,
                                  double* scratch = nullptr, const SetupEarlyOpen* early = nullptr) {
  if (scratch != nullptr && nlanes == 32 && c.model == MOPT_MODEL_POINT2POINT && c.jacobian == MOPT_JAC_ANALYTICAL) {
    setup_p2p_analytical_warp(c, x, pb, lane, scratch, early);
    return;
  }
  const int P = c.P;
  const bool f32 = (c.compute_dtype == MOPT_F32);
  const int nsets = (c.jacobian == MOPT_JAC_ANALYTICAL) ? 1 : (c.jacobian == MOPT_JAC_FORWARD ? 1 + P : 1 + 2 * P);
  for (int s = lane; s < nsets; s += nlanes) {
    if (s == 0) {  // the unperturbed set: the one every cost evaluation and hypothesis score reads
      setup_base_set(c, x, pb->sets[0]);
      continue;
    }
    double xs[kMaxP];
    scalar_x(c, x, xs);
    const int j = (s - 1) % P;
    const bool minus = (s - 1) >= P;
    double h;
    double step_fwd, step_cen;  // the steps actually taken (see ParamBlock::hstep_*)
    if (f32) {
      const float ms = sqrtf(1.1920928955078125e-07f);
      float hf = ms * fabsf(float(x[j]));
      if (hf == 0.0f) hf = ms;
      h = double(hf);
      const float xpl = float(x[j]) + hf, xmi = float(x[j]) - hf;
      xs[j] = double(minus ? xmi : xpl);
      step_fwd = double(xpl) - double(float(x[j]));
      step_cen = double(xpl) - double(xmi);
    } else {
      const double ms = sqrt(2.220446049250313e-16);
      h = ms * fabs(x[j]);
      if (h == 0.0) h = ms;
      xs[j] = minus ? x[j] - h : x[j] + h;
      step_fwd = (x[j] + h) - x[j];
      step_cen = (x[j] + h) - (x[j] - h);
    }
    if (c.manifold == MOPT_MANIFOLD_SO3_LEFT && c.rot_offset >= 0 && j >= c.rot_offset && j < c.rot_offset + 3) {
      // tangent coordinate of the rotation block is 0 at x, so the reference's rule (:85-87) gives h = sqrt(eps)
      h = f32 ? double(sqrtf(1.1920928955078125e-07f)) : sqrt(2.220446049250313e-16);
      double d[kMaxP];
      for (int i = 0; i < P; ++i) d[i] = 0.0;
      d[j] = minus ? -h : h;
      double base[kMaxP];
      for (int i = 0; i < P; ++i) base[i] = f32 ? double(float(x[i])) : x[i];
      retract_dev(c, base, d, xs, f32);
      step_fwd = h;  // the tangent-space step is not a coordinate difference of x
      step_cen = 2.0 * h;
    }
    if (!minus) {
      pb->h[j] = h;
      pb->hstep_fwd[j] = step_fwd;
      pb->hstep_cen[j] = step_cen;
    }
    setup_one_set(c, xs, pb->sets[s]);
  }
  __syncwarp();  // the sets written by the other lanes are read below
  if (lane == 0) {
    for (int i = 0; i < P; ++i) pb->x[i] = x[i];
    if (c.model == MOPT_MODEL_POINT2POINT && c.jacobian == MOPT_JAC_ANALYTICAL) setup_p2p_affine(c, x, pb->jaff);
    if (c.model == MOPT_MODEL_POINT2POINT && c.jacobian != MOPT_JAC_ANALYTICAL) {
      // r = R p + t - y is affine in p, so the finite-difference Jacobian of linearization.h:97-111 is too:
      //   (r(x + h_j e_j) - r(x)) / h_j = ((R_j - R) p + (t_j - t)) / h_j        (central: +- sets, 2 h_j)
      // which lets the numerical linearization run on the moment kernel (q = p) at the analytical kernel's cost.
      const bool central = (c.jacobian == MOPT_JAC_CENTRAL);
      for (int k = 0; k < 4; ++k)
        for (int i = 0; i < 18; ++i) pb->jaff[k][i] = 0.0;
      for (int j = 0; j < P; ++j) {
        const double* sp = pb->sets[1 + j];
        const double* sm = central ? pb->sets[1 + P + j] : pb->sets[0];
        const double inv = 1.0 / (central ? 2.0 * pb->h[j] : pb->h[j]);
        for (int r = 0; r < 3; ++r) {
          const double dt = f32 ? double(float(sp[9 + r])) - double(float(sm[9 + r])) : sp[9 + r] - sm[9 + r];
          pb->jaff[0][r * 6 + j] = dt * inv;
          for (int k = 0; k < 3; ++k) {
            const double dr = f32 ? double(float(sp[r * 3 + k])) - double(float(sm[r * 3 + k])) : sp[r * 3 + k] - sm[r * 3 + k];
            pb->jaff[k + 1][r * 6 + j] = dr * inv;
          }
        }
      }
    }
  }
}

// One entry of J(q) = J0 + q_x J1 + q_y J2 + q_z J3 (setup_p2p_affine above, same sums in the same order).
__device__ inline double p2p_affine_entry(int variant, const double* Jl, int k, int idx) {
  int r = idx / 6, col = idx % 6;
  if (variant == MOPT_P2P_REFTEST_COLMAJOR) {  // tst/point2point.cpp:18,71 (see setup_p2p_affine)
    const int cc = idx / 3, rr = idx % 3;
    r = rr; col = cc;
  }
  if (k == 0) return (col < 3 && r == col) ? 1.0 : 0.0;
  if (col < 3) return 0.0;
  const double E[3][9] = {{0, 0, 0, 0, 0, 1, 0, -1, 0}, {0, 0, -1, 0, 0, 0, 1, 0, 0}, {0, 1, 0, -1, 0, 0, 0, 0, 0}};
  double s = 0.0;
  for (int m = 0; m < 3; ++m) s += E[k - 1][r * 3 + m] * Jl[m * 3 + (col - 3)];
  return s;
}

// setup_cost for the analytical point2point model, spread over one warp: lane 0 derives (R, t) and J_l(omega) exactly
// as setup_one_set / setup_p2p_affine do, then the 72 affine Jacobian entries are formed one per lane (the generic
// path runs ~1 500 serial instructions on lane 0 for this; the optimizer step of a small problem waits on it).
__device__ inline void setup_p2p_analytical_warp(const CostDev& c, const double* x, ParamBlock* pb, int lane, double* Jl,
                                                 const SetupEarlyOpen* early) {
  const bool f32 = (c.compute_dtype == MOPT_F32);
  double xs[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) xs[i] = f32 ? double(float(x[i])) : x[i];
  const double w[3] = {xs[3], xs[4], xs[5]};
  const double wj[3] = {x[3], x[4], x[5]};  // the Jacobian takes omega with a double Scalar
  double R[9], J[9], A, B;
  so3_exp_jl_warp(w, wj, c.so3_guard, lane, R, A, B);
  // The pass needs (R, t) when it starts and the Jacobian pieces only when its result is assembled: the persistent LM
  // kernel releases the data CTAs here, before anything else of the set-up is stored.
  if (early && early->rt_words) {
    const int idx = lane >> 1;
    double v = R[0];
#pragma unroll
    for (int i = 1; i < 9; ++i) v = (idx == i) ? R[i] : v;
    v = (idx == 9) ? xs[0] : (idx == 10 ? xs[1] : (idx == 11 ? xs[2] : v));
    publish_rt(early->rt_words, early->value, v, lane);
    if (lane == 0) *early->opened = 1;
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) J[i] = (i % 4 == 0) ? 1.0 : 0.0;
  if (c.variant == MOPT_P2P_EXACT) so3_left_jacobian_entries(wj, A, B, J);
  if (lane < 9) {
    double v = R[0];
#pragma unroll
    for (int i = 1; i < 9; ++i) v = (lane == i) ? R[i] : v;
    pb->sets[0][lane] = v;
    double j = J[0];
#pragma unroll
    for (int i = 1; i < 9; ++i) j = (lane == i) ? J[i] : j;
    Jl[lane] = j;
  } else if (lane < 12) {
    pb->sets[0][lane] = lane == 9 ? xs[0] : (lane == 10 ? xs[1] : xs[2]);
  } else if (lane < kSetSize) {
    pb->sets[0][lane] = 0.0;
  }
  if (lane < c.P) pb->x[lane] = x[lane];
  __syncwarp();
  for (int i = lane; i < 4 * 18; i += 32) pb->jaff[i / 18][i % 18] = p2p_affine_entry(c.variant, Jl, i / 18, i % 18);
  __syncwarp();
}

}  // namespace mopt
