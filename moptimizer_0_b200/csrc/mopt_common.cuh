// Shared device/host helpers for the sm_100a linearization kernels.
#pragma once

// This header is also compiled at run time by NVRTC (mopt_rtc.cu: user-defined device models), where no
// host headers exist: everything host-only sits behind !__CUDACC_RTC__.
#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>
#include <exception>
#include <new>
#include <string>
#else
typedef int int32_t;
typedef unsigned int uint32_t;
typedef long long int64_t;
typedef unsigned long long uint64_t;
#endif

#include "mopt_capi.h"

namespace mopt {

#ifndef __CUDACC_RTC__
// ------------------------------------------------------------------ errors ----
void set_last_error(const std::string& msg);

#define MOPT_CUDA_TRY(expr)                                                                  \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      (void)cudaGetLastError(); /* reported here: must not resurface in a later launch check */ \
      ::mopt::set_last_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e) +     \
                             " (" __FILE__ ":" + std::to_string(__LINE__) + ")");            \
      return (_e == cudaErrorMemoryAllocation) ? MOPT_ERR_OUT_OF_MEMORY : MOPT_ERR_CUDA;     \
    }                                                                                        \
  } while (0)

#define MOPT_REQUIRE(cond, msg)                                                  \
  do {                                                                           \
    if (!(cond)) {                                                               \
      ::mopt::set_last_error(std::string("invalid argument: ") + (msg));         \
      return MOPT_ERR_INVALID_ARGUMENT;                                          \
    }                                                                            \
  } while (0)

// No C++ exception may cross the C ABI: every `int mopt_*` entry point is a function-try-block closed by this.
#define MOPT_ABI_CATCH                                                        \
  catch (const std::bad_alloc&) {                                             \
    ::mopt::set_last_error("out of host memory");                             \
    return MOPT_ERR_OUT_OF_MEMORY;                                            \
  }                                                                           \
  catch (const std::exception& e) {                                           \
    ::mopt::set_last_error(std::string("internal error: ") + e.what());       \
    return MOPT_ERR_INVALID_ARGUMENT;                                         \
  }                                                                           \
  catch (...) {                                                               \
    ::mopt::set_last_error("internal error: unknown exception");              \
    return MOPT_ERR_INVALID_ARGUMENT;                                         \
  }

#define MOPT_TRY(expr)              \
  do {                              \
    int _s = (expr);                \
    if (_s != MOPT_OK) return _s;   \
  } while (0)
#endif  // !__CUDACC_RTC__

// --------------------------------------------------------------- constants ----
constexpr int kMaxP = MOPT_MAX_PARAMETERS;
constexpr int kMaxO = MOPT_MAX_OUTPUTS;
constexpr int kMaxStreams = 6;
constexpr int kSetSize = 24;                 // doubles per model parameter set
constexpr int kMaxRaw = 160;                 // raw sums a pass kernel may reduce (multiple of 32, >= kPackedMax)
constexpr int kMaxSets = 1 + 2 * kMaxP;      // base, P plus, P minus
constexpr int kPackedMax = kMaxP * (kMaxP + 1) / 2 + kMaxP + 1;  // packed (H upper, b, sum)
constexpr int kMaxGrid = 148 * 8;

// Pass modes (device-side control word read by every pass kernel).
enum PassMode : int { PASS_SKIP = 0, PASS_LINEARIZE = 1, PASS_COST = 2 };

// ---------------------------------------------------------------- POD types ----
// Result of model->setup(x) for x and for each finite-difference perturbation
// (linearization.h:81-95), produced on the device by mopt_setup.cuh.
struct ParamBlock {
  double x[kMaxP];
  double h[kMaxP];                    // finite-difference steps (linearization.h:85-87)
  double sets[kMaxSets][kSetSize];    // [0] base, [1+j] x + h_j e_j, [1+P+j] x - h_j e_j
  double jaff[4][18];                 // point2point analytical J(q) = J0 + q_x J1 + q_y J2 + q_z J3 (3x6 row-major)
  // Steps actually taken after rounding in the compute Scalar: (x_j + h_j) - x_j and (x_j + h_j) - (x_j - h_j).
  // With a float Scalar they differ from h_j, 2 h_j by up to eps_f32 |x_j| / h_j ~ 1e-4 relative, which the
  // reference's float quotient (it divides by the nominal h_j, linearization.h:105) inherits as a per-column scale
  // error; the AFFINE_FD kernels divide by the step taken.
  double hstep_fwd[kMaxP];
  double hstep_cen[kMaxP];
};

// Per-cost constants that live on the device (copied once per call).
struct CostDev {
  int model, variant, P, O;
  int jacobian, loss, has_cov, compute_dtype;
  double loss_param;
  double cov[kMaxO * kMaxO];  // column-major O x O
  double consts[32];
  int manifold;    // mopt_manifold
  int rot_offset;  // index of the rotation-vector block of x, or -1
  double so3_guard;  // so3::Exp returns I for |omega| <= so3_guard (src/so3.cpp:47: 10 eps of the Scalar; see mopt_setup.cuh)
};

// One cost term on the device: its constants and the result of setup(x).
struct CostSlot {
  CostDev cost;
  ParamBlock pb;
};

// A parameter vector passed by value as a kernel argument (no staging buffer for asynchronous calls).
struct XArg {
  double v[kMaxP];
};

// Packed result of one pass: H upper triangle (row-major, P(P+1)/2), then b (P), then sum.
struct PassResult {
  double v[kPackedMax];
};

__host__ __device__ inline int packed_size(int P) { return P * (P + 1) / 2 + P + 1; }
__host__ __device__ inline int tri_index(int P, int r, int c) {  // r <= c
  return r * P - r * (r - 1) / 2 + (c - r);
}

// Planar device streams of one store (dtype is a kernel template parameter).
struct StreamPtrs {
  const void* p[kMaxStreams];
};

// -------------------------------------------------------------- warp utils ----
#ifdef __CUDACC__

template <typename T>
__device__ __forceinline__ T shfl_xor(T v, int off) {
  return __shfl_xor_sync(0xffffffffu, v, off);
}

// Transposing warp reduction: every lane holds V partial sums v[0..V); on return lane l holds the
// warp total of element (l >> (5 - log2 V)) (for V == 32: element l).  V-1 + (5 - log2 V) shuffles
// instead of 5 V.  V must be a power of two <= 32.  Order of additions is fixed => deterministic.
template <int V, typename T>
__device__ __forceinline__ T warp_reduce_transpose(T (&v)[V]) {
  static_assert(V >= 1 && V <= 32 && (V & (V - 1)) == 0, "V must be a power of two <= 32");
  const int lane = threadIdx.x & 31;
  int off = 16;
#pragma unroll
  for (int cnt = V; cnt > 1; cnt >>= 1) {
    const bool up = (lane & off) != 0;
    const int half = cnt >> 1;
#pragma unroll
    for (int k = 0; k < half; ++k) {
      const T keep = up ? v[k + half] : v[k];
      const T send = up ? v[k] : v[k + half];
      v[k] = keep + shfl_xor(send, off);
    }
    off >>= 1;
  }
  T r = v[0];
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    if (o <= off) r += shfl_xor(r, o);
  }
  return r;
}

template <int V>
struct Log2 {
  static constexpr int value = 1 + Log2<V / 2>::value;
};
template <>
struct Log2<1> {
  static constexpr int value = 0;
};

__host__ __device__ constexpr int next_pow2(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// Streaming (read-once) vector loads: bypass L1 allocation, data is never reused.
__device__ __forceinline__ float4 ld_stream(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ double2 ld_stream(const double2* p) {
  double2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
  return r;
}

// 16-byte shared-memory load that the compiler may neither hoist out of a loop nor merge with an earlier one:
// used to RE-READ loop-invariant parameter sets per use instead of keeping them live in (spilled) registers.
__device__ __forceinline__ void lds16_reload(const float* p, float (&v)[4]) {
  const unsigned addr = static_cast<unsigned>(__cvta_generic_to_shared(p));
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(addr));
}
__device__ __forceinline__ void lds16_reload(const double* p, double (&v)[2]) {
  const unsigned addr = static_cast<unsigned>(__cvta_generic_to_shared(p));
  asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v[0]), "=d"(v[1]) : "r"(addr));
}

// Reciprocal for Jacobian entries whose numerator already carries a few ulp: one MUFU.RCP (<= 1 ulp) in fp32.
__host__ __device__ __forceinline__ float fast_rcp(float x) {
#ifdef __CUDA_ARCH__
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
#else
  return 1.0f / x;
#endif
}
__host__ __device__ __forceinline__ double fast_rcp(double x) { return 1.0 / x; }
// |x| < t in every lane of a value (scalars here; the packed pair F2 has its own overload)
__host__ __device__ __forceinline__ bool all_abs_below(float x, float t) { return fabsf(x) < t; }
__host__ __device__ __forceinline__ bool all_abs_below(double x, float t) { return fabs(x) < double(t); }

template <typename ST>
struct VecOf;
template <>
struct VecOf<float> {
  using type = float4;
  static constexpr int N = 4;
};
template <>
struct VecOf<double> {
  using type = double2;
  static constexpr int N = 2;
};

template <typename ST, typename CT>
__device__ __forceinline__ void load_vec(const ST* base, int64_t group, CT (&out)[VecOf<ST>::N]);

template <>
__device__ __forceinline__ void load_vec<float, float>(const float* base, int64_t g, float (&o)[4]) {
  const float4 v = ld_stream(reinterpret_cast<const float4*>(base) + g);
  o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
}
template <>
__device__ __forceinline__ void load_vec<float, double>(const float* base, int64_t g, double (&o)[4]) {
  const float4 v = ld_stream(reinterpret_cast<const float4*>(base) + g);
  o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
}
template <>
__device__ __forceinline__ void load_vec<double, double>(const double* base, int64_t g, double (&o)[2]) {
  const double2 v = ld_stream(reinterpret_cast<const double2*>(base) + g);
  o[0] = v.x; o[1] = v.y;
}
template <>
__device__ __forceinline__ void load_vec<double, float>(const double* base, int64_t g, float (&o)[2]) {
  const double2 v = ld_stream(reinterpret_cast<const double2*>(base) + g);
  o[0] = float(v.x); o[1] = float(v.y);
}

// IRLS weight  w(e2)  (loss_function.h:16 contract).  `kind` is warp-uniform.
template <typename T>
__device__ __forceinline__ T loss_weight(int kind, T param, T e2);
template <>
__device__ __forceinline__ float loss_weight<float>(int kind, float k, float e2) {
  if (kind == MOPT_LOSS_NONE) return 1.0f;
  if (kind == MOPT_LOSS_GEMAN_MCCLURE) {
    const float d = e2 + k;
    return (k * k) / (d * d);
  }
  return (e2 <= k * k) ? 1.0f : k * rsqrtf(e2);
}
template <>
__device__ __forceinline__ double loss_weight<double>(int kind, double k, double e2) {
  if (kind == MOPT_LOSS_NONE) return 1.0;
  if (kind == MOPT_LOSS_GEMAN_MCCLURE) {
    const double d = e2 + k;
    return (k * k) / (d * d);
  }
  return (e2 <= k * k) ? 1.0 : k / sqrt(e2);
}

#endif  // __CUDACC__

}  // namespace mopt
