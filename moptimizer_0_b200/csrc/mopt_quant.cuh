// Exact residual quantiles (mopt_residual_quantiles): an MSD radix select over the keys e_i = r_i^T r_i of a store.
// e_i >= 0 (+0, finite, +inf) or NaN, so the IEEE bit pattern of e_i read as an unsigned integer orders the keys.
// One streaming sweep per 8-bit digit of that pattern (4 for fp32 keys, 8 for fp64 keys): sweep d recomputes every
// e_i and, for the element whose top 8d bits equal one of the active prefixes, adds 1 to that prefix's bin of digit
// d.  Between sweeps a one-CTA step (mopt_quant.cu) walks the histogram for each target rank, appends the digit its
// rank falls in and builds the next sweep's prefix table.  Counts are integers, so the result does not depend on
// the grid or on the order of the additions.  There is no O(n) scratch: the store is read once per sweep.
// The model is a template parameter and mopt_models.cuh is not included: this header is also compiled by NVRTC
// for run-time compiled user models (mopt_rtc.cu), exactly like mopt_eval.cuh.
#pragma once

#include "mopt_common.cuh"
#include "mopt_pass.cuh"

namespace mopt {

constexpr int kQuantThreads = 256;
constexpr int kQuantMaxQ = MOPT_MAX_QUANTILES + 1;           // the caller's levels, then the median's 0.5
constexpr int kQuantMaxRanks = 2 * kQuantMaxQ;               // lo and hi of each level
constexpr int kQuantBins = 256;                              // one 8-bit digit per sweep

// Device state of one call, allocated with the context and zeroed before sweep 0.  The head up to `rem` is what the
// host reads back after the last sweep.
struct QuantState {
  unsigned long long n_nan;                         // valid elements with a NaN key (counted in sweep 0)
  unsigned long long n_ranked;                      // sum of sweep 0's histogram
  int n_rank;                                       // distinct target ranks
  int n_prefix;                                     // distinct prefixes of the next sweep (0: nothing to select)
  long long rank[kQuantMaxRanks];                   // target order statistics, ascending and distinct
  unsigned long long key[kQuantMaxRanks];           // the digits of each rank's key resolved so far
  long long rem[kQuantMaxRanks];                    // the rank among the elements whose key starts with `key`
  unsigned long long prefix[kQuantMaxRanks];        // ascending and distinct
  unsigned long long hist[kQuantMaxRanks][kQuantBins];
};

struct QuantArgs {
  int64_t first;
  int64_t count;
  QuantState* st;
  int sweep;  // digit d: bits [8 (D - 1 - d), 8 (D - d)) of the key
};

struct QuantLevels {  // the levels of one call, by value into the step after sweep 0
  double q[kQuantMaxQ];
};

#ifdef __CUDACC__

// e = r_0 r_0 (+ r_o r_o)..., each product and sum rounded on its own (no FMA), and its bit pattern.
template <typename CT>
struct QuantKey;
template <>
struct QuantKey<float> {
  using U = unsigned int;
  static constexpr int D = 4;
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ U bits(float e) { return __float_as_uint(e); }
};
template <>
struct QuantKey<double> {
  using U = unsigned long long;
  static constexpr int D = 8;
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ U bits(double e) { return static_cast<U>(__double_as_longlong(e)); }
};

// One sweep.  Grid-stride over VEC-element groups of the store with 16-byte loads of every stream, each warp taking
// 32 consecutive groups per round (evaluate_kernel's skeleton); CTA 0 takes the < VEC elements of the range before
// its first and after its last aligned group.  Bins are counted in shared memory with warp aggregation: the lanes
// of a warp that hit the same bin (in sweep 0 nearly all of them: the top byte of a key is mostly its exponent) add
// their count with one atomic.  The CTA's histogram then goes to the global one with one atomic per non-zero bin.
template <class M, typename ST, typename CT>
__global__ void __launch_bounds__(kQuantThreads) quantile_sweep_kernel(const PassArgs a, const QuantArgs qa) {
  using K = QuantKey<CT>;
  using U = typename K::U;
  constexpr int THREADS = kQuantThreads;
  constexpr int O = M::O, NS = M::NS, NSX = NS > 0 ? NS : 1;
  constexpr int VEC = VecOf<ST>::N;
  constexpr int SETN = M::SETN > 0 ? M::SETN : 1;
  __shared__ CT s_set[SETN];
  __shared__ U s_prefix[kQuantMaxRanks];
  __shared__ unsigned int s_hist[kQuantMaxRanks * kQuantBins];

  QuantState* st = qa.st;
  const int np = qa.sweep == 0 ? 1 : st->n_prefix;  // written by the previous step; uniform over the grid
  if (np == 0) return;                               // empty sample: nothing left to select
  for (int i = threadIdx.x; i < M::SETN; i += THREADS) s_set[i] = CT(a.pb->sets[0][i]);
  for (int i = threadIdx.x; i < np; i += THREADS) s_prefix[i] = U(st->prefix[i]);
  for (int i = threadIdx.x; i < np * kQuantBins; i += THREADS) s_hist[i] = 0u;
  const bool masked = a.masked != 0;
  __syncthreads();

  const ST* __restrict__ sp[NSX];
#pragma unroll
  for (int s = 0; s < NS; ++s) sp[s] = static_cast<const ST*>(a.streams.p[s]);
  const int shift = 8 * (K::D - 1 - qa.sweep);
  unsigned long long nans = 0;

  // the bin of one element (prefix index * 256 + digit), or -1: no correspondence, a NaN key, or no active prefix
  auto bin_of = [&](const CT (&e)[NSX]) -> int {
    if (NS > 0 && masked) {  // NaN in the first B-group stream: no correspondence (mopt_icp.cu)
      const CT probe = e[(M::NA < NS) ? M::NA : 0];
      if (probe != probe) return -1;
    }
    CT r[O];
    M::template residual<CT>(s_set, e, r);
    CT e2 = K::mul(r[0], r[0]);
#pragma unroll
    for (int o = 1; o < O; ++o) e2 = K::add(e2, K::mul(r[o], r[o]));
    if (e2 != e2) {
      ++nans;
      return -1;
    }
    const U key = K::bits(e2);
    const int digit = int((key >> shift) & U(0xff));
    if (qa.sweep == 0) return digit;
    const U pre = key >> (shift + 8);
    for (int p = 0; p < np; ++p)
      if (s_prefix[p] == pre) return p * kQuantBins + digit;
    return -1;
  };
  // warp-uniform: every lane passes its bin (or -1); one atomic per distinct bin of the warp
  auto count_bin = [&](int bin) {
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && int(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&s_hist[bin], unsigned(__popc(peers)));
  };

  const int64_t end = qa.first + qa.count;
  const int64_t gb = (qa.first + VEC - 1) / VEC, ge = end / VEC;  // whole aligned groups inside the range: [gb, ge)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t stride = int64_t(gridDim.x) * THREADS;
  for (int64_t base = gb + int64_t(blockIdx.x) * THREADS + warp * 32; base < ge; base += stride) {
    const int64_t g = base + lane;
    int bins[VEC];
    if (g < ge) {
      CT vals[NSX][VEC];
#pragma unroll
      for (int s = 0; s < NS; ++s) load_vec<ST, CT>(sp[s], g, vals[s]);
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        CT e[NSX];
        e[0] = CT(0);
#pragma unroll
        for (int s = 0; s < NS; ++s) e[s] = vals[s][v];
        bins[v] = bin_of(e);
      }
    } else {
#pragma unroll
      for (int v = 0; v < VEC; ++v) bins[v] = -1;
    }
#pragma unroll
    for (int v = 0; v < VEC; ++v) count_bin(bins[v]);
  }
  if (blockIdx.x == 0) {  // the unaligned head and tail of the range
    const int64_t head_end = (gb * VEC < end) ? gb * VEC : end;
    const int64_t tail_begin = (ge * VEC > head_end) ? ge * VEC : head_end;
    const int64_t nhead = head_end - qa.first;
    const int64_t k = threadIdx.x;
    const int64_t i = (k < nhead) ? qa.first + k : tail_begin + (k - nhead);
    int bin = -1;
    if (i < end) {
      CT e[NSX];
      e[0] = CT(0);
#pragma unroll
      for (int s = 0; s < NS; ++s) e[s] = CT(sp[s][i]);
      bin = bin_of(e);
    }
    count_bin(bin);
  }
  if (qa.sweep == 0) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) nans += shfl_xor(nans, o);
    if (lane == 0 && nans) atomicAdd(&st->n_nan, nans);
  }
  __syncthreads();
  unsigned long long* hist = &st->hist[0][0];
  for (int i = threadIdx.x; i < np * kQuantBins; i += THREADS)
    if (s_hist[i]) atomicAdd(hist + i, (unsigned long long)s_hist[i]);
}

#endif  // __CUDACC__

}  // namespace mopt
