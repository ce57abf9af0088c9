// Instantiations of the radix-select sweep (mopt_quant.cuh) for the builtin models, and the one-CTA step
// between sweeps, which is the same for every model.
#include "mopt_internal.h"
#include "mopt_quant.cuh"
#include "mopt_quant_rule.h"

namespace mopt {
namespace {

// After sweep d: copy the histogram of the active prefixes to shared memory and zero it for the next sweep.  After
// sweep 0, n_ranked is the histogram's total and the target ranks follow from it (lo and hi of every level, deduped
// and sorted).  Then one warp per rank finds the bin its remaining rank falls in: each lane owns 8 consecutive bins,
// a warp scan of the lanes' totals names the lane, and that lane walks its 8 bins.  The digit is appended to the
// rank's key; the distinct keys, ascending because the ranks are, are the prefixes of the next sweep.
__global__ void __launch_bounds__(256) quantile_step_kernel(QuantState* st, int sweep, int n_q, QuantLevels lv) {
  __shared__ unsigned long long s_hist[kQuantMaxRanks * kQuantBins];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int np = sweep == 0 ? 1 : st->n_prefix;
  if (np == 0) return;
  unsigned long long* hist = &st->hist[0][0];
  for (int i = threadIdx.x; i < np * kQuantBins; i += blockDim.x) {
    s_hist[i] = hist[i];
    hist[i] = 0ull;
  }
  __syncthreads();
  if (sweep == 0) {
    if (warp == 0) {
      unsigned long long n = 0;
      for (int b = lane; b < kQuantBins; b += 32) n += s_hist[b];
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) n += shfl_xor(n, o);
      if (lane == 0) {
        st->n_ranked = n;
        int nr = 0;
        if (n > 0) {
          long long rk[kQuantMaxRanks];
          for (int k = 0; k < n_q; ++k) {
            const QuantRank r = quantile_rank(int64_t(n), lv.q[k]);
            const long long c[2] = {r.j, r.j1};
            for (int m = 0; m < 2; ++m) {  // insertion into the sorted, distinct list
              int pos = 0;
              while (pos < nr && rk[pos] < c[m]) ++pos;
              if (pos < nr && rk[pos] == c[m]) continue;
              for (int s = nr; s > pos; --s) rk[s] = rk[s - 1];
              rk[pos] = c[m];
              ++nr;
            }
          }
          for (int r = 0; r < nr; ++r) {
            st->rank[r] = rk[r];
            st->rem[r] = rk[r];
            st->key[r] = 0ull;
          }
        }
        st->n_rank = nr;
        st->n_prefix = nr > 0 ? 1 : 0;
        st->prefix[0] = 0ull;
      }
    }
    __syncthreads();
  }
  const int nr = st->n_rank;
  for (int r = warp; r < nr; r += int(blockDim.x >> 5)) {
    const unsigned long long key = st->key[r];
    int p = 0;
    while (p < np - 1 && st->prefix[p] != key) ++p;
    const unsigned long long* h = s_hist + p * kQuantBins + lane * 8;
    unsigned long long c[8], s = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      c[k] = h[k];
      s += c[k];
    }
    unsigned long long inc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    const unsigned long long rem = (unsigned long long)st->rem[r];
    unsigned long long cum = inc - s;
    if (rem >= cum && rem < inc) {  // exactly one lane: rem < the prefix's total by construction
      int b = 0;
      while (rem >= cum + c[b]) cum += c[b++];
      st->rem[r] = (long long)(rem - cum);
      st->key[r] = (key << 8) | (unsigned long long)(lane * 8 + b);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int n = 0;
    for (int r = 0; r < nr; ++r)
      if (n == 0 || st->prefix[n - 1] != st->key[r]) st->prefix[n++] = st->key[r];
    st->n_prefix = n;
  }
}

}  // namespace

int quantile_sweep_kernel_desc(int model, int store_dtype, int compute_dtype, KernelDesc* k) {
  return with_builtin_model(model, [&](auto m) {
    return with_dtypes(store_dtype, compute_dtype, [&](auto st, auto ct) {
      *k = builtin_kernel(
          reinterpret_cast<const void*>(quantile_sweep_kernel<decltype(m), decltype(st), decltype(ct)>), kQuantThreads);
      return MOPT_OK;
    });
  });
}

int launch_quantile_step(cudaStream_t stream, QuantState* st, int sweep, int n_q, const QuantLevels& lv) {
  quantile_step_kernel<<<1, 256, 0, stream>>>(st, sweep, n_q, lv);
  MOPT_CUDA_TRY(cudaGetLastError());
  return MOPT_OK;
}

}  // namespace mopt
