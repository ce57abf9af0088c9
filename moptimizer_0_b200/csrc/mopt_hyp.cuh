// Hypothesis scoring (mopt_score_hypotheses): mopt_evaluate's statistics of one store at many parameter vectors in
// one pass.  The lanes of a warp are hypotheses and the loop runs over the data: each warp loads 32 consecutive
// 16-byte groups of every stream (evaluate_kernel's reads), stages them in its slice of shared memory, and every lane
// walks the staged elements with broadcast reads, scoring them against the set of its own hypothesis, which it keeps
// in registers.  Counts, sums and the maximum stay in registers; the lanes, warps and CTAs are combined once, at the
// end, in a fixed order.  blockIdx.y selects a tile of 32 hypotheses, so the store is read once per tile.  Measured
// on a B200 (DESIGN.md 3.10): one hypothesis is bound by HBM, as mopt_evaluate is; from one full tile on the kernel is
// bound by instruction issue (33.5 issue slots per hypothesis-element for point2point fp32), not by HBM.
// A tile of K < 32 hypotheses spreads each over 32 / K' lanes (K' the next power of two >= K): those lanes share the
// staged elements and are combined by a fixed xor-shuffle tree.
// The model is a template parameter and mopt_models.cuh is not included: this header is also compiled by NVRTC
// for run-time compiled user models (mopt_rtc.cu), exactly like mopt_eval.cuh.
#pragma once

#include "mopt_common.cuh"
#include "mopt_pass.cuh"

namespace mopt {

constexpr int kHypThreads = 128;
constexpr int kHypTile = 32;                     // hypotheses per tile: one per lane
constexpr int kHypStats = 5;                     // n_valid, n_inliers, sum e2, inlier sum e2, max e2
constexpr int kHypRows = kHypTile * kHypStats;   // per-CTA partials of one tile

struct HypArgs {
  int64_t first;
  int64_t count;
  int n_hyp;
  float thr2f;           // fp32 keys: the largest float <= thr2 (mopt_hyp_rule.h), the same test without a conversion
  double thr2;           // fp64 keys: double(e2) <= thr2
  const double* sets;    // [n_hyp][kSetSize]: set 0 of every hypothesis (setup_hypotheses)
  double* partials;      // [tile][kHypRows][gridDim.x]
  unsigned int* tickets; // [tile], self-resetting
  double* out;           // [n_hyp][kHypStats], written by the last CTA of each tile
};

#ifdef __CUDACC__

__device__ __forceinline__ bool hyp_inlier(float e2, const HypArgs& h) { return e2 <= h.thr2f; }
__device__ __forceinline__ bool hyp_inlier(double e2, const HypArgs& h) { return e2 <= h.thr2; }

// One 16-byte broadcast read of CHUNK staged values.
__device__ __forceinline__ void hyp_lds(const float* p, float (&v)[4]) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void hyp_lds(const double* p, double (&v)[2]) {
  const double2 t = *reinterpret_cast<const double2*>(p);
  v[0] = t.x; v[1] = t.y;
}

// Minimum 1 CTA per SM: without it ptxas caps the registers of the camera models' fp64 instantiations below what
// their set, the staged values and the slow path of the fp64 division (a call) hold live, and spills.
template <class M, typename ST, typename CT>
__global__ void __launch_bounds__(kHypThreads, 1) hypothesis_score_kernel(const PassArgs a, const HypArgs h) {
  constexpr int THREADS = kHypThreads, NW = THREADS / 32;
  constexpr int O = M::O, NS = M::NS, NSX = NS > 0 ? NS : 1;
  constexpr int VEC = VecOf<ST>::N;
  constexpr int STAGE = 32 * VEC;             // elements a warp stages per round
  constexpr int CHUNK = 16 / int(sizeof(CT)); // elements of one stream per 16-byte shared read (divides VEC)
  constexpr int SETN = M::SETN > 0 ? M::SETN : 1;
  __shared__ __align__(16) CT s_el[NW][NSX][STAGE];
  __shared__ double s_warp[NW][kHypRows];
  __shared__ bool s_last;

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tile = blockIdx.y;
  const int nt = min(kHypTile, h.n_hyp - tile * kHypTile);  // hypotheses of this tile
  const int kp = next_pow2(nt);                               // lanes per element round: kp hypotheses side by side
  const int spread = kHypTile / kp;                           // lanes per hypothesis
  const int hl = lane & (kp - 1), sub = lane / kp;
  const int hyp = tile * kHypTile + min(hl, nt - 1);          // the lanes of a padding slot repeat the last hypothesis

  CT set[SETN];
#pragma unroll
  for (int i = 0; i < SETN; ++i) set[i] = CT(h.sets[size_t(hyp) * kSetSize + i]);
  const bool masked = a.masked != 0;

  const ST* __restrict__ sp[NSX];
#pragma unroll
  for (int s = 0; s < NS; ++s) sp[s] = static_cast<const ST*>(a.streams.p[s]);

  unsigned int nv = 0, ni = 0;
  double sum = 0.0, isum = 0.0;
  CT mx = CT(0);

  // mopt_evaluate's per-element statistics (evaluate_kernel's do_elem): same residual, same key, same test
  auto elem = [&](const CT (&e)[NSX]) {
    bool valid = true;
    if (NS > 0 && masked) {  // NaN in the first B-group stream: no correspondence (mopt_icp.cu)
      const CT probe = e[(M::NA < NS) ? M::NA : 0];
      valid = probe == probe;
    }
    CT r[O];
    M::template residual<CT>(set, e, r);
    CT e2 = CT(0);
#pragma unroll
    for (int o = 0; o < O; ++o) e2 = fma(r[o], r[o], e2);
    if (valid) {
      const double d = double(e2);
      nv += 1u;
      sum += d;
      mx = fmax(mx, e2);  // max in CT: the conversion to fp64 is monotone, and fmax drops NaN in either precision
      if (hyp_inlier(e2, h)) {
        ni += 1u;
        isum += d;
      }
    }
  };

  const int64_t end = h.first + h.count;
  const int64_t gb = (h.first + VEC - 1) / VEC, ge = end / VEC;  // whole aligned groups inside the range: [gb, ge)
  const int64_t stride = int64_t(gridDim.x) * THREADS;
  for (int64_t base = gb + int64_t(blockIdx.x) * THREADS + warp * 32; base < ge; base += stride) {
    const int64_t g = base + lane;
    if (g < ge) {
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        CT v[VEC];
        load_vec<ST, CT>(sp[s], g, v);
#pragma unroll
        for (int k = 0; k < VEC; ++k) s_el[warp][s][lane * VEC + k] = v[k];
      }
    }
    __syncwarp();
    const int nchunk = int((ge - base < 32) ? (ge - base) : 32) * (VEC / CHUNK);
    for (int c = sub; c < nchunk; c += spread) {
      CT v[NSX][CHUNK];
#pragma unroll
      for (int s = 0; s < NS; ++s) hyp_lds(&s_el[warp][s][c * CHUNK], v[s]);
#pragma unroll
      for (int k = 0; k < CHUNK; ++k) {
        CT e[NSX];
        e[0] = CT(0);
#pragma unroll
        for (int s = 0; s < NS; ++s) e[s] = v[s][k];
        elem(e);
      }
    }
    __syncwarp();  // the slice is refilled next round
  }
  if (blockIdx.x == 0 && warp == 0) {  // the < VEC elements of the range before its first and after its last group
    const int64_t head_end = (gb * VEC < end) ? gb * VEC : end;
    const int64_t tail_begin = (ge * VEC > head_end) ? ge * VEC : head_end;
    const int nhead = int(head_end - h.first);
    const int nel = nhead + int(end - tail_begin);
    if (lane < nel) {
      const int64_t i = (lane < nhead) ? h.first + lane : tail_begin + (lane - nhead);
#pragma unroll
      for (int s = 0; s < NS; ++s) s_el[0][s][lane] = CT(sp[s][i]);
    }
    __syncwarp();
    for (int j = sub; j < nel; j += spread) {
      CT e[NSX];
      e[0] = CT(0);
#pragma unroll
      for (int s = 0; s < NS; ++s) e[s] = s_el[0][s][j];
      elem(e);
    }
  }

  // the lanes of one hypothesis (lane bits >= log2 kp), by a fixed xor tree
  double mxd = double(mx);
  for (int o = kp; o < 32; o <<= 1) {
    nv += __shfl_xor_sync(0xffffffffu, nv, o);
    ni += __shfl_xor_sync(0xffffffffu, ni, o);
    sum += shfl_xor(sum, o);
    isum += shfl_xor(isum, o);
    mxd = fmax(mxd, shfl_xor(mxd, o));
  }
  if (sub == 0) {
    double* w = &s_warp[warp][hl * kHypStats];
    w[0] = double(nv);
    w[1] = double(ni);
    w[2] = sum;
    w[3] = isum;
    w[4] = mxd;
  }
  __syncthreads();
  // the warps of the CTA in order, one row of per-CTA partials per (hypothesis, statistic)
  const int rows = nt * kHypStats;
  double* part = h.partials + size_t(tile) * kHypRows * gridDim.x;
  for (int i = threadIdx.x; i < rows; i += THREADS) {
    const bool is_max = (i % kHypStats) == kHypStats - 1;
    double s = s_warp[0][i];
#pragma unroll
    for (int w = 1; w < NW; ++w) s = is_max ? fmax(s, s_warp[w][i]) : s + s_warp[w][i];
    part[size_t(i) * gridDim.x + blockIdx.x] = s;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(&h.tickets[tile], 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  // last CTA of the tile: each row over the CTAs, lanes striding, then a fixed xor butterfly
  for (int i = warp; i < rows; i += NW) {
    const bool is_max = (i % kHypStats) == kHypStats - 1;
    double s = 0.0;
    for (int c = lane; c < int(gridDim.x); c += 32) {
      const double v = __ldcg(part + size_t(i) * gridDim.x + c);
      s = is_max ? fmax(s, v) : s + v;
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
      const double t = shfl_xor(s, o);
      s = is_max ? fmax(s, t) : s + t;
    }
    if (lane == 0) h.out[size_t(tile) * kHypRows + i] = s;
  }
  if (threadIdx.x == 0) h.tickets[tile] = 0u;  // ready for the next launch (stream-ordered)
}

#endif  // __CUDACC__

}  // namespace mopt
