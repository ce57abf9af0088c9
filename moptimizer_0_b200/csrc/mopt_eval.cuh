// Per-residual evaluation (mopt_evaluate): CostComputation::computeCost's loop body (linearization.h:36-47) with each
// element's result kept instead of summed.  One streaming sweep over the elements [first, first + count) of a store:
//   residual r_i (model residual on set 0, compute dtype) -> loss weight w_i = loss(r_i^T r_i) ->
//   optional coalesced row-major writes of r_i (count x O) and w_i (count) in the output dtype OT ->
//   fit statistics accumulated per thread in fp64 -> the pass kernels' warp -> CTA -> last-CTA reduction
//   (grid_reduce, context partials / ticket) for the four sums, plus one row of per-CTA maxima for max r^T r.
// The model is a template parameter and mopt_models.cuh is not included: this header is also compiled by NVRTC
// for run-time compiled user models (mopt_rtc.cu), exactly like mopt_pass.cuh.
#pragma once

#include "mopt_common.cuh"
#include "mopt_pass.cuh"

namespace mopt {

constexpr int kEvalThreads = 256;
constexpr int kEvalSums = 4;  // [0] n_valid, [1] n_inliers, [2] sum r^T r, [3] inlier sum r^T r; row 4 of the partials: max

struct EvalArgs {
  int64_t first;   // store index of output row 0
  int64_t count;
  void* r;         // count x O row-major in OT, or null
  void* w;         // count in OT, or null
  double thr2;     // inlier test: double(r^T r) <= thr2
  double* stats;   // device: n_valid, n_inliers, sum_sq, inlier_sum_sq, max_sq (written by the last CTA)
};

#ifdef __CUDACC__

__device__ __forceinline__ void eval_store(float* p, float v) { __stcs(p, v); }
__device__ __forceinline__ void eval_store(double* p, double v) { __stcs(p, v); }

// Grid-stride over VEC-element groups of the store (16-byte loads of every stream, as the pass kernels read), each
// warp taking 32 consecutive groups per round so that its rows of r and w form one contiguous span: the lanes stage
// their rows in shared memory and the warp writes the span with consecutive addresses.  The < VEC elements of the
// range before its first and after its last aligned group are taken one per thread by CTA 0.
template <class M, typename ST, typename CT, typename OT>
__global__ void __launch_bounds__(kEvalThreads) evaluate_kernel(const PassArgs a, const EvalArgs ev) {
  constexpr int THREADS = kEvalThreads, NW = THREADS / 32;
  constexpr int O = M::O, NS = M::NS, NSX = NS > 0 ? NS : 1;
  constexpr int VEC = VecOf<ST>::N;
  constexpr int SETN = M::SETN > 0 ? M::SETN : 1;
  __shared__ CT s_set[SETN];
  __shared__ OT s_r[NW][32 * VEC * O];
  __shared__ OT s_w[NW][32 * VEC];
  __shared__ double s_warp[NW * kEvalSums];
  __shared__ double s_tot[kEvalSums];
  __shared__ double s_wmax[NW];

  for (int i = threadIdx.x; i < M::SETN; i += THREADS) s_set[i] = CT(a.pb->sets[0][i]);
  const int loss = a.cost->loss;
  const CT lossp = CT(a.cost->loss_param);
  const bool masked = a.masked != 0;
  __syncthreads();

  const ST* __restrict__ sp[NSX];
#pragma unroll
  for (int s = 0; s < NS; ++s) sp[s] = static_cast<const ST*>(a.streams.p[s]);
  OT* __restrict__ rout = static_cast<OT*>(ev.r);
  OT* __restrict__ wout = static_cast<OT*>(ev.w);

  double acc[kEvalSums] = {0.0, 0.0, 0.0, 0.0};
  double mx = 0.0;

  // one element: r and w into rdst[0..O) / *wdst (when writing), its statistics into acc / mx
  auto do_elem = [&](const CT (&e)[NSX], OT* rdst, OT* wdst) {
    bool valid = true;
    if (NS > 0 && masked) {  // NaN in the first B-group stream: no correspondence (mopt_icp.cu)
      const CT probe = e[(M::NA < NS) ? M::NA : 0];
      valid = probe == probe;
    }
    CT r[O];
    M::template residual<CT>(s_set, e, r);
    CT e2 = CT(0);
#pragma unroll
    for (int o = 0; o < O; ++o) e2 = fma(r[o], r[o], e2);
    CT w = loss_weight<CT>(loss, lossp, e2);
    if (valid) {
      const double d = double(e2);
      acc[0] += 1.0;
      acc[2] += d;
      mx = fmax(mx, d);
      if (d <= ev.thr2) {
        acc[1] += 1.0;
        acc[3] += d;
      }
    } else {
#pragma unroll
      for (int o = 0; o < O; ++o) r[o] = CT(__int_as_float(0x7fc00000));  // quiet NaN (no <cmath> under NVRTC)
      w = CT(0);
    }
    if (rdst) {
#pragma unroll
      for (int o = 0; o < O; ++o) rdst[o] = OT(r[o]);
    }
    if (wdst) *wdst = OT(w);
  };

  const int64_t end = ev.first + ev.count;
  const int64_t gb = (ev.first + VEC - 1) / VEC, ge = end / VEC;  // whole aligned groups inside the range: [gb, ge)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t stride = int64_t(gridDim.x) * THREADS;
  for (int64_t base = gb + int64_t(blockIdx.x) * THREADS + warp * 32; base < ge; base += stride) {
    const int64_t g = base + lane;
    const bool active = g < ge;
    if (active) {
      CT vals[NSX][VEC];
#pragma unroll
      for (int s = 0; s < NS; ++s) load_vec<ST, CT>(sp[s], g, vals[s]);
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        CT e[NSX];
        e[0] = CT(0);
#pragma unroll
        for (int s = 0; s < NS; ++s) e[s] = vals[s][v];
        do_elem(e, rout ? &s_r[warp][(lane * VEC + v) * O] : nullptr, wout ? &s_w[warp][lane * VEC + v] : nullptr);
      }
    }
    if (rout || wout) {  // warp-uniform: the warp's rows are one contiguous span of the outputs
      __syncwarp();
      const int64_t groups = (ge - base < 32) ? (ge - base) : 32;
      const int64_t row0 = base * VEC - ev.first;
      if (rout) {
        const int nv = int(groups) * VEC * O;
        for (int j = lane; j < nv; j += 32) eval_store(rout + row0 * O + j, s_r[warp][j]);
      }
      if (wout) {
        const int nv = int(groups) * VEC;
        for (int j = lane; j < nv; j += 32) eval_store(wout + row0 + j, s_w[warp][j]);
      }
      __syncwarp();
    }
  }
  if (blockIdx.x == 0) {  // the unaligned head and tail of the range
    const int64_t head_end = (gb * VEC < end) ? gb * VEC : end;
    const int64_t tail_begin = (ge * VEC > head_end) ? ge * VEC : head_end;
    const int64_t nhead = head_end - ev.first;
    const int64_t k = threadIdx.x;
    const int64_t i = (k < nhead) ? ev.first + k : tail_begin + (k - nhead);
    if (i < end) {
      CT e[NSX];
      e[0] = CT(0);
#pragma unroll
      for (int s = 0; s < NS; ++s) e[s] = CT(sp[s][i]);
      do_elem(e, rout ? rout + (i - ev.first) * O : nullptr, wout ? wout + (i - ev.first) : nullptr);
    }
  }

  // max r^T r: warp -> CTA, one per-CTA value in row kEvalSums of the partials (written before grid_reduce's fence)
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) mx = fmax(mx, shfl_xor(mx, o));
  if (lane == 0) s_wmax[warp] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    double m = 0.0;
#pragma unroll
    for (int w = 0; w < NW; ++w) m = fmax(m, s_wmax[w]);
    a.partials[size_t(kEvalSums) * gridDim.x + blockIdx.x] = m;
  }
  const double tot = warp_reduce_transpose<kEvalSums>(acc);
  const double lane_val[1] = {tot};
  if (!grid_reduce<kEvalSums, kEvalSums, 1, THREADS>(lane_val, a, s_tot, s_warp)) return;
  if (threadIdx.x < 32) {
    double m = 0.0;
    for (int c = lane; c < int(gridDim.x); c += 32) m = fmax(m, __ldcg(a.partials + size_t(kEvalSums) * gridDim.x + c));
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) m = fmax(m, shfl_xor(m, o));
    if (lane == 0) {
#pragma unroll
      for (int k = 0; k < kEvalSums; ++k) ev.stats[k] = s_tot[k];
      ev.stats[kEvalSums] = m;
    }
  }
}

#endif  // __CUDACC__

}  // namespace mopt
