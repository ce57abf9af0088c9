// Closed-form rigid alignment (mopt_align_terms): the weighted first and second moments of a point2point store's
// source points p (group A) and target points q (group B), over the elements that mopt_evaluate counts as inliers at
// x, in one streaming sweep.  Horn's solve (mopt_align.cu) turns them into the best rigid transform.
//
// The moments are kept in centred form: (W, mean p, mean q, sum w (p - mean p)(q - mean q)^T, sum w |p - mean p|^2,
// sum w |q - mean q|^2).  Raw sums (sum w p q^T - W mean p mean q^T) cancel catastrophically on a cloud far from the
// origin: about 12 digits of the cross term are lost at 1e6 from the origin with unit spread.  Each thread sums about
// its own pivot (its first used element), which keeps its sums at the scale of the spread; then threads, warps, CTAs
// and the last CTA combine centred moments by Chan's pairwise rule (align_merge) in a fixed order.
#pragma once

#include "mopt_common.cuh"
#include "mopt_pass.cuh"

namespace mopt {

constexpr int kAlignThreads = 256;

// The device form of mopt_align_moments: counts as doubles (exact below 2^53), the moments, and the rounding error of
// each mean (mean = mean_* + lo_*).  Far from the origin a mean rounded to one double is off by up to half an ulp
// (6e-11 at 1e6), and Chan's correction f d_src d_tgt^T takes that error at first order with every merge; with the
// error carried along, the differences of means are exact to rounding.  kAlignRows doubles.
struct AlignAcc {
  double n_valid, n_used;
  double w;
  double mean_src[3], mean_tgt[3];
  double cross[9];  // cross[3a + b] = sum w (p_a - mean_src_a)(q_b - mean_tgt_b)
  double var_src, var_tgt;
  double lo_src[3], lo_tgt[3];
};
constexpr int kAlignRows = int(sizeof(AlignAcc) / sizeof(double));
static_assert(kAlignRows <= kMaxRaw, "the per-CTA partials of the alignment kernel must fit the context's partials");

struct AlignArgs {
  int64_t first;
  int64_t count;
  double thr2;   // used: double(e2) <= thr2, mopt_evaluate's inlier test
  double* out;   // device: kAlignRows doubles (an AlignAcc), written by the last CTA
};

// s + e = a + b exactly (Knuth's TwoSum); the same bits for (b, a).
__host__ __device__ inline void two_sum(double a, double b, double& s, double& e) {
  s = a + b;
  const double bb = s - a;
  e = (a - (s - bb)) + (b - bb);
}

// Chan's pairwise combination of the terms of two disjoint sets.  merge(a, b) and merge(b, a) give the same bits:
// every formula is symmetric under the swap (d -> -d, Wb - Wa -> Wa - Wb), the merged mean taken as the midpoint plus
// (Wb - Wa) / 2W d.  An operand of weight 0 contributes no moments and leaves the other's unchanged; counts always
// add.  `o` may alias `a` or `b`.
__host__ __device__ inline void align_merge(const AlignAcc& a, const AlignAcc& b, AlignAcc& o) {
  AlignAcc r;
  if (a.w == 0.0 || b.w == 0.0) {
    const AlignAcc zero{};
    r = (b.w == 0.0) ? (a.w == 0.0 ? zero : a) : b;  // both empty: zero moments, whichever order
  } else {
    const double W = a.w + b.w;
    const double f = (a.w * b.w) / W, g = (b.w - a.w) / (2.0 * W);
    double ds[3], dt[3];
    for (int k = 0; k < 3; ++k) {
      ds[k] = (b.mean_src[k] - a.mean_src[k]) + (b.lo_src[k] - a.lo_src[k]);
      dt[k] = (b.mean_tgt[k] - a.mean_tgt[k]) + (b.lo_tgt[k] - a.lo_tgt[k]);
      double s, e;
      two_sum(a.mean_src[k], b.mean_src[k], s, e);
      two_sum(0.5 * s, 0.5 * (e + (a.lo_src[k] + b.lo_src[k])) + g * ds[k], r.mean_src[k], r.lo_src[k]);
      two_sum(a.mean_tgt[k], b.mean_tgt[k], s, e);
      two_sum(0.5 * s, 0.5 * (e + (a.lo_tgt[k] + b.lo_tgt[k])) + g * dt[k], r.mean_tgt[k], r.lo_tgt[k]);
    }
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) r.cross[3 * i + j] = (a.cross[3 * i + j] + b.cross[3 * i + j]) + (f * ds[i]) * dt[j];
    r.var_src = (a.var_src + b.var_src) + f * (ds[0] * ds[0] + ds[1] * ds[1] + ds[2] * ds[2]);
    r.var_tgt = (a.var_tgt + b.var_tgt) + f * (dt[0] * dt[0] + dt[1] * dt[1] + dt[2] * dt[2]);
    r.w = W;
  }
  r.n_valid = a.n_valid + b.n_valid;
  r.n_used = a.n_used + b.n_used;
  o = r;
}

#ifdef __CUDACC__

// Every lane ends with the warp's total: at each level a lane and its xor partner merge the same pair in opposite
// orders, which gives the same bits.
__device__ __forceinline__ void align_warp_merge(AlignAcc& v) {
#pragma unroll 1
  for (int o = 16; o >= 1; o >>= 1) {
    AlignAcc p;
    double* pv = reinterpret_cast<double*>(&p);
    const double* vv = reinterpret_cast<const double*>(&v);
#pragma unroll
    for (int k = 0; k < kAlignRows; ++k) pv[k] = shfl_xor(vv[k], o);
    align_merge(v, p, v);
  }
}

// Grid-stride over VEC-element groups of the store (evaluate_kernel's 16-byte loads); the < VEC elements of the range
// before its first and after its last aligned group are taken one per thread by CTA 0.
template <class M, typename ST, typename CT>
__global__ void __launch_bounds__(kAlignThreads) align_terms_kernel(const PassArgs a, const AlignArgs al) {
  static_assert(M::NS == 6 && M::NA == 3, "closed-form alignment reads a point2point store: p = A[0..3), q = B[0..3)");
  constexpr int THREADS = kAlignThreads, NW = THREADS / 32, NS = 6;
  constexpr int VEC = VecOf<ST>::N;
  __shared__ CT s_set[M::SETN];
  __shared__ AlignAcc s_warp[NW];
  __shared__ bool s_last;

  for (int i = threadIdx.x; i < M::SETN; i += THREADS) s_set[i] = CT(a.pb->sets[0][i]);
  const int loss = a.cost->loss;
  const CT lossp = CT(a.cost->loss_param);
  const bool masked = a.masked != 0;
  __syncthreads();

  const ST* __restrict__ sp[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) sp[s] = static_cast<const ST*>(a.streams.p[s]);

  // sums about the pivot (cp, cq): W, S_p = sum w dp, S_q = sum w dq, S_pq = sum w dp dq^T, S_pp, S_qq
  double nv = 0.0, nu = 0.0, W = 0.0, Sp[3] = {0.0, 0.0, 0.0}, Sq[3] = {0.0, 0.0, 0.0}, Spq[9], Spp = 0.0, Sqq = 0.0;
#pragma unroll
  for (int k = 0; k < 9; ++k) Spq[k] = 0.0;
  double cp[3] = {0.0, 0.0, 0.0}, cq[3] = {0.0, 0.0, 0.0};
  bool piv = false;

  // mopt_evaluate's per-element rule (evaluate_kernel's do_elem): same validity, residual, key, test and weight
  auto elem = [&](const CT (&e)[NS]) {
    bool valid = true;
    if (masked) {  // NaN in the first B-group stream: no correspondence (mopt_icp.cu)
      const CT probe = e[M::NA];
      valid = probe == probe;
    }
    CT r[M::O];
    M::template residual<CT>(s_set, e, r);
    CT e2 = CT(0);
#pragma unroll
    for (int o = 0; o < M::O; ++o) e2 = fma(r[o], r[o], e2);
    if (!valid) return;
    nv += 1.0;
    if (!(double(e2) <= al.thr2)) return;  // NaN keys never enter
    nu += 1.0;
    const double w = double(loss_weight<CT>(loss, lossp, e2));
    if (!piv) {
#pragma unroll
      for (int k = 0; k < 3; ++k) cp[k] = double(e[k]), cq[k] = double(e[3 + k]);
      piv = true;
    }
    double dp[3], dq[3], wdp[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      dp[k] = double(e[k]) - cp[k];
      dq[k] = double(e[3 + k]) - cq[k];
      wdp[k] = w * dp[k];
      Sp[k] += wdp[k];
      Sq[k] = fma(w, dq[k], Sq[k]);
    }
    W += w;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) Spq[3 * i + j] = fma(wdp[i], dq[j], Spq[3 * i + j]);
    Spp = fma(wdp[0], dp[0], fma(wdp[1], dp[1], fma(wdp[2], dp[2], Spp)));
    Sqq = fma(w, fma(dq[0], dq[0], fma(dq[1], dq[1], dq[2] * dq[2])), Sqq);
  };

  const int64_t end = al.first + al.count;
  const int64_t gb = (al.first + VEC - 1) / VEC, ge = end / VEC;  // whole aligned groups inside the range: [gb, ge)
  const int64_t stride = int64_t(gridDim.x) * THREADS;
  for (int64_t g = gb + int64_t(blockIdx.x) * THREADS + threadIdx.x; g < ge; g += stride) {
    CT vals[NS][VEC];
#pragma unroll
    for (int s = 0; s < NS; ++s) load_vec<ST, CT>(sp[s], g, vals[s]);
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      CT e[NS];
#pragma unroll
      for (int s = 0; s < NS; ++s) e[s] = vals[s][v];
      elem(e);
    }
  }
  if (blockIdx.x == 0) {  // the unaligned head and tail of the range
    const int64_t head_end = (gb * VEC < end) ? gb * VEC : end;
    const int64_t tail_begin = (ge * VEC > head_end) ? ge * VEC : head_end;
    const int64_t nhead = head_end - al.first;
    const int64_t k = threadIdx.x;
    const int64_t i = (k < nhead) ? al.first + k : tail_begin + (k - nhead);
    if (i < end) {
      CT e[NS];
#pragma unroll
      for (int s = 0; s < NS; ++s) e[s] = CT(sp[s][i]);
      elem(e);
    }
  }

  // the thread's centred moments
  AlignAcc m;
  m.n_valid = nv;
  m.n_used = nu;
  m.w = W;
  const double iw = W > 0.0 ? 1.0 / W : 0.0;
#pragma unroll
  for (int k = 0; k < 3; ++k) {  // pivot + mean offset, rounded, with the rounding error kept
    two_sum(cp[k], Sp[k] * iw, m.mean_src[k], m.lo_src[k]);
    two_sum(cq[k], Sq[k] * iw, m.mean_tgt[k], m.lo_tgt[k]);
  }
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) m.cross[3 * i + j] = W > 0.0 ? Spq[3 * i + j] - Sp[i] * (Sq[j] * iw) : 0.0;
  m.var_src = W > 0.0 ? Spp - (Sp[0] * Sp[0] + Sp[1] * Sp[1] + Sp[2] * Sp[2]) * iw : 0.0;
  m.var_tgt = W > 0.0 ? Sqq - (Sq[0] * Sq[0] + Sq[1] * Sq[1] + Sq[2] * Sq[2]) * iw : 0.0;

  // lanes -> warps (in order, thread 0) -> one row of per-CTA partials per field
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  align_warp_merge(m);
  if (lane == 0) s_warp[warp] = m;
  __syncthreads();
  const unsigned G = gridDim.x;
  if (threadIdx.x == 0) {
    AlignAcc c = s_warp[0];
    for (int w = 1; w < NW; ++w) align_merge(c, s_warp[w], c);
    const double* cv = reinterpret_cast<const double*>(&c);
    for (int k = 0; k < kAlignRows; ++k) a.partials[size_t(k) * G + blockIdx.x] = cv[k];
    __threadfence();
    s_last = atomicAdd(a.ticket, 1u) == G - 1;
  }
  __syncthreads();
  if (!s_last || warp != 0) return;
  __threadfence();
  // last CTA: lane l folds CTAs l, l + 32, ... in order, then the lanes by the butterfly
  AlignAcc t = {};
  for (unsigned c = lane; c < G; c += 32) {
    AlignAcc v;
    double* vv = reinterpret_cast<double*>(&v);
    for (int k = 0; k < kAlignRows; ++k) vv[k] = __ldcg(a.partials + size_t(k) * G + c);
    align_merge(t, v, t);
  }
  align_warp_merge(t);
  if (lane == 0) {
    const double* tv = reinterpret_cast<const double*>(&t);
    for (int k = 0; k < kAlignRows; ++k) al.out[k] = tv[k];
    *a.ticket = 0u;  // ready for the next launch (stream-ordered)
  }
}

#endif  // __CUDACC__

}  // namespace mopt
