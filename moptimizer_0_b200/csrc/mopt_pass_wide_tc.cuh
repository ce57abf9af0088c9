// The n x n calibration case (P up to 15: 136 packed sums), fp32 store + fp32 compute, second generation.
//
// wide_pass_kernel (mopt_pass.cuh) spends ~40 % of its issue slots on the warp-level product C += J^T B over the
// residual rows of 32 observations (352 FFMA per lane) and the rest on one finite-difference Jacobian per lane.
// Here
//   1. every lane evaluates TWO observations at once in packed fp32 (F2 = one float2 per value, fma.rn.f32x2 etc.),
//      the models' templated hooks (affine / finish_diff / tail_partials / stage1 / stage2) instantiated for F2;
//   2. the lane scales its rows by sqrt(w) and stores X = sqrt(w) [J | r] TRANSPOSED (parameter-major, the residual
//      rows of the warp's 64 observations contiguous) into the warp's shared tile, one conflict-free 8-byte store per
//      value pair;
//   3. H and b are the Gram matrix X^T X (column P of X holds sqrt(w) r, so column P of the product is b), computed
//      on the tensor cores: mma.sync.m16n8k8 TF32 with the operands split as x = hi + lo (hi = x rounded to TF32,
//      lo = x - hi) and three products hi.hi + hi.lo + lo.hi accumulated in fp32 — the split holds 6e-8 in the scale
//      sqrt(H_ii H_jj), as good as the FFMA loop (scripts/analysis_tf32_split.py; one TF32 product alone: 1.9e-5).
//      Because A = B = X the B fragments ARE the A fragments' registers (m16n8k4: b0 of n-tile 0 / 1 = a0 / a1 of the
//      ldmatrix.x4 that fetched A), and X_lo^T X_hi = (X_hi^T X_lo)^T, so only S = X_hi^T X_hi and T = X_hi^T X_lo
//      are accumulated and H = S + T + T^T is formed once at the end: one ldmatrix and four splits feed eight
//      k4-MMAs per 8 residual rows;
//   4. fp32 accumulators are folded into fp64 every FLUSH groups, then the usual warp -> CTA -> grid reduction.
// Identity covariance only (C = I: src/cost_function_*_dyn.cpp:14-15 default); setCovariance problems take the
// first-generation kernel.  Replaces the loop of computeHessianNumerical (linearization.h:65-124) for the
// pinhole + distortion model (BASELINE.json configs[4]).
#pragma once

#include <type_traits>

#include "mopt_models.cuh"
#include "mopt_pass.cuh"

namespace mopt {
#ifdef __CUDACC__

// ---- packed pair of floats with the arithmetic the model hooks use -------------------------------------------
struct F2 {
  float2 v;
  F2() = default;
  template <typename T, typename = typename std::enable_if<std::is_arithmetic<T>::value>::type>
  MOPT_HD F2(T a) : v{float(a), float(a)} {}
  MOPT_HD F2(float a, float b) : v{a, b} {}
};
MOPT_HD F2 operator+(F2 a, F2 b) {
#ifdef __CUDA_ARCH__
  F2 r; r.v = __fadd2_rn(a.v, b.v); return r;
#else
  return F2(a.v.x + b.v.x, a.v.y + b.v.y);
#endif
}
MOPT_HD F2 operator-(F2 a) { return F2(-a.v.x, -a.v.y); }
MOPT_HD F2 operator-(F2 a, F2 b) { return a + (-b); }
MOPT_HD F2 operator*(F2 a, F2 b) {
#ifdef __CUDA_ARCH__
  F2 r; r.v = __fmul2_rn(a.v, b.v); return r;
#else
  return F2(a.v.x * b.v.x, a.v.y * b.v.y);
#endif
}
MOPT_HD F2 operator/(F2 a, F2 b) { return F2(a.v.x / b.v.x, a.v.y / b.v.y); }
MOPT_HD F2 fma(F2 a, F2 b, F2 c) {
#ifdef __CUDA_ARCH__
  F2 r; r.v = __ffma2_rn(a.v, b.v, c.v); return r;
#else
  return F2(fmaf(a.v.x, b.v.x, c.v.x), fmaf(a.v.y, b.v.y, c.v.y));
#endif
}
MOPT_HD F2 fast_rcp(F2 a) { return F2(fast_rcp(a.v.x), fast_rcp(a.v.y)); }
MOPT_HD F2 exp(F2 a) { return F2(expf(a.v.x), expf(a.v.y)); }
MOPT_HD bool all_abs_below(F2 a, float t) { return fabsf(a.v.x) < t && fabsf(a.v.y) < t; }

// ---- tensor-core helpers -----------------------------------------------------------------------------------
__device__ __forceinline__ void ldmatrix_x4(const float* p, unsigned (&r)[4]) {
  const unsigned addr = static_cast<unsigned>(__cvta_generic_to_shared(p));
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
// x = hi + lo for the 3 x TF32 product.  hi is x rounded to nearest at TF32's 10-bit mantissa: x + 0x1000 as an integer,
// the 13 low bits are ignored by the tensor core (the operand needs no masking); lo = x - (hi with the low bits
// cleared) is exact in fp32.  (cvt.rna.tf32.f32 is emulated on sm_100 with an Inf / NaN guard: 4 instructions; the
// residual rows here are finite.)
__device__ __forceinline__ void split_tf32(unsigned x, unsigned& hi, float& lo) {
  hi = x + 0x1000u;
  lo = __uint_as_float(x) - __uint_as_float(hi & 0xffffe000u);
}
// D(16x8, fp32) += A(16x4, tf32, row) * B(4x8, tf32, col).  The k4 shape takes ONE register for B, so the B fragments
// of the Gram product are the A fragment's own registers (no register-pair shuffling as the k8 shape would need).
__device__ __forceinline__ void mma_tf32_k4(float (&c)[4], unsigned a0, unsigned a1, unsigned b0) {
  asm volatile("mma.sync.aligned.m16n8k4.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(b0));
}

// D = A * B (no accumulator input): starts a short accumulation chain, see the k-loop of wide_tc_kernel
__device__ __forceinline__ void mma_tf32_k4_first(float (&d)[4], unsigned a0, unsigned a1, unsigned b0) {
  asm volatile("mma.sync.aligned.m16n8k4.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%7,%7,%7,%7};"
               : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
               : "r"(a0), "r"(a1), "r"(b0), "f"(0.f));
}

// Columns (= rows of the transposed tile) of X: parameters 0..P-1, zeros, and sqrt(w) r in the last one.  P <= 7 fits
// ONE 8-column tile: half the MMAs (n-tile 0 only, the A rows 8..15 are don't-care) and half the shared memory.
// (Measured for the 6-parameter camera model, 50 M observations: 0.98 ms against 0.75 ms on dense_pass_kernel — with
// so few columns the shared-memory round trip and the legacy-rate HMMA cost more than the FFMAs they replace, so that
// model stays on the register kernel; the narrow tile is kept for run-time compiled models with 7 < packed size.)
__host__ __device__ constexpr int wide_tc_cols(int P) { return P + 1 <= 8 ? 8 : 16; }
__host__ __device__ constexpr int wide_tc_row(int O) { return 64 * O + 4; }  // floats per parameter row of a warp tile: == 4 mod 32 (ldmatrix conflict-free)
__host__ __device__ constexpr size_t wide_tc_smem_bytes(int O, int setn, int P, int threads) {
  return size_t(4) * (size_t(threads / 32) * wide_tc_cols(P) * wide_tc_row(O) + size_t(1 + 2 * P) * ((setn + 3) / 4 * 4) + P) + 16;
}

template <class M, int THREADS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB) wide_tc_kernel(const PassArgs a) {
  const int mode = a.mode_override >= 0 ? a.mode_override : *a.mode_ptr;
  if (mode == PASS_SKIP) return;
  if (peer_failed(a)) return;
  constexpr int P = M::P, O = M::O, NS = M::NS;
  static_assert(P + 1 <= 16, "wide_tc_kernel: at most 15 parameters (one 16 x 16 Gram tile)");
  constexpr int kWideTcCols = wide_tc_cols(P);
  constexpr int NTILES = kWideTcCols / 8;       // 8-column output tiles of the m16n8 MMA
  constexpr int NRAW = P * (P + 1) / 2 + P + 1;
  constexpr int NCH = (NRAW + 31) / 32;
  constexpr int STRIDE = NCH * 32;
  constexpr int NW = THREADS / 32;
  constexpr int ROW = wide_tc_row(O);
  constexpr int KSTEPS = 8 * O;                 // k-steps of 8 residual rows over the warp's 64 observations
  constexpr int FLUSH_GROUPS = 4;               // the fp32 accumulators are folded into fp64 every 4 * 64 observations
  constexpr int NSETS = 1 + 2 * P;
  constexpr int SETN = (M::SETN + 3) / 4 * 4;
  constexpr int S1P = WideStage<M>::PARAMS;
  constexpr int NTMP = WideStage<M>::NT;
  constexpr int NAFF = M::NAFF;

  extern __shared__ __align__(16) unsigned char wide_tc_smem[];
  float* s_x = reinterpret_cast<float*>(wide_tc_smem);          // [NW][kWideTcCols][ROW]
  float* s_sets = s_x + size_t(NW) * kWideTcCols * ROW;         // [NSETS][SETN]
  float* s_h = s_sets + NSETS * SETN;                           // [P]: the step actually taken, H_j
  __shared__ double s_warp[NW * STRIDE];
  __shared__ double s_tot[STRIDE];

  const bool central = (a.cost->jacobian == MOPT_JAC_CENTRAL);
  const int nsets = central ? 1 + 2 * P : 1 + P;
  for (int i = threadIdx.x; i < nsets * SETN; i += THREADS) {
    const int si = i / SETN, k = i % SETN;
    double v = (k < M::SETN) ? a.pb->sets[si][k] : 0.0;
    if (si >= 1 && si <= P && k < M::SETN) {  // D_j = (set(x + h_j e_j) - set_ref) / H_j, in fp64 (AFFINE_FD)
      const int j = si - 1;
      v = central ? (v - a.pb->sets[1 + P + j][k]) / a.pb->hstep_cen[j] : (v - a.pb->sets[0][k]) / a.pb->hstep_fwd[j];
    }
    s_sets[i] = float(v);
  }
  for (int i = threadIdx.x; i < P; i += THREADS) s_h[i] = float(central ? a.pb->hstep_cen[i] : a.pb->hstep_fwd[i]);
  for (int i = threadIdx.x; i < NW * kWideTcCols * ROW; i += THREADS) s_x[i] = 0.f;  // unused columns stay zero
  for (int i = threadIdx.x; i < NW * STRIDE; i += THREADS) s_warp[i] = 0.0;
  const int loss = a.cost->loss;
  const float lossp = float(a.cost->loss_param);
  __syncthreads();

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* tile = s_x + size_t(warp) * kWideTcCols * ROW;
  const float* __restrict__ sp[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) sp[s] = static_cast<const float*>(a.streams.p[s]);

  // a parameter set as broadcast pairs (the compiler turns F2(x, x) into FFMA2's scalar operand)
  auto load_set = [&](int idx, F2 (&sr)[SETN]) {
#pragma unroll
    for (int k = 0; k < SETN; k += 4) {
      const float4 t = *reinterpret_cast<const float4*>(s_sets + idx * SETN + k);
      sr[k] = F2(t.x); sr[k + 1] = F2(t.y); sr[k + 2] = F2(t.z); sr[k + 3] = F2(t.w);
    }
  };

  // fp32 accumulators, n-tile 0 / 1 of the m16n8 output fragments: S = X_hi^T X_hi and T = X_hi^T X_lo
  float cs[NTILES][4], ct[NTILES][4];
  double ds[NTILES][4], dt[NTILES][4];
#pragma unroll
  for (int t = 0; t < NTILES; ++t)
#pragma unroll
    for (int q = 0; q < 4; ++q) { cs[t][q] = 0.f; ct[t][q] = 0.f; ds[t][q] = 0.0; dt[t][q] = 0.0; }
  F2 acc_e2(0.f);
  double dacc_e2 = 0.0;

  // ldmatrix row address of this lane: matrix (lane / 8) = rows 0-7 | 8-15 of X at k columns +0 | +4 (with one
  // 8-row tile the "rows 8-15" matrices re-read rows 0-7: they only feed output rows nobody reads)
  const float* ld_base = tile + ((lane & 7) + (NTILES == 2 ? 8 * ((lane >> 3) & 1) : 0)) * ROW + 4 * (lane >> 4);

  const int64_t ngroups = (a.n + 63) / 64;
  const int64_t wstride = int64_t(gridDim.x) * NW;
  int since_flush = 0;
  // this lane's two observations of group g; past the end (last group only) the store's last observation is re-read,
  // its weight is forced to 0 below
  auto load_obs = [&](int64_t g, F2 (&e)[NS]) {
    const int64_t i0 = g * 64 + 2 * lane;
    if (i0 + 1 < a.n) {
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        const float2 t = *reinterpret_cast<const float2*>(sp[s] + i0);
        e[s] = F2(t.x, t.y);
      }
    } else {
      const int64_t j0 = i0 < a.n ? i0 : a.n - 1;
#pragma unroll
      for (int s = 0; s < NS; ++s) e[s] = F2(sp[s][j0], sp[s][a.n - 1]);
    }
  };
  // The next group's observations are requested before this group's tensor-core phase: the first instruction that
  // used them was 10 % of all stall samples of the kernel (ncu source page, one FFMA2 waiting for the global loads).
  F2 e_next[NS];
  {
    const int64_t g_first = int64_t(blockIdx.x) * NW + warp;
    if (g_first < ngroups) load_obs(g_first, e_next);
  }
  for (int64_t g = int64_t(blockIdx.x) * NW + warp; g < ngroups; g += wstride) {
    const int64_t i0 = g * 64 + 2 * lane;
    const bool v0 = i0 < a.n, v1 = i0 + 1 < a.n;
    // ---- 1. this lane's two observations --------------------------------------------------------------------
    F2 e[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) e[s] = e_next[s];
    F2 r[O], tmp[NTMP], s0[SETN];
    load_set(0, s0);
    if constexpr (S1P < P) {
      M::template stage1<F2>(s0, e, tmp);
      M::template stage2<F2>(s0, e, tmp, r);
    } else {
      M::template residual<F2>(s0, e, r);
    }
    F2 e2(0.f);
#pragma unroll
    for (int o = 0; o < O; ++o) e2 = fma(r[o], r[o], e2);
    if (!v0) e2.v.x = 0.f;
    if (!v1) e2.v.y = 0.f;
    acc_e2 = acc_e2 + e2;
    if (mode != PASS_COST) {
      F2 sw;  // sqrt of the IRLS weight (loss_function.h:16 contract): H = sum (sqrt(w) J)^T (sqrt(w) J)
      if (loss == MOPT_LOSS_NONE) {
        sw = F2(1.f);
      } else {
        const float w0 = loss_weight<float>(loss, lossp, e2.v.x), w1 = loss_weight<float>(loss, lossp, e2.v.y);
        float q0, q1;
        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(q0) : "f"(w0));
        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(q1) : "f"(w1));
        sw = F2(q0, q1);
      }
      if (!v0) sw.v.x = 0.f;
      if (!v1) sw.v.y = 0.f;
      float* my = tile + 2 * lane;  // + p * ROW + o * 64: the pair (observation 2 lane, 2 lane + 1) of row (o, p)
      F2 u0[NAFF];
      M::template affine<F2>(s0, e, u0);
#pragma unroll
      for (int j = 0; j < S1P; ++j) {
        F2 du[NAFF], d[O], sr[SETN];
        load_set(1 + j, sr);
        M::template affine<F2>(sr, e, du);
        if (central) {
          F2 um[NAFF];
          load_set(1 + P + j, sr);
          M::template affine<F2>(sr, e, um);
          M::template finish_diff<F2>(s0, um, du, F2(s_h[j]), e, d);
        } else {
          M::template finish_diff<F2>(s0, u0, du, F2(s_h[j]), e, d);
        }
#pragma unroll
        for (int o = 0; o < O; ++o) *reinterpret_cast<float2*>(my + j * ROW + o * 64) = (sw * d[o]).v;
      }
      if constexpr (S1P < P) {
        F2 Jt[O * (P - S1P)];
        M::template tail_partials<F2>(s0, tmp, Jt);
#pragma unroll
        for (int o = 0; o < O; ++o)
#pragma unroll
          for (int k = 0; k < P - S1P; ++k)
            *reinterpret_cast<float2*>(my + (S1P + k) * ROW + o * 64) = (sw * Jt[o * (P - S1P) + k]).v;
      }
#pragma unroll
      for (int o = 0; o < O; ++o) *reinterpret_cast<float2*>(my + (kWideTcCols - 1) * ROW + o * 64) = (sw * r[o]).v;
      __syncwarp();
      if (g + wstride < ngroups) load_obs(g + wstride, e_next);
      // ---- 2. Gram matrix of the tile on the tensor cores: C += X^T X, 3 x TF32 ------------------------------
      // The tensor core's fp32 accumulation truncates: a chain of n dependent MMAs on one accumulator biases a sum of
      // same-signed products (the diagonal of H) low by ~n * 2^-25 relative (measured: 5.3e-6 / 3.2e-6 / 2.3e-6 of
      // sqrt(H_ii H_jj) with the accumulators folded every 4 / 2 / 1 groups, profiles/r2_wide_tc_study.txt).  So the
      // large term S is accumulated in chains of 4 MMAs (two k-steps) that start from zero and are then added to the
      // running sums with ordinary round-to-nearest FADDs; T is 2^-11 of S and keeps the long chain.
      static_assert(KSTEPS % 2 == 0, "k-steps are processed in pairs");
#pragma unroll 2
      for (int ks = 0; ks < KSTEPS; ks += 2) {
        float ps[NTILES][4];
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
          unsigned x[4], hi[4];
          float lo[4];
          ldmatrix_x4(ld_base + (ks + kk) * 8, x);  // x0, x1: rows g, g + 8 at k = t;  x2, x3: the same rows at k = t + 4
#pragma unroll
          for (int q = 0; q < 4; q += (NTILES == 2 ? 1 : 2)) split_tf32(x[q], hi[q], lo[q]);
          if constexpr (NTILES == 1) { hi[1] = 0u; hi[3] = 0u; }
#pragma unroll
          for (int h = 0; h < 2; ++h) {  // the two k4 halves of this k-step
            if (kk == 0 && h == 0) {
              mma_tf32_k4_first(ps[0], hi[0], hi[1], hi[0]);
              if constexpr (NTILES == 2) mma_tf32_k4_first(ps[1], hi[0], hi[1], hi[1]);
            } else {
              mma_tf32_k4(ps[0], hi[2 * h], hi[2 * h + 1], hi[2 * h]);
              if constexpr (NTILES == 2) mma_tf32_k4(ps[1], hi[2 * h], hi[2 * h + 1], hi[2 * h + 1]);
            }
            mma_tf32_k4(ct[0], hi[2 * h], hi[2 * h + 1], __float_as_uint(lo[2 * h]));
            if constexpr (NTILES == 2) mma_tf32_k4(ct[1], hi[2 * h], hi[2 * h + 1], __float_as_uint(lo[2 * h + 1]));
          }
        }
#pragma unroll
        for (int t = 0; t < NTILES; ++t)
#pragma unroll
          for (int q = 0; q < 4; ++q) cs[t][q] += ps[t][q];
      }
      __syncwarp();
    } else if (g + wstride < ngroups) {
      load_obs(g + wstride, e_next);  // cost-only pass: no tensor-core phase to put the loads in front of
    }
    if (++since_flush >= FLUSH_GROUPS) {
#pragma unroll
      for (int t = 0; t < NTILES; ++t)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          ds[t][q] += double(cs[t][q]); cs[t][q] = 0.f;
          dt[t][q] += double(ct[t][q]); ct[t][q] = 0.f;
        }
      dacc_e2 += double(acc_e2.v.x) + double(acc_e2.v.y);
      acc_e2 = F2(0.f);
      since_flush = 0;
    }
  }
#pragma unroll
  for (int t = 0; t < NTILES; ++t)
#pragma unroll
    for (int q = 0; q < 4; ++q) { ds[t][q] += double(cs[t][q]); dt[t][q] += double(ct[t][q]); }
  dacc_e2 += double(acc_e2.v.x) + double(acc_e2.v.y);

  // fragment element (t, q): row i = lane / 4 + 8 (q / 2), column j = 8 t + 2 (lane % 4) + (q % 2).  X^T X =
  // S + T + T^T: every lane parks its T entries in the warp's (now idle) tile, then adds T(i, j) + T(j, i) to its S
  // entries; every needed entry of the packed layout (H upper row-major, b, sum) has exactly one owner lane.
  __syncwarp();
  double* tt = reinterpret_cast<double*>(tile);  // [16][16] (rows / columns >= kWideTcCols hold don't-care values)
#pragma unroll
  for (int t = 0; t < NTILES; ++t)
#pragma unroll
    for (int q = 0; q < 4; ++q) tt[((lane >> 2) + 8 * (q >> 1)) * 16 + 8 * t + 2 * (lane & 3) + (q & 1)] = dt[t][q];
  __syncwarp();
  double* mine = s_warp + warp * STRIDE;
#pragma unroll
  for (int t = 0; t < NTILES; ++t)
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int i = (lane >> 2) + 8 * (q >> 1), j = 8 * t + 2 * (lane & 3) + (q & 1);
      if (i >= kWideTcCols) continue;
      const double v = ds[t][q] + (tt[i * 16 + j] + tt[j * 16 + i]);
      if (i < P && j < P && i <= j) mine[tri_index(P, i, j)] = v;
      else if (i < P && j == kWideTcCols - 1) mine[P * (P + 1) / 2 + i] = v;
    }
  {  // sum r^T r: the warp's lanes in a fixed order
    double s = dacc_e2;
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) s += shfl_xor(s, off);
    if (lane == 0) mine[NRAW - 1] = s;
  }
  __syncthreads();

  if (!grid_reduce_shared<NRAW, STRIDE, THREADS>(a, s_tot, s_warp)) return;
  if (mode == PASS_COST) {
    if (threadIdx.x == 0) a.out->v[NRAW - 1] = a.accumulate ? a.out->v[NRAW - 1] + s_tot[NRAW - 1] : s_tot[NRAW - 1];
  } else {
    for (int i = threadIdx.x; i < NRAW; i += THREADS) a.out->v[i] = a.accumulate ? a.out->v[i] + s_tot[i] : s_tot[i];
  }
  peer_push(a, NRAW);
}

#endif  // __CUDACC__
}  // namespace mopt
