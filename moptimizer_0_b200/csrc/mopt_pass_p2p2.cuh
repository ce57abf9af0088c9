// Point-to-point moment kernel, fp32 streams + fp32 compute, second generation (the headline kernel):
//   * the six planar streams travel HBM -> shared memory by TMA bulk copies (cp.async.bulk, SASS UBLKCP) into a
//     ring of STAGES stages per CTA, completion on mbarriers.  The bytes in flight per SM are the ring (up to
//     ~190 KB), no longer "registers per thread x resident threads", so the compute side is free to use 128
//     registers per thread;
//   * the arithmetic is packed fp32 (fma/add/mul .f32x2 -> SASS FFMA2 / FADD2 / FMUL2): the two correspondences of
//     each half of a float4 are processed by one instruction stream, constants enter as broadcast scalars
//     (FFMA2's .F32 operand), the 23 moment accumulators are register pairs (even / odd correspondence) that are
//     added together at every fp64 flush.
// Same moments, same raw layout, same reductions and epilogue (p2p_finish) as p2p_moment_kernel in mopt_pass.cuh,
// which stays the kernel of the fp64-compute paths.  Replaces the loop of CostComputation::computeHessian
// (include/moptimizer/linearization.h:126-158) for the model of tst/point2point.cpp:24-84.
#pragma once

#include "mopt_pass.cuh"

namespace mopt {
#ifdef __CUDACC__

// ---- packed fp32 helpers ------------------------------------------------------------------------------------
__device__ __forceinline__ float2 bc2(float a) { return make_float2(a, a); }  // becomes FFMA2's scalar .F32 operand
__device__ __forceinline__ float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }  // folds into an operand modifier
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, neg2(b)); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }

// ---- mbarrier / bulk-copy helpers ---------------------------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "MOPT_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra MOPT_DONE;\n"
      "bra MOPT_WAIT;\n"
      "MOPT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// TMA bulk copy global -> shared (1-D, `bytes` a multiple of 16, both addresses 16-byte aligned); completes on `bar`.
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// IRLS weight (loss_function.h:16 contract) with the loss kind known at compile time.  Huber: one MUFU.RSQ without
// rsqrtf's denormal rescaling (6 more instructions per correspondence); e2 is clamped to the smallest normal float,
// which only matters for k < 1.1e-19 (a denormal e2 cannot exceed k^2 otherwise).
template <int LOSS>
__device__ __forceinline__ float loss_weight_fast(float k, float e2) {
  if constexpr (LOSS == MOPT_LOSS_HUBER) {
    float rs;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rs) : "f"(fmaxf(e2, 1.17549435e-38f)));
    return (e2 <= k * k) ? 1.0f : k * rs;
  } else {
    return loss_weight<float>(LOSS, k, e2);
  }
}

// ---- two correspondences at a time ---------------------------------------------------------------------------
// Same operations, in the same order per correspondence, as p2p_moments (mopt_pass.cuh); lane .x / .y of every
// float2 belongs to the even / odd correspondence of the pair.
template <int LOSS, bool QROT, bool MASKED>
__device__ __forceinline__ void p2p_moments_x2(const float (&R)[9], const float (&t)[3], float lossp, float2 px, float2 py,
                                               float2 pz, float2 yx, float2 yy, float2 yz, float2 (&acc)[kP2PRaw]) {
  bool skip0 = false, skip1 = false;
  if constexpr (MASKED) {  // NaN target = no correspondence (f returned false, linearization.h:102,144): contributes nothing
    skip0 = yx.x != yx.x; skip1 = yx.y != yx.y;
    if (skip0) { px.x = py.x = pz.x = 0.f; yx.x = t[0]; yy.x = t[1]; yz.x = t[2]; }  // q = 0 and r = (0 + t) - t = 0
    if (skip1) { px.y = py.y = pz.y = 0.f; yx.y = t[0]; yy.y = t[1]; yz.y = t[2]; }
  }
  // q = R p ; r = (q + t) - y          (tst/point2point.cpp:41-44)
  const float2 q0 = fma2(px, bc2(R[0]), fma2(py, bc2(R[1]), mul2(pz, bc2(R[2]))));
  const float2 q1 = fma2(px, bc2(R[3]), fma2(py, bc2(R[4]), mul2(pz, bc2(R[5]))));
  const float2 q2 = fma2(px, bc2(R[6]), fma2(py, bc2(R[7]), mul2(pz, bc2(R[8]))));
  const float2 r0 = sub2(add2(q0, bc2(t[0])), yx);
  const float2 r1 = sub2(add2(q1, bc2(t[1])), yy);
  const float2 r2 = sub2(add2(q2, bc2(t[2])), yz);
  const float2 e2 = fma2(r0, r0, fma2(r1, r1, mul2(r2, r2)));
  float2 w;
  w.x = loss_weight_fast<LOSS>(lossp, e2.x);
  w.y = loss_weight_fast<LOSS>(lossp, e2.y);
  if constexpr (MASKED) {
    if (skip0) w.x = 0.f;
    if (skip1) w.y = 0.f;
  }
  const float2 a0 = QROT ? q0 : px, a1 = QROT ? q1 : py, a2 = QROT ? q2 : pz;
  const float2 w0 = mul2(w, a0), w1 = mul2(w, a1), w2 = mul2(w, a2);
  acc[0] = add2(acc[0], w);
  acc[1] = add2(acc[1], w0); acc[2] = add2(acc[2], w1); acc[3] = add2(acc[3], w2);
  acc[4] = fma2(w0, a0, acc[4]); acc[5] = fma2(w0, a1, acc[5]); acc[6] = fma2(w0, a2, acc[6]);
  acc[7] = fma2(w1, a1, acc[7]); acc[8] = fma2(w1, a2, acc[8]); acc[9] = fma2(w2, a2, acc[9]);
  acc[10] = fma2(w, r0, acc[10]); acc[11] = fma2(w, r1, acc[11]); acc[12] = fma2(w, r2, acc[12]);
  acc[13] = fma2(w0, r0, acc[13]); acc[14] = fma2(w0, r1, acc[14]); acc[15] = fma2(w0, r2, acc[15]);
  acc[16] = fma2(w1, r0, acc[16]); acc[17] = fma2(w1, r1, acc[17]); acc[18] = fma2(w1, r2, acc[18]);
  acc[19] = fma2(w2, r0, acc[19]); acc[20] = fma2(w2, r1, acc[20]); acc[21] = fma2(w2, r2, acc[21]);
  acc[22] = add2(acc[22], e2);
}

template <bool MASKED>
__device__ __forceinline__ void p2p_cost_x2(const float (&R)[9], const float (&t)[3], float2 px, float2 py, float2 pz,
                                            float2 yx, float2 yy, float2 yz, float2 (&acc)[kP2PRaw]) {
  const float2 r0 = sub2(add2(fma2(px, bc2(R[0]), fma2(py, bc2(R[1]), mul2(pz, bc2(R[2])))), bc2(t[0])), yx);
  const float2 r1 = sub2(add2(fma2(px, bc2(R[3]), fma2(py, bc2(R[4]), mul2(pz, bc2(R[5])))), bc2(t[1])), yy);
  const float2 r2 = sub2(add2(fma2(px, bc2(R[6]), fma2(py, bc2(R[7]), mul2(pz, bc2(R[8])))), bc2(t[2])), yz);
  float2 e2 = fma2(r0, r0, fma2(r1, r1, mul2(r2, r2)));
  if constexpr (MASKED) {
    if (yx.x != yx.x) e2.x = 0.f;
    if (yx.y != yx.y) e2.y = 0.f;
  }
  acc[22] = add2(acc[22], e2);
}

// Shared-memory footprint of the ring: STAGES x 6 streams x (U * THREADS) float4.
constexpr size_t p2p2_ring_bytes(int threads, int stages, int u) { return size_t(stages) * 6 * size_t(u) * threads * 16; }

// U: float4 groups per thread per stream per round.
template <int LOSS, bool QROT, bool MASKED, bool FUSED, int THREADS, int MINB, int STAGES, int U, int FLUSH_ROUNDS>
__global__ void __launch_bounds__(THREADS, MINB) p2p_moment2_kernel(const PassArgs a) {
  static_assert(STAGES > 0, "p2p_moment2_kernel: the ring needs at least one stage");
  const int mode = a.mode_override >= 0 ? a.mode_override : *a.mode_ptr;
  if (mode == PASS_SKIP) return;
  if (peer_failed(a)) return;
  constexpr int NW = THREADS / 32;
  constexpr int CHUNK = THREADS * U;  // float4 groups per stream per CTA per round

  __shared__ double s_warp[NW * 32];
  __shared__ double s_tot[32];
  __shared__ double s_set0[FUSED ? 12 : 1];
  __shared__ __align__(8) uint64_t s_full[STAGES];
  __shared__ __align__(8) uint64_t s_empty[STAGES];
  extern __shared__ __align__(128) unsigned char p2p2_ring[];
  float4* ring = reinterpret_cast<float4*>(p2p2_ring);  // [STAGES][6][CHUNK]

  const int lane = threadIdx.x & 31;
  const double* set0 = FUSED ? s_set0 : a.pb->sets[0];
  if constexpr (FUSED) {
    if (threadIdx.x == 0) {
      double xl[6];  // a copy: taking the address of a kernel parameter would spill the whole PassArgs to local memory
#pragma unroll
      for (int i = 0; i < 6; ++i) xl[i] = a.x.v[i];
      p2p_fused_set0(a.cost, xl, s_set0);
    }
  }
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&s_full[s], 1);
      mbar_init(&s_empty[s], NW);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  const float* __restrict__ sp[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) sp[k] = static_cast<const float*>(a.streams.p[k]);

  const int64_t ngroups = a.n / 4;
  const int64_t stride = int64_t(gridDim.x) * CHUNK;   // groups per round over the whole grid
  const int64_t full_rounds = a.no_ring ? 0 : ngroups / stride;

  // producer (thread 0): the CTA's 6 x CHUNK x 16 B slices of round rr into stage rr % STAGES
  auto issue_to = [&](int64_t rr, int s) {
    const int64_t g = rr * stride + int64_t(blockIdx.x) * CHUNK;
    mbar_expect_tx(&s_full[s], 6u * CHUNK * 16u);
#pragma unroll
    for (int k = 0; k < 6; ++k)
      bulk_g2s(ring + (size_t(s) * 6 + k) * CHUNK, reinterpret_cast<const float4*>(sp[k]) + g, CHUNK * 16u, &s_full[s]);
  };
  if (threadIdx.x == 0)
    for (int rr = 0; rr < STAGES && rr < full_rounds; ++rr) issue_to(rr, rr);

  float R[9], t[3];
#pragma unroll
  for (int i = 0; i < 9; ++i) R[i] = float(set0[i]);
#pragma unroll
  for (int i = 0; i < 3; ++i) t[i] = float(set0[9 + i]);
  const float lossp = float(a.cost->loss_param);

  float2 acc[kP2PRaw];
#pragma unroll
  for (int i = 0; i < kP2PRaw; ++i) acc[i] = make_float2(0.f, 0.f);
  double dacc[1] = {0.0};

  // All 32 lanes of the warp must call flush() together: warp_reduce_transpose is a full-mask shuffle.
  auto flush = [&]() {
    float s[32];
#pragma unroll
    for (int i = 0; i < kP2PRaw; ++i) s[i] = acc[i].x + acc[i].y;
#pragma unroll
    for (int i = kP2PRaw; i < 32; ++i) s[i] = 0.f;
    const float v = warp_reduce_transpose<32>(s);
    dacc[0] += double(v);
#pragma unroll
    for (int i = 0; i < kP2PRaw; ++i) acc[i] = make_float2(0.f, 0.f);
  };

  auto consume = [&](const float4 (&v)[6]) {
    if (mode == PASS_COST) {
      p2p_cost_x2<MASKED>(R, t, make_float2(v[0].x, v[0].y), make_float2(v[1].x, v[1].y), make_float2(v[2].x, v[2].y),
                          make_float2(v[3].x, v[3].y), make_float2(v[4].x, v[4].y), make_float2(v[5].x, v[5].y), acc);
      p2p_cost_x2<MASKED>(R, t, make_float2(v[0].z, v[0].w), make_float2(v[1].z, v[1].w), make_float2(v[2].z, v[2].w),
                          make_float2(v[3].z, v[3].w), make_float2(v[4].z, v[4].w), make_float2(v[5].z, v[5].w), acc);
    } else {
      p2p_moments_x2<LOSS, QROT, MASKED>(R, t, lossp, make_float2(v[0].x, v[0].y), make_float2(v[1].x, v[1].y),
                                         make_float2(v[2].x, v[2].y), make_float2(v[3].x, v[3].y),
                                         make_float2(v[4].x, v[4].y), make_float2(v[5].x, v[5].y), acc);
      p2p_moments_x2<LOSS, QROT, MASKED>(R, t, lossp, make_float2(v[0].z, v[0].w), make_float2(v[1].z, v[1].w),
                                         make_float2(v[2].z, v[2].w), make_float2(v[3].z, v[3].w),
                                         make_float2(v[4].z, v[4].w), make_float2(v[5].z, v[5].w), acc);
    }
  };
  auto direct_group = [&](int64_t g) {
    float4 v[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) v[k] = ld_stream(reinterpret_cast<const float4*>(sp[k]) + g);
    consume(v);
  };

  int since_flush = 0;
  // stage index and phase parity advance incrementally (no 64-bit division per round)
  int s = 0;
  unsigned ph = 0;
  const float4* st = ring + threadIdx.x;
  for (int64_t r = 0; r < full_rounds; ++r) {
    mbar_wait(&s_full[s], ph);
    float4 v[U][6];
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
      for (int k = 0; k < 6; ++k) v[u][k] = st[(s * 6 + k) * CHUNK + u * THREADS];
    // the stage is in registers: hand it back (one arrival per warp), thread 0 refills it for round r + STAGES
    __syncwarp();
    if (lane == 0) mbar_arrive(&s_empty[s]);
    if (threadIdx.x == 0 && r + STAGES < full_rounds) {
      mbar_wait(&s_empty[s], ph);
      issue_to(r + STAGES, s);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) consume(v[u]);
    if (++since_flush >= FLUSH_ROUNDS) {
      flush();
      since_flush = 0;
    }
    if (++s == STAGES) {
      s = 0;
      ph ^= 1u;
    }
  }
  {  // ragged remainder (< one grid round of groups) + scalar tail (n % 4 residuals)
    for (int64_t g = full_rounds * stride + int64_t(blockIdx.x) * THREADS + threadIdx.x; g < ngroups;
         g += int64_t(gridDim.x) * THREADS) {
      direct_group(g);
      // a warp's lanes hold g = 32 w .. 32 w + 31, so (g | 31) is its last lane's: where that lane has no group this is
      // the warp's last iteration and only some of its lanes are here, so the flush after the loop takes this one
      if (++since_flush >= FLUSH_ROUNDS && (g | 31) < ngroups) {
        flush();
        since_flush = 0;
      }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      for (int64_t i = ngroups * 4; i < a.n; ++i) {
        // one correspondence in lane .x; lane .y is a dummy (p = 0, y = t) whose sums are discarded
        float2 one[kP2PRaw];
#pragma unroll
        for (int k = 0; k < kP2PRaw; ++k) one[k] = make_float2(0.f, 0.f);
        const float2 px = make_float2(sp[0][i], 0.f), py = make_float2(sp[1][i], 0.f), pz = make_float2(sp[2][i], 0.f);
        const float2 yx = make_float2(sp[3][i], t[0]), yy = make_float2(sp[4][i], t[1]), yz = make_float2(sp[5][i], t[2]);
        if (mode == PASS_COST) p2p_cost_x2<MASKED>(R, t, px, py, pz, yx, yy, yz, one);
        else p2p_moments_x2<LOSS, QROT, MASKED>(R, t, lossp, px, py, pz, yx, yy, yz, one);
#pragma unroll
        for (int k = 0; k < kP2PRaw; ++k) acc[k].x += one[k].x;
      }
    }
  }
  flush();
  p2p_finish<FUSED, THREADS>(a, mode, dacc, s_tot, s_warp);
}

#endif  // __CUDACC__
}  // namespace mopt
