// Finite-difference pass of the small models with an affine first stage (the 6-parameter pinhole camera of
// tst/camera_calibration.cpp), fp32 store + fp32 compute, second generation: every thread evaluates TWO observations at
// once in packed fp32 (F2, mopt_pass_wide_tc.cuh: fma / add / mul .f32x2), the model's hooks (affine / finish /
// finish_diff) instantiated for F2, parameter sets re-read from shared memory as broadcast scalars.  The packed
// upper-triangular H, b and sum r^T r are accumulated in register PAIRS (even / odd observation) and folded into fp64
// by the transposing warp reduction, exactly like dense_pass_kernel (mopt_pass.cuh), whose common-denominator
// difference quotient (AFFINE_FD) this kernel evaluates: same formulas, half the instruction stream per observation.
// Identity covariance, no NaN-masked stores (both take dense_pass_kernel).  Replaces the loop of
// computeHessianNumerical (include/moptimizer/linearization.h:65-124).
#pragma once

#include <type_traits>

#include "mopt_pass_wide_tc.cuh"
#include "mopt_setup.cuh"

namespace mopt {
#ifdef __CUDACC__

// model->setup(x) and the finite-difference sets inside the pass kernel (PassArgs::fused_setup; host-driven passes of
// parameter-only models, where a set is x +- h e_j and the separate one-warp set-up kernel plus its dependent launch
// are a third of a 10 M-sample step): the CTA's first warp fills a ParamBlock in shared memory exactly as
// setup_kernel does in global memory.  One copy per translation unit.
static __device__ __noinline__ void dense_fused_setup(const CostDev* c, XArg x, ParamBlock* pb, int lane) {
  setup_cost(*c, x.v, pb, lane, 32);
}

template <class M, int THREADS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB) dense_f2_kernel(const PassArgs a) {
  const int mode = a.mode_override >= 0 ? a.mode_override : *a.mode_ptr;
  if (mode == PASS_SKIP) return;
  if (peer_failed(a)) return;
  constexpr int P = M::P, O = M::O, NS = M::NS, NAFF = M::NAFF;
  constexpr int NRAW = P * (P + 1) / 2 + P + 1;
  constexpr int V = next_pow2(NRAW);
  static_assert(V <= 32, "dense_f2_kernel: packed size must fit one transposing-reduce chunk");
  constexpr int FLUSH_ROUNDS = 8;   // fp32 pair partials are folded into fp64 every 8 rounds (32 observations per thread)
  constexpr int NSETS = 1 + 2 * P;
  constexpr int SETN = (M::SETN + 3) / 4 * 4;

  __shared__ double s_warp[(THREADS / 32) * V];
  __shared__ double s_tot[V];
  __shared__ __align__(16) float s_sets[NSETS][SETN];
  __shared__ float s_h[P];

  // fused set-up: parameter-only models (the host asks for it only for those, can_fuse_setup in mopt_capi.cu)
  constexpr bool kCanFuse = (P <= 2);
  __shared__ typename std::conditional<kCanFuse, ParamBlock, char>::type s_pb;
  const ParamBlock* pb = a.pb;
  if constexpr (kCanFuse) {
    if (a.fused_setup) {
      if (threadIdx.x < 32) dense_fused_setup(a.cost, a.x, &s_pb, threadIdx.x);
      __syncthreads();
      pb = &s_pb;
    }
  }
  const bool central = (a.cost->jacobian == MOPT_JAC_CENTRAL);
  const int nsets = central ? 1 + 2 * P : 1 + P;
  for (int i = threadIdx.x; i < nsets * SETN; i += THREADS) {
    const int si = i / SETN, k = i % SETN;
    double v = (k < M::SETN) ? pb->sets[si][k] : 0.0;
    if (si >= 1 && si <= P && k < M::SETN) {  // D_j = (set(x + h_j e_j) - set_ref) / H_j, in fp64
      const int j = si - 1;
      v = central ? (v - pb->sets[1 + P + j][k]) / pb->hstep_cen[j] : (v - pb->sets[0][k]) / pb->hstep_fwd[j];
    }
    s_sets[si][k] = float(v);
  }
  for (int i = threadIdx.x; i < P; i += THREADS) s_h[i] = float(central ? pb->hstep_cen[i] : pb->hstep_fwd[i]);
  const int loss = a.cost->loss;
  const float lossp = float(a.cost->loss_param);
  __syncthreads();

  const float* __restrict__ sp[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) sp[s] = static_cast<const float*>(a.streams.p[s]);

  F2 acc[NRAW];
#pragma unroll
  for (int i = 0; i < NRAW; ++i) acc[i] = F2(0.f);
  double dacc[1] = {0.0};

  // All 32 lanes of the warp must call flush() together: warp_reduce_transpose is a full-mask shuffle.
  auto flush = [&]() {
    float s[V];
#pragma unroll
    for (int i = 0; i < NRAW; ++i) s[i] = acc[i].v.x + acc[i].v.y;
#pragma unroll
    for (int i = NRAW; i < V; ++i) s[i] = 0.f;
    const float v = warp_reduce_transpose<V>(s);
    dacc[0] += double(v);
#pragma unroll
    for (int i = 0; i < NRAW; ++i) acc[i] = F2(0.f);
  };
  // a parameter set as broadcast pairs, re-read at every use (an asm volatile load the compiler cannot hoist: the
  // 1 + 2P sets do not fit in registers next to J and the accumulators)
  // (small models — P <= 2, SETN <= 4 — keep all 1 + 2P sets in registers instead: 20 values for the exp curve)
  constexpr bool kSetsInRegs = (P <= 2 && SETN <= 4);
  float sreg[kSetsInRegs ? NSETS : 1][kSetsInRegs ? SETN : 1];
  if constexpr (kSetsInRegs) {
#pragma unroll
    for (int i = 0; i < NSETS; ++i)
#pragma unroll
      for (int k = 0; k < SETN; ++k) sreg[i][k] = (i < nsets) ? s_sets[i][k] : 0.f;
  }
  auto load_set = [&](int idx, F2 (&sr)[SETN]) {
    if constexpr (kSetsInRegs) {
#pragma unroll
      for (int k = 0; k < SETN; ++k) sr[k] = F2(sreg[idx][k]);
    } else {
#pragma unroll
      for (int k = 0; k < SETN; k += 4) {
        float t[4];
        lds16_reload(&s_sets[idx][k], t);
        sr[k] = F2(t[0]); sr[k + 1] = F2(t[1]); sr[k + 2] = F2(t[2]); sr[k + 3] = F2(t[3]);
      }
    }
  };

  // two observations: lane .x / .y of every value; wx / wy = 0 drops a lane (scalar tail)
  auto do_pair = [&](const F2 (&e)[NS], bool valid_y) {
    F2 s0[SETN], u0[NAFF], r[O];
    load_set(0, s0);
    M::template affine<F2>(s0, e, u0);
    M::template finish<F2>(s0, u0, e, r);
    F2 e2(0.f);
#pragma unroll
    for (int o = 0; o < O; ++o) e2 = fma(r[o], r[o], e2);
    if (!valid_y) e2.v.y = 0.f;
    if (mode == PASS_COST) {
      acc[NRAW - 1] = acc[NRAW - 1] + e2;
      return;
    }
    F2 J[O * P];
#pragma unroll
    for (int j = 0; j < P; ++j) {
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
      for (int o = 0; o < O; ++o) J[o * P + j] = d[o];
    }
    F2 w(loss_weight<float>(loss, lossp, e2.v.x), loss_weight<float>(loss, lossp, e2.v.y));
    if (!valid_y) w.v.y = 0.f;
    int idx = 0;
#pragma unroll
    for (int i = 0; i < P; ++i) {
      F2 wj[O];
#pragma unroll
      for (int o = 0; o < O; ++o) wj[o] = w * J[o * P + i];
#pragma unroll
      for (int j = i; j < P; ++j) {
        F2 s = acc[idx];
#pragma unroll
        for (int o = 0; o < O; ++o) s = fma(wj[o], J[o * P + j], s);
        acc[idx] = s;
        ++idx;
      }
    }
#pragma unroll
    for (int i = 0; i < P; ++i) {
      F2 s = acc[idx];
#pragma unroll
      for (int o = 0; o < O; ++o) s = fma(w * J[o * P + i], r[o], s);
      acc[idx] = s;
      ++idx;
    }
    acc[NRAW - 1] = acc[NRAW - 1] + e2;
  };

  auto load_group = [&](int64_t g, float4 (&v)[NS]) {  // four consecutive observations of every stream
#pragma unroll
    for (int s = 0; s < NS; ++s) v[s] = ld_stream(reinterpret_cast<const float4*>(sp[s]) + g);
  };
  auto do_group = [&](const float4 (&v)[NS]) {  // two pairs
    F2 e[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) e[s] = F2(v[s].x, v[s].y);
    do_pair(e, true);
#pragma unroll
    for (int s = 0; s < NS; ++s) e[s] = F2(v[s].z, v[s].w);
    do_pair(e, true);
  };

  // Hiding the latency of the round's global loads:
  //   small models (exp curve: 80 registers) run a software pipeline in registers — the next round's loads are issued
  //     before this round is evaluated (ncu: long_scoreboard 36 % of the exp curve's stall time; 41.4 -> 39.5 us per 10 M);
  //   the camera model sits at its 128-register cap and loses to 20 more live registers (0.594 -> 0.636 ms), so its
  //     next round travels global -> shared memory by cp.async (LDGSTS: no registers) into the thread's own slot of a
  //     double buffer and is picked up with LDS.128 (long_scoreboard was 18 % of its stall time).
  constexpr bool kPipelined = (P <= 2);
  constexpr bool kStaged = !kPipelined;
  __shared__ float4 s_stage[kStaged ? 2 : 1][kStaged ? NS : 1][kStaged ? THREADS : 1];
  auto stage_group = [&](int buf, int64_t gg) {
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      const unsigned dst = static_cast<unsigned>(__cvta_generic_to_shared(&s_stage[buf][s][threadIdx.x]));
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(reinterpret_cast<const float4*>(sp[s]) + gg) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  const int64_t ngroups = a.n / 4;
  const int64_t stride = int64_t(gridDim.x) * THREADS;
  int since_flush = 0;
  int64_t g = int64_t(blockIdx.x) * THREADS + threadIdx.x;
  float4 v_next[NS];
  int buf = 0;
  if (g < ngroups) {
    if constexpr (kPipelined) load_group(g, v_next); else stage_group(0, g);
  }
  for (; g < ngroups; g += stride) {
    float4 v[NS];
    if constexpr (kPipelined) {
#pragma unroll
      for (int s = 0; s < NS; ++s) v[s] = v_next[s];
      if (g + stride < ngroups) load_group(g + stride, v_next);
    } else {
      if (g + stride < ngroups) {
        stage_group(buf ^ 1, g + stride);
        asm volatile("cp.async.wait_group 1;" ::: "memory");  // everything but the group just committed has landed
      } else {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      }
#pragma unroll
      for (int s = 0; s < NS; ++s) v[s] = s_stage[buf][s][threadIdx.x];
      buf ^= 1;
    }
    do_group(v);
    // a warp's lanes hold g = 32 w .. 32 w + 31, so (g | 31) is its last lane's: where that lane has no group this is
    // the warp's last iteration and only some of its lanes are here, so the flush after the loop takes this one
    if (++since_flush >= FLUSH_ROUNDS && (g | 31) < ngroups) {
      flush();
      since_flush = 0;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {  // scalar tail (n % 4 observations): lane .y repeats lane .x with weight 0
    for (int64_t i = ngroups * 4; i < a.n; ++i) {
      F2 e[NS];
#pragma unroll
      for (int s = 0; s < NS; ++s) e[s] = F2(sp[s][i], sp[s][i]);
      do_pair(e, false);
    }
  }
  flush();

  if (!grid_reduce<NRAW, V, 1, THREADS>(dacc, a, s_tot, s_warp)) return;
  if (mode == PASS_COST) {
    if (threadIdx.x == 0) a.out->v[NRAW - 1] = a.accumulate ? a.out->v[NRAW - 1] + s_tot[NRAW - 1] : s_tot[NRAW - 1];
  } else {
    for (int i = threadIdx.x; i < NRAW; i += THREADS) a.out->v[i] = a.accumulate ? a.out->v[i] + s_tot[i] : s_tot[i];
  }
  peer_push(a, NRAW);
}

#endif  // __CUDACC__
}  // namespace mopt
