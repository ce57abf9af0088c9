// Small problems: the WHOLE Levenberg-Marquardt loop in one persistent kernel.
//
// With a few tens of thousands of residuals a pass takes microseconds and mopt_lm_minimize's per-trial sequence
// [pass kernel] -> [lm_step_kernel] is bound by the two dependent launches and the one-warp optimizer step between
// them (tst/point2point's 29 310-point cloud: pass 8.6 us, step 17.7 us, 22 k LM iterations per second).  Here one
// cooperative launch keeps every CTA resident; each trial is
//     pass over the CTA's residuals -> CTA partials -> arrival ticket ->
//     CTA 0 (always the same SM: the serial tail stays in its instruction cache) reduces, assembles (H, b, sum), runs the optimizer transition (accept / reject, LDL^T solve,
//     x (+) delta, model->setup) and opens the grid barrier -> every CTA reads the new parameter block and goes on,
// until the state machine sets PASS_SKIP.  No launch, no host round trip and no second kernel per trial.
// Restates the loop of LevenbergMarquadtDynamic::minimize (src/levenberg_marquadt_dyn.cpp:34-119) around
// p2p_moment_body (mopt_pass.cuh); same arithmetic and summation order as the multi-launch path with the same grid.
#pragma once

#include "mopt_lm.cuh"
#include "mopt_pass.cuh"

namespace mopt {

struct MonoArgs {
  LmState* st;
  LmState* host_st;             // mapped host copy of the state: final state and trace are written there too,
  int* host_flag;               // then this mapped word is set to 1
  CostSlot* slots;
  unsigned long long* rt_words; // 24 tagged words: (R, t) of the next pass + its control word = the grid barrier (publish_rt)
  unsigned long long gen_base;  // barrier targets of this launch start here (monotonic over the context's life)
  int max_slots;
  int loss, qrot;               // mopt_loss_kind / "the moments are taken in q = R p" of the pass, chosen at run time here
  LmInit init;                  // prepare() arguments: CTA 0 initialises the state before the first pass
};

#ifdef __CUDACC__

// The loss kind and the Jacobian form are run-time switches over the six instantiations of the pass body (a small
// problem does not care), so that there is ONE entry per (store, compute) type pair: ptxas compiles the optimizer
// transition once per entry, and with a kernel per (loss, form) this translation unit took six minutes to build.
template <typename ST, typename CT, int THREADS, int UNROLL, int FLUSH_ROUNDS>
__device__ __forceinline__ void p2p_mono_pass(const PassArgs& a, int mode, int loss, bool qrot, const double* rt) {
#define MOPT_MONO_BODY(L, Q) p2p_moment_body<ST, CT, L, Q, THREADS, UNROLL, FLUSH_ROUNDS, false, true>(a, mode, rt)
  switch (loss) {
    case MOPT_LOSS_NONE: qrot ? MOPT_MONO_BODY(MOPT_LOSS_NONE, true) : MOPT_MONO_BODY(MOPT_LOSS_NONE, false); break;
    case MOPT_LOSS_GEMAN_MCCLURE:
      qrot ? MOPT_MONO_BODY(MOPT_LOSS_GEMAN_MCCLURE, true) : MOPT_MONO_BODY(MOPT_LOSS_GEMAN_MCCLURE, false);
      break;
    default: qrot ? MOPT_MONO_BODY(MOPT_LOSS_HUBER, true) : MOPT_MONO_BODY(MOPT_LOSS_HUBER, false); break;
  }
#undef MOPT_MONO_BODY
}

// A data CTA's warp 0 waits for publication `target` of (R, t) (publish_rt, mopt_setup.cuh): every lane < 24 polls its
// own word until the tag matches, then the halves are put together into rt[0..12) (shared memory).  Returns the
// PassMode that came with it.
__device__ __forceinline__ int mono_wait_rt(const unsigned long long* words, unsigned long long target, double* rt, int lane) {
  const unsigned full = 0xffffffffu;
  const unsigned want = unsigned((target << 2) & 0xffffffffull) >> 2;
  unsigned long long wv = 0;
  for (;;) {
    bool ok = true;
    if (lane < 24) {
      asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(wv) : "l"(words + lane) : "memory");
      ok = (unsigned(wv & 0xffffffffull) >> 2) == want;
    }
    if (__all_sync(full, ok)) break;
    __nanosleep(20);
  }
  const unsigned half = unsigned(wv >> 32);
  const int src = 2 * (lane % 12);
  const unsigned lo = __shfl_sync(full, half, src), hi = __shfl_sync(full, half, src + 1);
  if (lane < 12) rt[lane] = __hiloint2double(int(hi), int(lo));
  return int(__shfl_sync(full, unsigned(wv & 3ull), 0));
}

// CTA 0 is the optimizer: it takes no residuals.  Per trial it (a) forms the parts of the assembly that depend on its
// own set-up alone while CTAs 1.. stream their residuals, (b) waits for their partials, finishes (H, b, sum) in shared
// memory, (c) runs the transition on warp 0 with the state resident in shared memory, and (d) releases the data CTAs
// as soon as the next pass's (R, t) exists — the rest of the set-up (left Jacobian, 72 affine entries) overlaps
// the pass.  (R, t) and the control word of the next pass ("linearize / cost only / stop") travel in 24 tagged words
// that ARE the barrier: no fence, and a waiting CTA has its inputs with the load that releases it.
template <typename ST, typename CT, int THREADS, int MINB, int UNROLL, int FLUSH_ROUNDS>
__global__ void __launch_bounds__(THREADS, MINB) p2p_lm_mono_kernel(const PassArgs a, const MonoArgs m) {
  __shared__ LmStepShared s_sh;  // CTA 0: LDL^T scratch, the optimizer state (resident from the first trial to the last), the pass result
  __shared__ CostDev s_cost;     // CTA 0: the cost term's constants for the optimizer step
  __shared__ double s_rt[12];    // data CTAs: (R, t) of the current pass
  __shared__ int s_mode, s_opened;
  // warp 0 of CTA 0, when the set-up did not publish by itself: (R, t) as the set-up left it in the ParamBlock
  auto publish_from_pb = [&](unsigned long long target, int mode) {
    const int lane = threadIdx.x;
    const double v = lane < 24 ? __ldcg(&a.pb->sets[0][lane >> 1]) : 0.0;
    publish_rt(m.rt_words, (target << 2) | (unsigned long long)(mode), v, lane);
  };
  const bool master = blockIdx.x == 0;
  // prepare() + the first setup(x0): CTA 0, everyone else waits (no separate init kernel, no launch gap)
  if (master) {
    for (int i = threadIdx.x; i < int(sizeof(CostDev) / 4); i += THREADS)
      reinterpret_cast<int*>(&s_cost)[i] = reinterpret_cast<const int*>(&m.slots[0].cost)[i];
    __syncthreads();
    if (threadIdx.x < 32) {  // the state is born in shared memory; global memory sees it when the loop ends
      lm_init_warp(reinterpret_cast<LmState*>(s_sh.hot), m.slots, m.init, &s_sh, threadIdx.x, true, &s_cost);
      __syncwarp();
      publish_from_pb(m.gen_base + 1, PASS_LINEARIZE);
    }
    if (threadIdx.x == 0) s_mode = PASS_LINEARIZE;
  } else if (threadIdx.x < 32) {
    const int mode = mono_wait_rt(m.rt_words, m.gen_base + 1, s_rt, threadIdx.x);
    if (threadIdx.x == 0) s_mode = mode;
  }
  __syncthreads();
  for (int slot = 0; slot < m.max_slots; ++slot) {
    const int mode = s_mode;  // written before the __syncthreads that ends the previous iteration
    if (mode == PASS_SKIP) break;
    const unsigned long long target = m.gen_base + 2ull + (unsigned long long)(slot);
    if (!master) {
      p2p_mono_pass<ST, CT, THREADS, UNROLL, FLUSH_ROUNDS>(a, mode, m.loss, m.qrot != 0, s_rt);
      // (every thread has read s_rt and s_mode: the grid reduction inside the pass synchronises the CTA)
      if (threadIdx.x < 32) {
        const int next = mono_wait_rt(m.rt_words, target, s_rt, threadIdx.x);
        if (threadIdx.x == 0) s_mode = next;
      }
    } else {
      p2p_master_tail<THREADS>(a, mode, &s_sh.trial);
      if (threadIdx.x == 0) s_opened = 0;
      __syncthreads();  // the pass result complete (assembled by the whole CTA, in shared memory)
      if (threadIdx.x < 32) {
        LmStepIo io;
        io.load_state = false;
        io.store_state = (slot == m.max_slots - 1);  // and whenever the state machine ends (lm_step_warp_t)
        io.trial_staged = true;
        io.cost0 = &s_cost;
        io.rt_words = m.rt_words;
        io.gen_target = target;
        io.opened = &s_opened;
        io.host_state = m.host_st;
        io.host_flag = m.host_flag;
        lm_step_warp(m.st, &s_sh.trial, m.slots, &s_sh, threadIdx.x, m.init.P, m.init.scalar_f32 != 0, io);
        __syncwarp();
        const int next = reinterpret_cast<const LmState*>(s_sh.hot)->pass_mode;
        if (!s_opened) publish_from_pb(target, next);  // generic set-ups, and the final "stop"
        if (threadIdx.x == 0) s_mode = next;
      }
    }
    __syncthreads();
  }
}

#endif  // __CUDACC__
}  // namespace mopt
