// Device-resident Levenberg-Marquardt state machine.
// Restates LevenbergMarquadtDynamic<Scalar>::minimize (src/levenberg_marquadt_dyn.cpp:34-119) as a
// one-warp kernel that runs between pass kernels: it consumes the packed (H, b, sum) a pass wrote,
// decides accept / reject / terminate, solves the damped system with an LDL^T restated from
// Eigen::LDLT (pivoted, Eigen 3.4 Cholesky/LDLT.h), proposes x + delta, runs model setup for it and
// sets the control word the next pass kernel obeys.  No host round trip per iteration.
#pragma once

#include <cstddef>

#include "mopt_common.cuh"
#include "mopt_setup.cuh"

namespace mopt {

enum LmPhase : int { LM_PHASE_LIN = 0, LM_PHASE_TRIAL = 1 };

struct LmState {
  // configuration (written by lm_init_kernel)
  int P, n_costs, max_it, lm_max_it, speculative, scalar_f32;
  double lambda_factor;
  int flags;  // mopt_lm_flags
  int pad0_;
  // optimizer state
  double x[kMaxP], xi[kMaxP], delta[kMaxP], x_eval[kMaxP];
  PassResult cur;  // accepted linearization at x
  double lambda, nu;
  int it, k, phase, status, done, executed, num_trials, num_passes;
  int pass_mode;  // PassMode control word read by the pass kernels
  int pad_;
  mopt_lm_trial trials[MOPT_MAX_TRACE];
};

// Everything of LmState before the trace: what an optimizer transition reads and writes (staged in shared memory).
constexpr int kLmHotWords = int(offsetof(LmState, trials) / 8);
static_assert(offsetof(LmState, trials) % 8 == 0, "LmState hot part is copied in 8-byte words");
static_assert(kPackedMax <= 160, "lm_step_warp_t stages the pass result with five loads per lane");

// Arguments of levenberg_marquadt_dyn.cpp:15-26 (prepare), passed by value to the kernel that initialises the state.
struct LmInit {
  int P, n_costs, max_it, lm_max_it, speculative, scalar_f32;
  double lambda_factor;
  int flags;
  double x0[kMaxP];
};

#ifdef __CUDACC__

// Eigen 3.4 LDLT restated: in-place L D L^T of the lower triangle with symmetric diagonal pivoting
// (largest |a_kk|), left-looking column update; solve x = P^T L^-T D^+ L^-1 P b, D^+ with tolerance
// numeric_limits::min().  A column-major n x n (overwritten), n <= kMaxP.
template <typename S>
__device__ inline void ldlt_solve_dev(int n, S* A, const S* rhs, S* out) {
  int tr[kMaxP];
  S tmp[kMaxP], y[kMaxP];
#define MOPT_A(r, c) A[(r) + (c) * n]
  bool zero_matrix = false;
  for (int k = 0; k < n && !zero_matrix; ++k) {
    int piv = k;
    S best = fabs(MOPT_A(k, k));
    for (int i = k + 1; i < n; ++i) {
      const S v = fabs(MOPT_A(i, i));
      if (v > best) { best = v; piv = i; }
    }
    tr[k] = piv;
    if (piv != k) {
      for (int c = 0; c < k; ++c) { const S t = MOPT_A(k, c); MOPT_A(k, c) = MOPT_A(piv, c); MOPT_A(piv, c) = t; }
      for (int r = piv + 1; r < n; ++r) { const S t = MOPT_A(r, k); MOPT_A(r, k) = MOPT_A(r, piv); MOPT_A(r, piv) = t; }
      { const S t = MOPT_A(k, k); MOPT_A(k, k) = MOPT_A(piv, piv); MOPT_A(piv, piv) = t; }
      for (int i = k + 1; i < piv; ++i) { const S t = MOPT_A(i, k); MOPT_A(i, k) = MOPT_A(piv, i); MOPT_A(piv, i) = t; }
    }
    if (k > 0) {
      for (int c = 0; c < k; ++c) tmp[c] = MOPT_A(c, c) * MOPT_A(k, c);
      S s = S(0);
      for (int c = 0; c < k; ++c) s += MOPT_A(k, c) * tmp[c];
      MOPT_A(k, k) -= s;
      for (int r = k + 1; r < n; ++r) {
        S t = S(0);
        for (int c = 0; c < k; ++c) t += MOPT_A(r, c) * tmp[c];
        MOPT_A(r, k) -= t;
      }
    }
    const S akk = MOPT_A(k, k);
    const bool valid = fabs(akk) > S(0);
    if (k == 0 && !valid) {
      for (int j = 0; j < n; ++j) tr[j] = j;
      zero_matrix = true;
      break;
    }
    if (valid)
      for (int r = k + 1; r < n; ++r) MOPT_A(r, k) /= akk;
  }
  for (int i = 0; i < n; ++i) y[i] = rhs[i];
  for (int k = 0; k < n; ++k) { const S t = y[k]; y[k] = y[tr[k]]; y[tr[k]] = t; }
  for (int r = 0; r < n; ++r)
    for (int c = 0; c < r; ++c) y[r] -= MOPT_A(r, c) * y[c];
  const S tol = (sizeof(S) == 4) ? S(1.17549435e-38) : S(2.2250738585072014e-308);
  for (int i = 0; i < n; ++i) y[i] = (fabs(MOPT_A(i, i)) > tol) ? y[i] / MOPT_A(i, i) : S(0);
  for (int r = n - 1; r >= 0; --r)
    for (int c = r + 1; c < n; ++c) y[r] -= MOPT_A(c, r) * y[c];
  for (int k = n - 1; k >= 0; --k) { const S t = y[k]; y[k] = y[tr[k]]; y[tr[k]] = t; }
  for (int i = 0; i < n; ++i) out[i] = y[i];
#undef MOPT_A
}

template <typename S>
__device__ inline S scalar_eps() { return (sizeof(S) == 4) ? S(1.1920928955078125e-07) : S(2.220446049250313e-16); }

// include/moptimizer/optimizer.h:26-29
template <typename S>
__device__ inline bool is_cost_small(S c) { return fabs(c) < S(8) * scalar_eps<S>(); }

__device__ inline void lm_finish(LmState* st, int status) {
  st->status = status;
  st->executed = st->it;
  st->done = 1;
  st->pass_mode = PASS_SKIP;
}

// Warp-cooperative form of ldlt_solve_dev with VIRTUAL pivoting.  Same arithmetic on the same values in the same
// order as the serial restatement above (bit-identical factors and solution, cross-checked by mopt_ldlt_solve on every
// call), but
//   * the symmetric row / column exchanges of a pivot step move no data: a permutation (4 bits per index in one
//     64-bit word, identical on every lane) maps the algorithm's logical index to the row / column where the value
//     physically sits.  A must come in as the FULL symmetric matrix: logical entry (r, c), r > c, is read at physical
//     (perm r, perm c), which holds either the original a_rc = a_cr or, once column c is processed, L(r, c);
//   * the O(n^3) factorization runs with one lane per matrix row (every row's dot product keeps the serial summation
//     order), the divisions of a column and of the diagonal solve run one per lane;
//   * the O(n^2) substitutions stay on lane 0 in the serial order.
// The earlier form exchanged rows and columns in shared memory with four divergent branches per pivot step: 18 000
// cycles per 6 x 6 solve on a B200 against ~5 000 now.  A (n x n, column-major, overwritten), tmp, y and tr live in
// shared memory; n <= 16.  NC > 0: the size is known at compile time (the loops unroll).
template <typename S, int NC = 0>
__device__ inline void ldlt_solve_warp(int n_rt, S* A, const S* rhs, S* out, S* tmp, S* y, int* tr, int lane) {
  const int n = NC > 0 ? NC : n_rt;
  unsigned long long perm = 0xFEDCBA9876543210ull;
  auto PH = [&](int i) { return int((perm >> (4 * i)) & 15ull); };
#define MOPT_A(pr, pc) A[(pr) + (pc) * n]
  bool zero_matrix = false;
#pragma unroll
  for (int k = 0; k < n && !zero_matrix; ++k) {
    int piv = k;  // every lane scans the remaining diagonal itself: same result, no broadcast needed
    S best = fabs(MOPT_A(PH(k), PH(k)));
#pragma unroll
    for (int i = k + 1; i < n; ++i) {
      const S v = fabs(MOPT_A(PH(i), PH(i)));
      if (v > best) { best = v; piv = i; }
    }
    if (lane == 0) tr[k] = piv;
    {  // exchange logical k and piv
      const unsigned long long a = (perm >> (4 * k)) & 15ull, b = (perm >> (4 * piv)) & 15ull;
      perm = (perm & ~(15ull << (4 * k)) & ~(15ull << (4 * piv))) | (b << (4 * k)) | (a << (4 * piv));
    }
    const int pk = PH(k);
    if (k > 0) {
      if (lane < k) tmp[lane] = MOPT_A(PH(lane), PH(lane)) * MOPT_A(pk, PH(lane));
      __syncwarp();
      if (lane >= k && lane < n) {  // row `lane`: A(r, k) -= sum_c A(r, c) tmp[c]   (r == k: the diagonal update)
        const int pr = PH(lane);
        S t = S(0);
#pragma unroll
        for (int c = 0; c < k; ++c) t += MOPT_A(pr, PH(c)) * tmp[c];
        MOPT_A(pr, pk) -= t;
      }
      __syncwarp();
    }
    const S akk = MOPT_A(pk, pk);
    const bool valid = fabs(akk) > S(0);
    if (k == 0 && !valid) {
      if (lane < n) tr[lane] = lane;
      zero_matrix = true;
      __syncwarp();
      break;
    }
    if (valid && lane > k && lane < n) MOPT_A(PH(lane), pk) /= akk;
    __syncwarp();
  }
  if (lane == 0) {
    for (int i = 0; i < n; ++i) y[i] = rhs[i];
    for (int k = 0; k < n; ++k) { const S t = y[k]; y[k] = y[tr[k]]; y[tr[k]] = t; }
    for (int r = 0; r < n; ++r) {
      const int pr = PH(r);
      S v = y[r];
      for (int c = 0; c < r; ++c) v -= MOPT_A(pr, PH(c)) * y[c];
      y[r] = v;
    }
  }
  __syncwarp();
  if (lane < n) {  // D^+ with tolerance numeric_limits::min(): one division per lane
    const S tol = (sizeof(S) == 4) ? S(1.17549435e-38) : S(2.2250738585072014e-308);
    const S dd = MOPT_A(PH(lane), PH(lane));
    y[lane] = (fabs(dd) > tol) ? y[lane] / dd : S(0);
  }
  __syncwarp();
  if (lane == 0) {
    for (int r = n - 1; r >= 0; --r) {
      const int pr = PH(r);
      S v = y[r];
      for (int c = r + 1; c < n; ++c) v -= MOPT_A(PH(c), pr) * y[c];
      y[r] = v;
    }
    for (int k = n - 1; k >= 0; --k) { const S t = y[k]; y[k] = y[tr[k]]; y[tr[k]] = t; }
    for (int i = 0; i < n; ++i) out[i] = y[i];
  }
  __syncwarp();
#undef MOPT_A
}

// Shared-memory scratch of lm_solve_propose_warp (sized for doubles; the float instantiation uses the front).
struct LmSolveScratch {
  double A[kMaxP * kMaxP], nb[kMaxP], d[kMaxP], tmp[kMaxP], y[kMaxP];
  int tr[kMaxP];
};

// Solve (H + lambda diag(H)) delta = -b (levenberg_marquadt_dyn.cpp:65,78-80), xi = x (+) delta (:83), executed by
// one full warp: the lanes build the damped matrix and factor it together.
template <typename S, int PC = 0>
__device__ inline void lm_solve_propose_warp(LmState* st, const CostDev& cost0, LmSolveScratch* sc, int lane) {
  const int P = PC > 0 ? PC : st->P;
  S* A = reinterpret_cast<S*>(sc->A);
  S* nb = reinterpret_cast<S*>(sc->nb);
  S* d = reinterpret_cast<S*>(sc->d);
  const S lam = S(st->lambda);
  for (int e = lane; e < P * P; e += 32) {
    const int r = e % P, c = e / P;
    const S h = S(st->cur.v[r <= c ? tri_index(P, r, c) : tri_index(P, c, r)]);
    A[r + c * P] = (r == c) ? h + lam * h : h;  // Marquardt damping of the diagonal (:65)
  }
  if (lane < P) nb[lane] = -S(st->cur.v[P * (P + 1) / 2 + lane]);
  __syncwarp();
  ldlt_solve_warp<S, PC>(P, A, nb, d, reinterpret_cast<S*>(sc->tmp), reinterpret_cast<S*>(sc->y), sc->tr, lane);
  if (cost0.manifold == MOPT_MANIFOLD_SO3_LEFT) {
    if (lane == 0) {
      for (int i = 0; i < P; ++i) st->delta[i] = double(d[i]);
      retract_dev(cost0, st->x, st->delta, st->xi, sizeof(S) == 4);  // opt-in manifold update (SURVEY.md §8f-3)
      for (int i = 0; i < P; ++i) st->x_eval[i] = st->xi[i];
    }
  } else if (lane < P) {  // one parameter per lane
    const S dl = d[lane];
    const double xi = double(S(st->x[lane]) + dl);  // levenberg_marquadt_dyn.cpp:83
    st->delta[lane] = double(dl);
    st->xi[lane] = xi;
    st->x_eval[lane] = xi;
  }
  if (lane == 0) {
    st->phase = LM_PHASE_TRIAL;
    st->pass_mode = st->speculative ? PASS_LINEARIZE : PASS_COST;
  }
  __syncwarp();
}

// One transition of the optimizer, run by ONE thread.  Returns 0 if the optimization ended, 1 if a new evaluation
// point x_eval was set (the caller then runs model setup for every cost), 2 if the damped system has to be solved
// and a step proposed first (lm_solve_propose_warp, by the whole warp), followed by the same setup.
// Bit 2 (value 4) of the result: the caller must copy the whole pass result into st->cur (by the warp, one word per
// lane: on one thread the 28 shared-memory load / store pairs are a 1 000-cycle dependent chain); the thread has
// read what it needs of the new linearization from `trial` itself.
// `st` may be a shared-memory copy of the hot part of the state (everything before `trials`): the trace is written
// through `trials` (the array of the state in global memory), never through st->trials.
constexpr int kLmCopyTrial = 4;
template <typename S, int PC = 0>
__device__ inline int lm_step_thread(LmState* st, const PassResult* trial, const CostDev& cost0, mopt_lm_trial* trials) {
  if (st->done) return 0;
  const int P = PC > 0 ? PC : st->P;
  const int npk = packed_size(P);
  st->num_passes += 1;
  int copy = 0;                      // kLmCopyTrial once the accepted linearization is the one in `trial`
  const PassResult* lin = &st->cur;  // where (H, b, y0) of the accepted point are to be read from below
  if (st->phase == LM_PHASE_LIN) {
    copy = kLmCopyTrial;
    lin = trial;
  } else {
    const S yi = S(trial->v[npk - 1]);
    const S y0 = S(st->cur.v[npk - 1]);
    if (isnan(yi)) {  // :88-91
      lm_finish(st, MOPT_NUMERIC_ERROR);
      return 0;
    }
    const S lam = S(st->lambda);
    S den = S(0);
    for (int i = 0; i < P; ++i) {
      const S d = S(st->delta[i]);
      den += d * (lam * d - S(st->cur.v[P * (P + 1) / 2 + i]));
    }
    const S rho = (y0 - yi) / den;  // :93
    if (st->num_trials < MOPT_MAX_TRACE) {
      mopt_lm_trial& t = trials[st->num_trials];
      t.outer_iteration = st->it; t.k = st->k; t.accepted = !(rho < S(0)); t.reserved = 0;
      t.y0 = double(y0); t.yi = double(yi); t.rho = double(rho); t.lambda = st->lambda; t.nu = st->nu;
    }
    st->num_trials += 1;
    if (rho < S(0)) {  // :97-110 (a NaN rho compares false and is accepted, as in the reference)
      S m = S(0);
      for (int i = 0; i < P; ++i) m = fmax(m, fabs(S(st->delta[i])));
      if (m < sqrt(scalar_eps<S>())) {  // isDeltaSmall, delta.h:11-16
        lm_finish(st, is_cost_small<S>(yi) ? MOPT_CONVERGED : MOPT_SMALL_DELTA);
        return 0;
      }
      st->lambda = double(S(st->nu) * lam);
      st->nu = double(S(2) * S(st->nu));
      st->k += 1;
      if (st->k < st->lm_max_it) {
        return 2;
      }
      // inner tries exhausted: the outer loop re-linearizes at the unchanged x (identical H, b, y0)
      st->it += 1;
      if (st->it >= st->max_it) {
        lm_finish(st, MOPT_MAXIMUM_ITERATIONS_REACHED);
        return 0;
      }
    } else {  // :112-114
      for (int i = 0; i < P; ++i) st->x[i] = st->xi[i];
      // MOPT_LM_STAGNATION_STOP (not in the reference): a step below isDeltaSmall's threshold that leaves the cost
      // bit-for-bit unchanged is "accepted" with rho = 0 by :97 and doubles lambda (:113) for as long as iterations
      // remain.  The reference leaves this state by chance: its y0 (serial loop, linearization.h:142-154) and yi
      // (TBB parallel_reduce, :52-62) are summed in different orders, so rho's sign is rounding noise and the next
      // negative one ends in SMALL_DELTA (:98-101).  Both sums come from the same deterministic kernel here.
      if ((st->flags & MOPT_LM_STAGNATION_STOP) && yi == y0) {
        S m = S(0);
        for (int i = 0; i < P; ++i) m = fmax(m, fabs(S(st->delta[i])));
        if (m < sqrt(scalar_eps<S>())) {
          lm_finish(st, is_cost_small<S>(yi) ? MOPT_CONVERGED : MOPT_SMALL_DELTA);
          return 0;
        }
      }
      // std::pow(2 rho - 1, 3) evaluated in double (:113); v*v*v is within 1 ulp of it and keeps the library pow
      // (hundreds of instructions of a kernel that is instruction-fetch bound, DESIGN.md §3.4) out of the step
      const double v = double(S(2) * rho - S(1));
      const double f = fmax(1.0 / 3.0, 1.0 - v * v * v);
      st->lambda = double(S(double(lam) * f));
      st->it += 1;
      if (st->it >= st->max_it) {
        if (st->speculative) {
          lm_finish(st, MOPT_MAXIMUM_ITERATIONS_REACHED);
          return kLmCopyTrial;  // done (bits 0-1 clear); the final state holds the trial's linearization
        }
        st->cur.v[npk - 1] = trial->v[npk - 1];
        lm_finish(st, MOPT_MAXIMUM_ITERATIONS_REACHED);
        return 0;
      }
      if (st->speculative) {
        copy = kLmCopyTrial;
        lin = trial;
      } else {
        st->cur.v[npk - 1] = trial->v[npk - 1];
        for (int i = 0; i < P; ++i) st->x_eval[i] = st->x[i];
        st->phase = LM_PHASE_LIN;
        st->pass_mode = PASS_LINEARIZE;
        return 1;
      }
    }
  }
  // start of an outer iteration (:62-77) with (H, b, y0) = *lin
  for (;;) {
    const S y0 = S(lin->v[npk - 1]);
    if (is_cost_small<S>(y0)) {
      lm_finish(st, MOPT_CONVERGED);
      return copy;
    }
    if (st->lambda < 0.0) {
      S mx = S(0);
      for (int i = 0; i < P; ++i) mx = fmax(mx, fabs(S(lin->v[tri_index(P, i, i)])));
      st->lambda = double(S(st->lambda_factor) * mx);
    }
    st->nu = 2.0;
    st->k = 0;
    if (st->lm_max_it > 0) {
      return 2 | copy;
    }
    st->it += 1;
    if (st->it >= st->max_it) {
      lm_finish(st, MOPT_MAXIMUM_ITERATIONS_REACHED);
      return copy;
    }
  }
}

// One optimizer transition between two passes is executed by ONE WARP (lane = 0..31): accept / reject / terminate on
// lane 0, the damped solve and the proposal by the warp, then model->setup(x_eval) for every cost term.  Used by
// lm_step_kernel (one launch per transition) and by the persistent LM kernel (mopt_lm_mono.cuh).
// Shared memory of one optimizer transition: the LDL^T scratch, the hot part of the state and the pass result.
struct LmStepShared {
  LmSolveScratch sc;
  double hot[kLmHotWords];
  PassResult trial;
};

// How a transition finds its inputs.  The launch-per-trial path stages the state from and to global memory around
// every transition; the persistent kernel keeps it in CTA 0's shared memory from the first trial to the last
// (load_state on the first, store_state on the last or once `done` is set), gets the pass result in shared memory
// from the pass itself (trial_staged) and reads the cost constants from a shared-memory copy (cost0): every one of
// these was an L2 round trip of ~800 cycles in the dependent chain of a trial.
struct LmStepIo {
  bool load_state = true, store_state = true, trial_staged = false;
  const CostDev* cost0 = nullptr;  // cost term 0's constants if the caller holds a copy, else read from the slot
  // persistent kernel: where (R, t) of the next pass is published, this trial's barrier target and a shared-memory
  // flag — a set-up that knows when the next pass's own inputs are complete releases the waiting CTAs itself
  // (SetupEarlyOpen, publish_rt, mopt_setup.cuh)
  unsigned long long* rt_words = nullptr;
  unsigned long long gen_target = 0;
  int* opened = nullptr;
  LmState* host_state = nullptr;  // mapped host memory: the trace and the final state are written there as well,
  int* host_flag = nullptr;       // then this word is set (after a system-scope fence): the host may stop waiting
};

// levenberg_marquadt_dyn.cpp:15-26 (prepare) + the first setup(x0), by one warp.
// `st` may be the shared-memory copy of the state itself (persistent kernel: resident = true, cost0 = its copy of the
// cost constants); otherwise it is the state in global memory and sh->hot is only borrowed for x0.
static __device__ __noinline__ void lm_init_warp(LmState* st, CostSlot* slots, const LmInit& in, LmStepShared* sh, int lane,
                                                 bool resident = false, const CostDev* cost0 = nullptr) {
  if (lane == 0) {
    st->P = in.P; st->n_costs = in.n_costs; st->max_it = in.max_it; st->lm_max_it = in.lm_max_it;
    st->speculative = in.speculative; st->scalar_f32 = in.scalar_f32; st->lambda_factor = in.lambda_factor;
    st->flags = in.flags;
    st->pad0_ = 0;
    st->lambda = -1.0; st->nu = 2.0;
    st->it = 0; st->k = 0; st->phase = LM_PHASE_LIN; st->status = MOPT_MAXIMUM_ITERATIONS_REACHED;
    st->done = 0; st->executed = 0; st->num_trials = 0; st->num_passes = 0;
    st->pass_mode = PASS_LINEARIZE;
    st->pad_ = 0;
  }
  if (lane < kMaxP) {
    const double v = lane < in.P ? (in.scalar_f32 ? double(float(in.x0[lane])) : in.x0[lane]) : 0.0;
    st->x[lane] = v; st->xi[lane] = v; st->x_eval[lane] = v; st->delta[lane] = 0.0;
    if (!resident) sh->hot[lane] = v;  // setup below reads x_eval from shared memory
  }
  for (int i = lane; i < kPackedMax; i += 32) st->cur.v[i] = 0.0;
  __syncwarp();
  const double* x = resident ? st->x_eval : sh->hot;
  for (int c = 0; c < in.n_costs; ++c)
    setup_cost((c == 0 && cost0) ? *cost0 : slots[c].cost, x, &slots[c].pb, lane, 32, sh->sc.tmp);
}

// The hot part of the state and the pass result are staged in shared memory by the whole warp (coalesced): the
// transition is a few thousand DEPENDENT instructions on one lane, and every access to the state in global memory
// costs an L2 round trip (measured on tst/point2point's cloud: 7 200 cycles for the accept / reject logic alone).
// Returns the state's `done` flag after the transition.
template <typename S, int PC>
__device__ inline int lm_step_warp_t(LmState* gst, const PassResult* gtrial, CostSlot* slots, LmStepShared* sh, int lane,
                                     int P_rt, const LmStepIo& io) {
  LmState* st = reinterpret_cast<LmState*>(sh->hot);
  const int npk = packed_size(PC > 0 ? PC : P_rt);
  {
    const double* g = reinterpret_cast<const double*>(gst);
    // past the L1: in the persistent kernel the state was last written by another SM (or by this one, earlier).
    // All loads are issued before the first store (the compiler cannot prove that the generic pointers do not alias
    // and would otherwise serialise eight L2 round trips).
    constexpr int kPerLane = (kLmHotWords + 31) / 32;
    double tmp[kPerLane];
    if (io.load_state) {
#pragma unroll
      for (int q = 0; q < kPerLane; ++q) tmp[q] = (lane + 32 * q < kLmHotWords) ? __ldcg(g + lane + 32 * q) : 0.0;
    }
    double tr0 = 0.0, tr1 = 0.0, tr2 = 0.0, tr3 = 0.0, tr4 = 0.0;  // npk <= kPackedMax = 152 <= 5 * 32
    if (!io.trial_staged) {
      if (lane < npk) tr0 = __ldcg(&gtrial->v[lane]);
      if (lane + 32 < npk) tr1 = __ldcg(&gtrial->v[lane + 32]);
      if (lane + 64 < npk) tr2 = __ldcg(&gtrial->v[lane + 64]);
      if (lane + 96 < npk) tr3 = __ldcg(&gtrial->v[lane + 96]);
      if (lane + 128 < npk) tr4 = __ldcg(&gtrial->v[lane + 128]);
    }
    if (io.load_state) {
#pragma unroll
      for (int q = 0; q < kPerLane; ++q)
        if (lane + 32 * q < kLmHotWords) sh->hot[lane + 32 * q] = tmp[q];
    }
    if (!io.trial_staged) {
      if (lane < npk) sh->trial.v[lane] = tr0;
      if (lane + 32 < npk) sh->trial.v[lane + 32] = tr1;
      if (lane + 64 < npk) sh->trial.v[lane + 64] = tr2;
      if (lane + 96 < npk) sh->trial.v[lane + 96] = tr3;
      if (lane + 128 < npk) sh->trial.v[lane + 128] = tr4;
    }
  }
  __syncwarp();
  const CostDev& cost0 = io.cost0 ? *io.cost0 : slots[0].cost;
  int act = 0;
  if (lane == 0) act = lm_step_thread<S, PC>(st, &sh->trial, cost0, io.host_state ? io.host_state->trials : gst->trials);
  act = __shfl_sync(0xffffffffu, act, 0);
  __syncwarp();  // lane 0's state writes are visible to the warp below
  if (act & kLmCopyTrial) {  // the accepted linearization is the one this pass produced
    for (int i = lane; i < npk; i += 32) st->cur.v[i] = sh->trial.v[i];
    __syncwarp();
    act &= ~kLmCopyTrial;
  }
  if (act == 2) {  // damped solve + proposal, the lanes sharing the factorization
    lm_solve_propose_warp<S, PC>(st, cost0, &sh->sc, lane);
    __syncwarp();
  }
  if (act) {
    const int nc = st->n_costs;
    const SetupEarlyOpen eo{io.rt_words, (io.gen_target << 2) | (unsigned long long)(st->pass_mode), io.opened};
    for (int c = 0; c < nc; ++c)
      setup_cost(c == 0 ? cost0 : slots[c].cost, st->x_eval, &slots[c].pb, lane, 32, sh->sc.tmp,
                 (io.rt_words != nullptr && nc == 1) ? &eo : nullptr);
  }
  __syncwarp();
  if (io.store_state || st->done) {
    double* g = reinterpret_cast<double*>(gst);
    for (int i = lane; i < kLmHotWords; i += 32) g[i] = sh->hot[i];
    if (io.host_state) {
      double* h = reinterpret_cast<double*>(io.host_state);
      for (int i = lane; i < kLmHotWords; i += 32) h[i] = sh->hot[i];
      __threadfence_system();
      __syncwarp();
      if (lane == 0 && io.host_flag) *reinterpret_cast<volatile int*>(io.host_flag) = 1;
    }
  }
  __syncwarp();
  return st->done;
}
// P and the Scalar of the LM arithmetic are launch-time constants of a minimize() call: the callers pass them as
// kernel arguments instead of reading them from the state (two dependent L2 round trips per transition).
// __noinline__: one copy per translation unit instead of one per kernel instantiation (the persistent LM kernel alone
// has 18; inlined, that translation unit took six minutes to compile).
static __device__ __noinline__ int lm_step_warp(LmState* st, const PassResult* trial, CostSlot* slots, LmStepShared* sh, int lane,
                                                int P, bool f32, const LmStepIo& io) {
  if (P == 6) {  // the 6-DoF registration case with unrolled loops
    return f32 ? lm_step_warp_t<float, 6>(st, trial, slots, sh, lane, P, io)
               : lm_step_warp_t<double, 6>(st, trial, slots, sh, lane, P, io);
  }
  return f32 ? lm_step_warp_t<float, 0>(st, trial, slots, sh, lane, P, io)
             : lm_step_warp_t<double, 0>(st, trial, slots, sh, lane, P, io);
}

#endif  // __CUDACC__
}  // namespace mopt
