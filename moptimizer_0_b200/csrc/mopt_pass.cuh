// Pass kernels: one full sweep over a store's residuals, fused
//   residual -> (analytical | finite-difference) Jacobian -> robust-loss weight ->
//   upper-triangular H / b / sum(r^T r) accumulation in registers ->
//   warp (transposing shuffle) -> CTA (shared memory) -> grid (last-CTA-done) reduction.
// Replaces the loops of CostComputation::{computeHessian, computeHessianNumerical, computeCost,
// parallelComputeCost} (include/moptimizer/linearization.h:36-158).
#pragma once

#include "mopt_common.cuh"
#include "mopt_setup.cuh"

namespace mopt {

// Cross-GPU exchange of the packed result over NVLink peer memory, fused into the pass kernel's last CTA instead
// of a separate NCCL all-reduce: every rank owns slots[parity][source rank]; the last CTA of a pass stores its
// packed (H, b, sum) into its slot on EVERY rank (P2P stores through NVSwitch), fences once at system scope, then
// writes a sequence flag next to each copy; the same warp then acquires every rank's flag in its OWN buffer and
// sums the slots in rank order, so all ranks obtain bit-identical totals (peer_push below).  Two parities suffice:
// a rank can only be two passes ahead of a peer after that peer has consumed the older slot.
constexpr int kMaxWorld = 8;
struct XSlot {
  double v[kPackedMax];
  unsigned long long seq;
  unsigned long long pad;
};
struct PeerArgs {
  XSlot* base[kMaxWorld];  // exchange buffer of rank r as mapped in this process (base[rank] is local)
  int world, rank, push;
  int fused;               // 1: the pushing warp also waits for every rank's slot and writes the totals to `out`
                           //    (no separate consumer kernel); 0: peer_reduce_kernel does that
  unsigned long long seq;  // sequence number of this exchange (>= 1)
  int* err;                // set to 1 when a peer's slot does not arrive in time (mapped host memory: the host polls it)
  int* err_dev;            // device copy of the same word: later kernels of the stream read it and skip their work
};

struct PassArgs {
  PeerArgs peer;
  StreamPtrs streams;
  int64_t n;                 // residuals in this store (this rank's shard)
  const ParamBlock* pb;      // setup(x) result (device)
  const CostDev* cost;       // cost constants (device)
  double* partials;          // [nraw][gridDim.x] per-CTA partial sums
  unsigned int* ticket;      // last-CTA-done counter (self-resetting)
  PassResult* out;           // packed (H upper, b, sum)
  int accumulate;            // 1: out += this pass (second and later cost terms)
  const int* mode_ptr;       // device control word (PassMode), used when mode_override < 0
  int mode_override;
  int masked;                // 1: a NaN in the first B-group stream marks "no correspondence" (model f returned
                             // false, linearization.h:102,144): the residual is skipped entirely
  // Host-driven point2point analytical passes (mopt_linearize & co): model->setup(x) runs INSIDE the pass kernel —
  // every CTA derives (R, t) from x itself and the last CTA derives the affine Jacobian pieces — instead of in a
  // one-warp kernel launched before it (6.8 us + a dependent-launch gap per step).  `pb` is then not read.
  int fused_setup;
  int no_ring;               // second-generation point2point kernel: 1 = no TMA ring (unaligned streams), direct loads only
  XArg x;
};

#ifdef __CUDACC__

// ---------------------------------------------------------------------------------------------
// CTA + grid reduction shared by all pass kernels.
//   lane_val[ch]: this warp's total of raw sum (ch*32 + owner index), held by the owner lane
//   NRAW raw sums; V = values per transposing-reduce chunk (power of two <= 32)
// After the call, in the LAST CTA only, s_tot[0..NRAW) holds the grid totals (fp64) and the
// function returns true for every thread of that CTA.
// Part 2: s_warp[w * STRIDE + i] holds warp w's total of raw sum i (all warps written, CTA synchronised).
// MASTER (persistent LM kernel only, every CTA co-resident): CTA 0 of that kernel takes no residuals; it waits for the
// partials of the gridDim.x - 1 data CTAs and does the serial tail (grid_final_reduce, assembly, optimizer step), so
// that code stays in ONE SM's instruction cache from trial to trial and overlaps its set-up work with the pass.  The
// data CTAs (this function, MASTER = true) number themselves blockIdx.x - 1 and always return false.
template <int NRAW, int THREADS>
__device__ __forceinline__ void grid_final_reduce(const double* partials, int G, double* s_tot) {
  constexpr int NW = THREADS / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // fixed-order reduction of the G per-CTA partials: lanes stride over CTAs, xor-butterfly combine.  A warp owns rows
  // warp, warp + NW, ...; it walks them TOGETHER (all their loads in flight at once, the butterflies interleaved):
  // every row still adds the same values in the same order, and the tail of a pass is one L2 round trip plus one
  // butterfly instead of ROWS of each in sequence.
  constexpr int ROWS = (NRAW + NW - 1) / NW;
  constexpr int RB = ROWS < 4 ? ROWS : 4;  // rows in flight per warp (bounded: the tail must not set the kernel's register count)
  for (int q0 = 0; q0 < ROWS; q0 += RB) {
    double s[RB];
#pragma unroll
    for (int q = 0; q < RB; ++q) s[q] = 0.0;
    for (int c = lane; c < G; c += 32) {
      double v[RB];
#pragma unroll
      for (int q = 0; q < RB; ++q) {
        const int i = warp + (q0 + q) * NW;
        v[q] = (i < NRAW) ? __ldcg(partials + size_t(i) * G + c) : 0.0;
      }
#pragma unroll
      for (int q = 0; q < RB; ++q) s[q] += v[q];
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
#pragma unroll
      for (int q = 0; q < RB; ++q) s[q] += shfl_xor(s[q], o);
    }
    if (lane == 0) {
#pragma unroll
      for (int q = 0; q < RB; ++q)
        if (warp + (q0 + q) * NW < NRAW) s_tot[warp + (q0 + q) * NW] = s[q];
    }
  }
}

template <int NRAW, int STRIDE, int THREADS, bool MASTER = false>
__device__ __forceinline__ bool grid_reduce_shared(const PassArgs& a, double* s_tot, const double* s_warp) {
  constexpr int NW = THREADS / 32;
  __shared__ bool s_last;
  const int G = MASTER ? int(gridDim.x) - 1 : int(gridDim.x);
  const int bid = MASTER ? int(blockIdx.x) - 1 : int(blockIdx.x);
  for (int i = threadIdx.x; i < NRAW; i += THREADS) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < NW; ++w) s += s_warp[w * STRIDE + i];
    a.partials[size_t(i) * G + bid] = s;
  }
  __threadfence();
  __syncthreads();
  if constexpr (MASTER) {
    if (threadIdx.x == 0) atomicAdd(a.ticket, 1u);
    return false;
  } else {
    if (threadIdx.x == 0) {
      const unsigned int t = atomicAdd(a.ticket, 1u);
      s_last = (t == unsigned(G - 1));
    }
    __syncthreads();
    if (!s_last) return false;
  }
  __threadfence();
  grid_final_reduce<NRAW, THREADS>(a.partials, G, s_tot);
  if (threadIdx.x == 0) *a.ticket = 0u;  // ready for the next launch (stream-ordered)
  __syncthreads();
  return true;
}

template <int NRAW, int V, int NCH, int THREADS, bool MASTER = false>
__device__ __forceinline__ bool grid_reduce(const double (&lane_val)[NCH], const PassArgs& a, double* s_tot,
                                            double* s_warp /* [THREADS/32][NCH*V] */) {
  constexpr int SHIFT = 5 - Log2<V>::value;  // owner lane of index i is (i << SHIFT)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if ((lane & ((1 << SHIFT) - 1)) == 0) {
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) s_warp[warp * (NCH * V) + ch * V + (lane >> SHIFT)] = lane_val[ch];
  }
  __syncthreads();
  return grid_reduce_shared<NRAW, NCH * V, THREADS, MASTER>(a, s_tot, s_warp);
}

// A peer exchange earlier in this stream timed out (a rank died): the totals are meaningless from here on, so every
// later pass returns at once instead of spinning ~10 s on the dead peer again; the host sees the mapped error word.
__device__ __forceinline__ bool peer_failed(const PassArgs& a) {
  return a.peer.push && *reinterpret_cast<const volatile int*>(a.peer.err_dev) != 0;
}

// Last CTA of a pass, after `out` is complete: push the packed result into this rank's slot on every rank.
__device__ __forceinline__ void peer_push(const PassArgs& a, int npk) {
  if (!a.peer.push) return;
  __syncthreads();  // a.out fully written by this CTA
  if (threadIdx.x >= 32) return;  // one warp pushes: a system-scope fence per thread of a 1024-thread CTA costs ~80 us
  const int lane = threadIdx.x;
  const int slot = int(a.peer.seq & 1ull) * kMaxWorld + a.peer.rank;
  for (int i = lane; i < npk * a.peer.world; i += 32) {
    const int r = i / npk, k = i - r * npk;
    a.peer.base[r][slot].v[k] = a.out->v[k];
  }
  __syncwarp();  // orders the lanes' stores before lane 0's fence
  if (lane == 0) {
    // ONE system-scope fence orders every slot store above before every flag store below; the flags themselves
    // are relaxed stores (a release store per peer repeats the fence: measured +100 us per step at 8 ranks)
    __threadfence_system();
    for (int r = 0; r < a.peer.world; ++r) {
      unsigned long long* flag = &a.peer.base[r][slot].seq;
      asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(flag), "l"(a.peer.seq) : "memory");
    }
  }
  if (!a.peer.fused) return;
  // Consumer side, same warp: lane r acquires rank r's flag in the LOCAL exchange buffer, then the warp sums the
  // slots in rank order into `out` — identical bits on every rank.  Nothing on another GPU waits for this CTA, so
  // spinning here cannot deadlock; a peer that died is reported after ~10 s instead of hanging the device.
  __syncwarp();
  XSlot* mine = a.peer.base[a.peer.rank] + int(a.peer.seq & 1ull) * kMaxWorld;
  bool ok = true;
  if (lane < a.peer.world) {
    const unsigned long long* flag = &mine[lane].seq;
    const long long t0 = clock64();
    for (;;) {
      unsigned long long v;
      asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
      if (v == a.peer.seq) break;
      if (clock64() - t0 > 20000000000LL) {
        ok = false;
        break;
      }
      __nanosleep(32);
    }
  }
  ok = __all_sync(0xffffffffu, ok);
  __syncwarp();  // memory ordering among the lanes: every lane's slot reads below come after the acquiring lanes' flag reads
  if (!ok) {
    if (lane == 0) {
      *a.peer.err = 1;
      *a.peer.err_dev = 1;
      __threadfence_system();
    }
    return;
  }
  for (int k = lane; k < npk; k += 32) {
    double s = 0.0;
    for (int r = 0; r < a.peer.world; ++r) s += *reinterpret_cast<volatile double*>(&mine[r].v[k]);
    a.out->v[k] = s;
  }
}

// =============================================================================================
// Point-to-point, analytical Jacobian: moment kernel.
//
// Every analytical Jacobian of this model is affine in a 3-vector q (q = R p for the exact form,
// q = p for the reference-test forms):  J = J0 + q_x J1 + q_y J2 + q_z J3.  Hence
//   H = sum w J^T C J  and  b = sum w J^T C r
// are linear in the 23 moments
//   Sw, Sw q (3), Sw q q^T (6), Sw r (3), Sw q r^T (9), S r^T r (1)
// which is all the streaming loop accumulates (~50 FMA per correspondence instead of ~110 for the
// dense 3x6 update); the last CTA assembles the packed 6x6 H and b from them in fp64.
// Raw layout: [0]=Sw [1..3]=Swq [4..9]=Swqq(xx,xy,xz,yy,yz,zz) [10..12]=Swr [13..21]=Swqr(row q, col r) [22]=Se2
// =============================================================================================
constexpr int kP2PRaw = 23;

template <typename CT, int LOSS, bool QROT>
__device__ __forceinline__ void p2p_moments(bool masked, const CT (&R)[9], const CT (&t)[3], CT lossp, CT px, CT py,
                                            CT pz, CT yx, CT yy, CT yz, CT (&acc)[32]) {
  // q = R p ; r = (q + t) - y          (tst/point2point.cpp:41-44)
  const CT q0 = fma(R[0], px, fma(R[1], py, R[2] * pz));
  const CT q1 = fma(R[3], px, fma(R[4], py, R[5] * pz));
  const CT q2 = fma(R[6], px, fma(R[7], py, R[8] * pz));
  CT r0 = (q0 + t[0]) - yx;
  CT r1 = (q1 + t[1]) - yy;
  CT r2 = (q2 + t[2]) - yz;
  const bool skip = masked && (yx != yx);  // NaN target = no correspondence: f returned false, skip the residual
  if (skip) { r0 = CT(0); r1 = CT(0); r2 = CT(0); }
  const CT e2 = fma(r0, r0, fma(r1, r1, r2 * r2));
  const CT w = skip ? CT(0) : loss_weight<CT>(LOSS, lossp, e2);
  const CT a0 = QROT ? q0 : px, a1 = QROT ? q1 : py, a2 = QROT ? q2 : pz;
  const CT w0 = w * a0, w1 = w * a1, w2 = w * a2;
  acc[0] += w;
  acc[1] += w0; acc[2] += w1; acc[3] += w2;
  acc[4] = fma(w0, a0, acc[4]); acc[5] = fma(w0, a1, acc[5]); acc[6] = fma(w0, a2, acc[6]);
  acc[7] = fma(w1, a1, acc[7]); acc[8] = fma(w1, a2, acc[8]); acc[9] = fma(w2, a2, acc[9]);
  acc[10] = fma(w, r0, acc[10]); acc[11] = fma(w, r1, acc[11]); acc[12] = fma(w, r2, acc[12]);
  acc[13] = fma(w0, r0, acc[13]); acc[14] = fma(w0, r1, acc[14]); acc[15] = fma(w0, r2, acc[15]);
  acc[16] = fma(w1, r0, acc[16]); acc[17] = fma(w1, r1, acc[17]); acc[18] = fma(w1, r2, acc[18]);
  acc[19] = fma(w2, r0, acc[19]); acc[20] = fma(w2, r1, acc[20]); acc[21] = fma(w2, r2, acc[21]);
  acc[22] += e2;
}

template <typename CT>
__device__ __forceinline__ void p2p_cost_only(bool masked, const CT (&R)[9], const CT (&t)[3], CT px, CT py, CT pz,
                                              CT yx, CT yy, CT yz, CT (&acc)[32]) {
  const CT r0 = (fma(R[0], px, fma(R[1], py, R[2] * pz)) + t[0]) - yx;
  const CT r1 = (fma(R[3], px, fma(R[4], py, R[5] * pz)) + t[1]) - yy;
  const CT r2 = (fma(R[6], px, fma(R[7], py, R[8] * pz)) + t[2]) - yz;
  const CT e2 = fma(r0, r0, fma(r1, r1, r2 * r2));
  acc[22] += (masked && (yx != yx)) ? CT(0) : e2;
}

// ---- model->setup(x) fused into the pass (PassArgs::fused_setup) -------------------------------------------
// Set 0 of the point2point model, exactly as setup_cost / setup_one_set (mopt_setup.cuh) build it.
static __device__ __noinline__ void p2p_fused_set0(const CostDev* c, const double* x, double* set) {
  const bool f32 = (c->compute_dtype == MOPT_F32);
  double xs[6];
  for (int i = 0; i < 6; ++i) xs[i] = f32 ? double(float(x[i])) : x[i];
  const double w[3] = {xs[3], xs[4], xs[5]};
  double R[9];
  if (f32) so3_exp_dev<float>(w, R, c->so3_guard); else so3_exp_dev<double>(w, R, c->so3_guard);
  for (int i = 0; i < 9; ++i) set[i] = R[i];
  set[9] = xs[0]; set[10] = xs[1]; set[11] = xs[2];
}
// J_l(omega) for the exact variant, identity otherwise (first lines of setup_p2p_affine).
static __device__ __noinline__ void p2p_fused_left_jacobian(const CostDev* c, const double* x, double* Jl) {
  for (int i = 0; i < 9; ++i) Jl[i] = (i % 4 == 0) ? 1.0 : 0.0;
  if (c->variant == MOPT_P2P_EXACT) {
    const double w[3] = {x[3], x[4], x[5]};
    so3_left_jacobian_dev(w, Jl);
  }
}
// Assemble packed (H upper, b, sum) of the 6-parameter problem from the 23 moment totals.  Called by the whole CTA.
// H(i, j) = sum_{k,l} Mt[k][l] * s_kl(i, j) with s_kl = sum_{a,b} J_k[a][i] C[a][b] J_l[b][j]: the 21 x 16 inner sums
// s_kl are spread over the CTA (`scratch`, 21 * 16 doubles of shared memory), then one thread per entry adds them
// up in the (k, l) order of the serial form — same operations in the same order, so the result is bit-identical to
// one thread doing all 144 products of an entry (which cost ~2.5 us of the last CTA's time on a small problem).
__device__ inline void p2p_assemble_inner(const double (*jaff)[18], const CostDev* cost, bool has_cov, int tid, int nthreads,
                                          double* scratch) {
  constexpr int P = 6, NH = P * (P + 1) / 2;
  // C = I (no covariance): the a != b terms of every sum are exact zeros and adding them changes nothing, so they are
  // skipped — the chains the last CTA waits on are 3, 16 and 12 fused multiply-adds long instead of 9, 16 and 36 (the
  // six entries of b were the longest: 2 200 cycles of dependent fp64 on a B200).  The products are spelled with
  // intrinsics so that both forms round identically wherever this function is inlined.
  double C[9];
  for (int i = 0; i < 9; ++i) C[i] = has_cov ? cost->cov[i] : ((i % 4 == 0) ? 1.0 : 0.0);
  for (int w = tid; w < NH * 16; w += nthreads) {
    const int e = w >> 4, k = (w >> 2) & 3, l = w & 3;
    int i = 0, rem = e;  // decode (i, j) of the packed upper triangle
    while (rem >= P - i) { rem -= P - i; ++i; }
    const int j = i + rem;
    double s = 0.0;
    if (has_cov) {
      for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b) s = __fma_rn(__dmul_rn(jaff[k][a * 6 + i], C[a + 3 * b]), jaff[l][b * 6 + j], s);
    } else {
      for (int a = 0; a < 3; ++a) s = __fma_rn(jaff[k][a * 6 + i], jaff[l][a * 6 + j], s);
    }
    scratch[w] = s;
  }
}
// Second half (after a CTA-wide synchronisation): needs the 23 totals.
__device__ inline void p2p_assemble_outer(const double* tot, const double (*jaff)[18], const CostDev* cost, bool has_cov,
                                          PassResult* out, int accumulate, int tid, int nthreads, const double* scratch) {
  constexpr int P = 6, NH = P * (P + 1) / 2;
  double C[9];
  for (int i = 0; i < 9; ++i) C[i] = has_cov ? cost->cov[i] : ((i % 4 == 0) ? 1.0 : 0.0);
  // augmented moment matrix Mt (4x4, q~ = (1, q)) and St (4x3) = sum w q~ r^T
  double Mt[4][4], St[4][3];
  Mt[0][0] = tot[0];
  for (int k = 0; k < 3; ++k) Mt[0][k + 1] = Mt[k + 1][0] = tot[1 + k];
  Mt[1][1] = tot[4]; Mt[1][2] = Mt[2][1] = tot[5]; Mt[1][3] = Mt[3][1] = tot[6];
  Mt[2][2] = tot[7]; Mt[2][3] = Mt[3][2] = tot[8]; Mt[3][3] = tot[9];
  for (int m = 0; m < 3; ++m) St[0][m] = tot[10 + m];
  for (int k = 0; k < 3; ++k)
    for (int m = 0; m < 3; ++m) St[k + 1][m] = tot[13 + k * 3 + m];
  const int npk = packed_size(P);
  for (int e = tid; e < npk; e += nthreads) {
    double val = 0.0;
    if (e < NH) {
      for (int k = 0; k < 4; ++k)
        for (int l = 0; l < 4; ++l) val = __fma_rn(Mt[k][l], scratch[e * 16 + k * 4 + l], val);
    } else if (e < npk - 1) {
      const int i = e - NH;
      if (has_cov) {
        for (int k = 0; k < 4; ++k)
          for (int a = 0; a < 3; ++a)
            for (int b = 0; b < 3; ++b) val = __fma_rn(__dmul_rn(jaff[k][a * 6 + i], C[a + 3 * b]), St[k][b], val);
      } else {
        for (int k = 0; k < 4; ++k)
          for (int a = 0; a < 3; ++a) val = __fma_rn(jaff[k][a * 6 + i], St[k][a], val);
      }
    } else {
      val = tot[22];
    }
    out->v[e] = accumulate ? out->v[e] + val : val;
  }
}
__device__ inline void p2p_assemble(const double* tot, const double (*jaff)[18], const CostDev* cost, bool has_cov,
                                    PassResult* out, int accumulate, int tid, int nthreads, double* scratch) {
  p2p_assemble_inner(jaff, cost, has_cov, tid, nthreads, scratch);
  __syncthreads();
  p2p_assemble_outer(tot, jaff, cost, has_cov, out, accumulate, tid, nthreads, scratch);
}

// Everything after a point2point streaming loop: CTA + grid reduction of the 23 moment sums (dacc[0]: the lane's
// fp64 total of moment `lane`), then, in the last CTA, assembly of the packed (H, b, sum) and the peer exchange.
// Returns true in the last CTA (after `out` is complete), false in every other CTA.
// COHERENT: this launch is the persistent LM kernel (mopt_lm_mono.cuh): the ParamBlock is rewritten by another CTA
// between passes, so it is read past the (incoherent) L1.
template <bool FUSED, int THREADS, bool COHERENT = false>
__device__ __forceinline__ bool p2p_finish(const PassArgs& a, int mode, const double (&dacc)[1], double* s_tot,
                                           double* s_warp) {
  if (!grid_reduce<kP2PRaw, 32, 1, THREADS, COHERENT>(dacc, a, s_tot, s_warp)) return false;
  if constexpr (COHERENT) {
    return false;  // data CTAs of the persistent LM kernel: p2p_master_tail (CTA 0) takes it from here
  } else {
    const bool has_cov = a.cost->has_cov != 0;
    if (mode == PASS_COST) {
      if (threadIdx.x == 0) {
        const int e = packed_size(6) - 1;
        a.out->v[e] = a.accumulate ? a.out->v[e] + s_tot[22] : s_tot[22];
      }
    } else {
      __shared__ double s_jl[FUSED ? 9 : 1];
      __shared__ double s_jaff[FUSED ? 4 : 1][18];
      const double(*jaff)[18] = FUSED ? s_jaff : a.pb->jaff;
      if constexpr (FUSED) {
        // the affine pieces of J, entry by entry (same sums, same order as setup_p2p_affine)
        if (threadIdx.x == 0) {
          double xl[6];  // a copy: taking the address of a kernel parameter would spill the whole PassArgs to local memory
#pragma unroll
          for (int i = 0; i < 6; ++i) xl[i] = a.x.v[i];
          p2p_fused_left_jacobian(a.cost, xl, s_jl);
        }
        __syncthreads();
        for (int i = threadIdx.x; i < 4 * 18; i += THREADS) s_jaff[i / 18][i % 18] = p2p_affine_entry(a.cost->variant, s_jl, i / 18, i % 18);
        __syncthreads();
      }
      __shared__ double s_asm[21 * 16];
      p2p_assemble(s_tot, jaff, a.cost, has_cov, a.out, a.accumulate, threadIdx.x, THREADS, s_asm);
    }
    peer_push(a, packed_size(6));
    return true;
  }
}

// CTA 0 of the persistent LM kernel: everything of a pass that is not streaming.  The Jacobian pieces this CTA's own
// set-up wrote and the 21 x 16 inner sums that depend on them alone are taken care of WHILE the data CTAs stream;
// then the totals of their partials, the outer sums, and the packed (H, b, sum) lands in `out` (shared memory).
template <int THREADS>
__device__ __forceinline__ void p2p_master_tail(const PassArgs& a, int mode, PassResult* out) {
  static_assert(THREADS >= 4 * 18, "one ParamBlock::jaff entry per thread");
  __shared__ double s_tot[32];
  __shared__ double s_jaff[4][18];
  __shared__ double s_asm[21 * 16];
  const int G = int(gridDim.x) - 1;
  const bool has_cov = a.cost->has_cov != 0;
  if (mode != PASS_COST) {
    if (threadIdx.x < 4 * 18) (&s_jaff[0][0])[threadIdx.x] = __ldcg(&a.pb->jaff[0][0] + threadIdx.x);
    __syncthreads();
    p2p_assemble_inner(s_jaff, a.cost, has_cov, threadIdx.x, THREADS, s_asm);
  }
  if (threadIdx.x == 0) {
    while (*reinterpret_cast<volatile unsigned int*>(a.ticket) != unsigned(G)) {}
  }
  __syncthreads();
  __threadfence();
  grid_final_reduce<kP2PRaw, THREADS>(a.partials, G, s_tot);
  if (threadIdx.x == 0) *a.ticket = 0u;
  __syncthreads();
  if (mode == PASS_COST) {
    if (threadIdx.x == 0) {
      const int e = packed_size(6) - 1;
      out->v[e] = a.accumulate ? out->v[e] + s_tot[22] : s_tot[22];
    }
  } else {
    p2p_assemble_outer(s_tot, s_jaff, a.cost, has_cov, out, a.accumulate, threadIdx.x, THREADS, s_asm);
  }
}

// FUSED: model->setup(x) runs inside the kernel (PassArgs::x; host-driven analytical passes), `pb` is not read.
// The pass itself, callable from the one-pass kernel below and from the persistent LM kernel (mopt_lm_mono.cuh).
// Returns true in the last CTA once `out` holds the packed result.
template <typename ST, typename CT, int LOSS, bool QROT, int THREADS, int UNROLL, int FLUSH_ROUNDS, bool FUSED, bool COHERENT>
__device__ __forceinline__ bool p2p_moment_body(const PassArgs& a, const int mode, const double* rt = nullptr) {
  // COHERENT: a data CTA of the persistent LM kernel, whose CTA 0 takes no residuals (grid_reduce_shared); (R, t)
  // comes in `rt` (shared memory, received with the barrier: publish_rt) instead of the ParamBlock
  const int bid = COHERENT ? int(blockIdx.x) - 1 : int(blockIdx.x);
  const int nb = COHERENT ? int(gridDim.x) - 1 : int(gridDim.x);
  constexpr int VEC = VecOf<ST>::N;
  constexpr bool kFp32Acc = (sizeof(CT) == 4);
  // fp32 partials are folded into fp64 every FLUSH_ROUNDS*VEC residuals/thread

  __shared__ double s_warp[(THREADS / 32) * 32];
  __shared__ double s_tot[32];

  __shared__ double s_set0[FUSED ? 12 : 1];
  const double* set0 = FUSED ? s_set0 : (COHERENT ? rt : a.pb->sets[0]);
  if constexpr (FUSED) {
    if (threadIdx.x == 0) {
      double xl[6];  // a copy: taking the address of a kernel parameter would spill the whole PassArgs to local memory
#pragma unroll
      for (int i = 0; i < 6; ++i) xl[i] = a.x.v[i];
      p2p_fused_set0(a.cost, xl, s_set0);
    }
    __syncthreads();
  }
  CT R[9], t[3];
#pragma unroll
  for (int i = 0; i < 9; ++i) R[i] = CT(set0[i]);
#pragma unroll
  for (int i = 0; i < 3; ++i) t[i] = CT(set0[9 + i]);
  const CT lossp = CT(a.cost->loss_param);
  const bool masked = a.masked != 0;

  const ST* __restrict__ sx = static_cast<const ST*>(a.streams.p[0]);
  const ST* __restrict__ sy = static_cast<const ST*>(a.streams.p[1]);
  const ST* __restrict__ sz = static_cast<const ST*>(a.streams.p[2]);
  const ST* __restrict__ tx = static_cast<const ST*>(a.streams.p[3]);
  const ST* __restrict__ ty = static_cast<const ST*>(a.streams.p[4]);
  const ST* __restrict__ tz = static_cast<const ST*>(a.streams.p[5]);

  CT acc[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) acc[i] = CT(0);
  double dacc[1] = {0.0};

  const int64_t ngroups = a.n / VEC;
  const int64_t stride = int64_t(nb) * THREADS;
  const int64_t full_rounds = ngroups / stride;
  const int64_t g0 = int64_t(bid) * THREADS + threadIdx.x;

  auto flush = [&]() {
    const CT v = warp_reduce_transpose<32>(acc);
    dacc[0] += double(v);
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = CT(0);
  };

  auto do_group = [&](int64_t g) {
    CT px[VEC], py[VEC], pz[VEC], qx[VEC], qy[VEC], qz[VEC];
    load_vec<ST, CT>(sx, g, px); load_vec<ST, CT>(sy, g, py); load_vec<ST, CT>(sz, g, pz);
    load_vec<ST, CT>(tx, g, qx); load_vec<ST, CT>(ty, g, qy); load_vec<ST, CT>(tz, g, qz);
    if (mode == PASS_COST) {
#pragma unroll
      for (int e = 0; e < VEC; ++e) p2p_cost_only<CT>(masked, R, t, px[e], py[e], pz[e], qx[e], qy[e], qz[e], acc);
    } else {
#pragma unroll
      for (int e = 0; e < VEC; ++e)
        p2p_moments<CT, LOSS, QROT>(masked, R, t, lossp, px[e], py[e], pz[e], qx[e], qy[e], qz[e], acc);
    }
  };

  int since_flush = 0;
  int64_t r = 0;
  // UNROLL grid-stride rounds per iteration: 6*UNROLL independent 16-byte loads in flight per thread
  for (; r + (UNROLL - 1) < full_rounds; r += UNROLL) {
    CT px[UNROLL][VEC], py[UNROLL][VEC], pz[UNROLL][VEC], qx[UNROLL][VEC], qy[UNROLL][VEC], qz[UNROLL][VEC];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const int64_t g = g0 + (r + u) * stride;
      load_vec<ST, CT>(sx, g, px[u]); load_vec<ST, CT>(sy, g, py[u]); load_vec<ST, CT>(sz, g, pz[u]);
      load_vec<ST, CT>(tx, g, qx[u]); load_vec<ST, CT>(ty, g, qy[u]); load_vec<ST, CT>(tz, g, qz[u]);
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      if (mode == PASS_COST) {
#pragma unroll
        for (int e = 0; e < VEC; ++e)
          p2p_cost_only<CT>(masked, R, t, px[u][e], py[u][e], pz[u][e], qx[u][e], qy[u][e], qz[u][e], acc);
      } else {
#pragma unroll
        for (int e = 0; e < VEC; ++e)
          p2p_moments<CT, LOSS, QROT>(masked, R, t, lossp, px[u][e], py[u][e], pz[u][e], qx[u][e], qy[u][e], qz[u][e], acc);
      }
    }
    if (kFp32Acc) {
      since_flush += UNROLL;
      if (since_flush >= FLUSH_ROUNDS) {
        flush();
        since_flush = 0;
      }
    }
  }
  for (; r < full_rounds; ++r) do_group(g0 + r * stride);
  {  // ragged last round + scalar tail (n % VEC residuals)
    const int64_t g = g0 + full_rounds * stride;
    if (g < ngroups) do_group(g);
    if (bid == 0 && threadIdx.x == 0) {
      for (int64_t i = ngroups * VEC; i < a.n; ++i) {
        if (mode == PASS_COST)
          p2p_cost_only<CT>(masked, R, t, CT(sx[i]), CT(sy[i]), CT(sz[i]), CT(tx[i]), CT(ty[i]), CT(tz[i]), acc);
        else
          p2p_moments<CT, LOSS, QROT>(masked, R, t, lossp, CT(sx[i]), CT(sy[i]), CT(sz[i]), CT(tx[i]), CT(ty[i]), CT(tz[i]), acc);
      }
    }
  }
  flush();

  return p2p_finish<FUSED, THREADS, COHERENT>(a, mode, dacc, s_tot, s_warp);
}

template <typename ST, typename CT, int LOSS, bool QROT, int THREADS, int MINB, int UNROLL = 2, int FLUSH_ROUNDS = 8,
          bool FUSED = false>
__global__ void __launch_bounds__(THREADS, MINB) p2p_moment_kernel(const PassArgs a) {
  const int mode = a.mode_override >= 0 ? a.mode_override : *a.mode_ptr;
  if (mode == PASS_SKIP) return;
  if (peer_failed(a)) return;
  p2p_moment_body<ST, CT, LOSS, QROT, THREADS, UNROLL, FLUSH_ROUNDS, FUSED, false>(a, mode);
}

// =============================================================================================
// Generic dense pass kernel for any builtin model: analytical (model f_df) or finite-difference
// Jacobian in registers, optional O x O covariance, packed upper-triangular accumulation.
// Raw layout == packed layout: H upper (row-major), b, sum.
// =============================================================================================
//
// AFFINE_FD (models that declare NAFF/affine/finish/finish_diff, i.e. residual = finish(affine(set, e)) with a first
// stage linear in the set): the staged sets 1 + j hold D_j = (set(x + h_j e_j) - set_ref) / H_j formed in fp64
// (set_ref = set(x - h_j e_j) for central differences, set(x) for the reference's forward scheme,
// linearization.h:97-111; H_j = the step actually taken between the two parameter vectors after rounding in the
// compute Scalar, ParamBlock::hstep_*), and column j of J is M::finish_diff(affine(set_ref), affine(D_j), H_j): the same
// difference quotient (f(x + h e_j) - f_ref) / H with the subtraction carried out over a common denominator
// instead of between two rounded quotients -- one reciprocal per column instead of 2 O divisions, and none of
// the eps / h amplification of the per-residual form (which MOPT_FLAG_GENERIC_KERNEL keeps selectable).
template <class M, typename ST, typename CT, bool NUMERIC, int THREADS, int MINB, bool AFFINE_FD = false>
__global__ void __launch_bounds__(THREADS, MINB) dense_pass_kernel(const PassArgs a) {
  const int mode = a.mode_override >= 0 ? a.mode_override : *a.mode_ptr;
  if (mode == PASS_SKIP) return;
  if (peer_failed(a)) return;
  constexpr int P = M::P, O = M::O, NS = M::NS;
  constexpr int VEC = VecOf<ST>::N;
  constexpr int NRAW = P * (P + 1) / 2 + P + 1;
  constexpr int V = next_pow2(NRAW);
  static_assert(V <= 32, "dense_pass_kernel: packed size must fit one transposing-reduce chunk");
  constexpr bool kFp32Acc = (sizeof(CT) == 4);
  constexpr int FLUSH_ROUNDS = 8;
  constexpr int NSETS = 1 + 2 * (P > 0 ? P : 0);
  constexpr int VPE = 16 / int(sizeof(CT));                       // elements per 16-byte shared-memory access
  constexpr int SETN = ((M::SETN > 0 ? M::SETN : 1) + VPE - 1) / VPE * VPE;  // sets padded to 16-byte units
  // Finite differences of the larger models (1 + 2P sets of SETN values, e.g. 13 x 12 for the pinhole camera) do not
  // fit in registers next to J and the accumulators; left alone the compiler hoists them all out of the streaming
  // loop and spills them to local memory.  They are re-read from shared memory with 16-byte loads at every use.
  constexpr bool kReloadSets = NUMERIC && (NSETS * SETN > 32);

  __shared__ double s_warp[(THREADS / 32) * V];
  __shared__ double s_tot[V];
  __shared__ __align__(16) CT s_sets[NSETS][SETN];
  __shared__ CT s_invh[P > 0 ? P : 1];
  __shared__ CT s_cov[O * O];

  const int jac = a.cost->jacobian;
  const bool central = (jac == MOPT_JAC_CENTRAL);
  const int nsets = !NUMERIC ? 1 : (central ? 1 + 2 * P : 1 + P);
  for (int i = threadIdx.x; i < nsets * SETN; i += THREADS) {
    const int si = i / SETN, k = i % SETN;
    double v = (k < M::SETN) ? a.pb->sets[si][k] : 0.0;
    if (AFFINE_FD && si >= 1 && si <= P && k < M::SETN) {
      const int j = si - 1;
      v = central ? (v - a.pb->sets[1 + P + j][k]) / a.pb->hstep_cen[j] : (v - a.pb->sets[0][k]) / a.pb->hstep_fwd[j];
    }
    s_sets[si][k] = CT(v);
  }
  for (int i = threadIdx.x; i < P; i += THREADS) {
    if (AFFINE_FD) s_invh[i] = CT(central ? a.pb->hstep_cen[i] : a.pb->hstep_fwd[i]);  // H_j itself in this mode
    else s_invh[i] = CT(central ? 1.0 / (2.0 * a.pb->h[i]) : 1.0 / a.pb->h[i]);
  }
  const bool has_cov = a.cost->has_cov != 0;
  for (int i = threadIdx.x; i < O * O; i += THREADS) s_cov[i] = CT(a.cost->cov[i]);
  const int loss = a.cost->loss;
  const CT lossp = CT(a.cost->loss_param);
  __syncthreads();

  const ST* __restrict__ sp[NS > 0 ? NS : 1];
#pragma unroll
  for (int s = 0; s < NS; ++s) sp[s] = static_cast<const ST*>(a.streams.p[s]);

  CT acc[V];
#pragma unroll
  for (int i = 0; i < V; ++i) acc[i] = CT(0);
  double dacc[1] = {0.0};

  auto flush = [&]() {
    const CT v = warp_reduce_transpose<V>(acc);
    dacc[0] += double(v);
#pragma unroll
    for (int i = 0; i < V; ++i) acc[i] = CT(0);
  };

  // one residual: e[] = its NS stream values
  const bool masked = a.masked != 0;
  auto do_elem = [&](const CT (&e)[NS > 0 ? NS : 1]) {
    CT r[O];
    if (NS > 0 && masked) {  // NaN in the first B-group stream: no correspondence, the residual is skipped
      const CT probe = e[(M::NA < NS) ? M::NA : 0];
      if (probe != probe) return;
    }
    if (mode == PASS_COST) {
      M::template residual<CT>(s_sets[0], e, r);
      CT e2 = CT(0);
#pragma unroll
      for (int o = 0; o < O; ++o) e2 = fma(r[o], r[o], e2);
      acc[NRAW - 1] += e2;
      return;
    }
    CT J[O * (P > 0 ? P : 1)];
    if constexpr (NUMERIC && AFFINE_FD) {
      constexpr int NAFF = M::NAFF;
      auto stage1 = [&](int idx, CT (&u)[NAFF]) {
        if constexpr (kReloadSets) {
          CT sr[SETN];
#pragma unroll
          for (int k = 0; k < SETN; k += VPE) {
            CT t[VPE];
            lds16_reload(&s_sets[idx][k], t);
#pragma unroll
            for (int v = 0; v < VPE; ++v) sr[k + v] = t[v];
          }
          M::template affine<CT>(sr, e, u);
        } else {
          M::template affine<CT>(s_sets[idx], e, u);
        }
      };
      CT u0[NAFF];
      M::template affine<CT>(s_sets[0], e, u0);
      M::template finish<CT>(s_sets[0], u0, e, r);
#pragma unroll
      for (int j = 0; j < P; ++j) {
        CT du[NAFF], d[O];
        stage1(1 + j, du);
        if (central) {
          CT um[NAFF];
          stage1(1 + P + j, um);
          M::template finish_diff<CT>(s_sets[0], um, du, s_invh[j], e, d);
        } else {
          M::template finish_diff<CT>(s_sets[0], u0, du, s_invh[j], e, d);
        }
#pragma unroll
        for (int o = 0; o < O; ++o) J[o * P + j] = d[o];
      }
    } else if constexpr (NUMERIC) {
      M::template residual<CT>(s_sets[0], e, r);
      auto eval = [&](int idx, CT (&out)[O]) {
        if constexpr (kReloadSets) {
          CT sr[SETN];
#pragma unroll
          for (int k = 0; k < SETN; k += VPE) {
            CT t[VPE];
            lds16_reload(&s_sets[idx][k], t);
#pragma unroll
            for (int u = 0; u < VPE; ++u) sr[k + u] = t[u];
          }
          M::template residual<CT>(sr, e, out);
        } else {
          M::template residual<CT>(s_sets[idx], e, out);
        }
      };
#pragma unroll
      for (int j = 0; j < P; ++j) {
        CT rp[O];
        eval(1 + j, rp);  // perturbed f's bool is ignored, linearization.h:104
        if (central) {
          CT rm[O];
          eval(1 + P + j, rm);
#pragma unroll
          for (int o = 0; o < O; ++o) J[o * P + j] = (rp[o] - rm[o]) * s_invh[j];
        } else {
#pragma unroll
          for (int o = 0; o < O; ++o) J[o * P + j] = (rp[o] - r[o]) * s_invh[j];
        }
      }
    } else {
      M::template residual_jacobian<CT>(s_sets[0], e, r, J);
    }
    CT e2 = CT(0);
#pragma unroll
    for (int o = 0; o < O; ++o) e2 = fma(r[o], r[o], e2);
    const CT w = loss_weight<CT>(loss, lossp, e2);
    // CJ = C J, Cr = C r  (identity unless setCovariance was called)
    CT CJ[O * (P > 0 ? P : 1)], Cr[O];
    if (has_cov) {
#pragma unroll
      for (int o = 0; o < O; ++o) {
        CT s = CT(0);
#pragma unroll
        for (int k = 0; k < O; ++k) s = fma(s_cov[o + k * O], r[k], s);
        Cr[o] = s;
#pragma unroll
        for (int p = 0; p < P; ++p) {
          CT sj = CT(0);
#pragma unroll
          for (int k = 0; k < O; ++k) sj = fma(s_cov[o + k * O], J[k * P + p], sj);
          CJ[o * P + p] = sj;
        }
      }
    } else {
#pragma unroll
      for (int o = 0; o < O; ++o) {
        Cr[o] = r[o];
#pragma unroll
        for (int p = 0; p < P; ++p) CJ[o * P + p] = J[o * P + p];
      }
    }
    int idx = 0;
#pragma unroll
    for (int i = 0; i < P; ++i) {
      CT wj[O];
#pragma unroll
      for (int o = 0; o < O; ++o) wj[o] = w * J[o * P + i];
#pragma unroll
      for (int j = i; j < P; ++j) {
        CT s = acc[idx];
#pragma unroll
        for (int o = 0; o < O; ++o) s = fma(wj[o], CJ[o * P + j], s);
        acc[idx] = s;
        ++idx;
      }
    }
#pragma unroll
    for (int i = 0; i < P; ++i) {
      CT s = acc[idx];
#pragma unroll
      for (int o = 0; o < O; ++o) s = fma(w * J[o * P + i], Cr[o], s);
      acc[idx] = s;
      ++idx;
    }
    acc[NRAW - 1] += e2;
  };

  auto do_group = [&](int64_t g) {
    CT vals[NS > 0 ? NS : 1][VEC];
#pragma unroll
    for (int s = 0; s < NS; ++s) load_vec<ST, CT>(sp[s], g, vals[s]);
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      CT e[NS > 0 ? NS : 1];
#pragma unroll
      for (int s = 0; s < NS; ++s) e[s] = vals[s][v];
      do_elem(e);
    }
  };

  if constexpr (NS == 0) {
    // data-free model (Powell): `n` identical residual blocks evaluated by thread 0
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      CT e[1] = {CT(0)};
      for (int64_t i = 0; i < a.n; ++i) do_elem(e);
    }
  } else {
    const int64_t ngroups = a.n / VEC;
    const int64_t stride = int64_t(gridDim.x) * THREADS;
    const int64_t full_rounds = ngroups / stride;
    const int64_t g0 = int64_t(blockIdx.x) * THREADS + threadIdx.x;
    int since_flush = 0;
    for (int64_t r = 0; r < full_rounds; ++r) {
      do_group(g0 + r * stride);
      if (kFp32Acc && ++since_flush >= FLUSH_ROUNDS) {
        flush();
        since_flush = 0;
      }
    }
    const int64_t g = g0 + full_rounds * stride;
    if (g < ngroups) do_group(g);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      for (int64_t i = ngroups * VEC; i < a.n; ++i) {
        CT e[NS];
#pragma unroll
        for (int s = 0; s < NS; ++s) e[s] = CT(sp[s][i]);
        do_elem(e);
      }
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

// =============================================================================================
// Wide pass kernel: models whose packed size P(P+1)/2 + P + 1 exceeds 32 (the n x n calibration case,
// e.g. P = 15 -> 120 + 15 + 1 = 136 sums).  That many per-thread accumulators do not fit in registers next
// to a 2 x 15 Jacobian, so each warp works in two phases on 32 residuals at a time:
//   1. every lane evaluates ONE residual and its Jacobian (finite differences or the model's f_df) and
//      stores the row  [ J (O x PA) | B = w C [J | r] (O x PB) ]  into the warp's shared tile with 16-byte
//      stores (row stride an odd number of 16-byte units: conflict-free);
//   2. the warp computes  C += J^T B  over the 32 rows as a register-tiled product over the 4x4 tiles on or
//      above the block diagonal (10 tiles for P = 15; columns 0..P-1 of C are H, column P is b): lane
//      (group g, tile t) accumulates tile t over rows g, g + NG, ... with two 16-byte shared loads per
//      16 FMAs; the NG row groups of a tile are merged in a fixed order at the end.
// Models may split their residual into a stage that depends only on the first STAGE1_PARAMS parameters
// (e.g. the rigid transform + perspective division) and a cheap second stage; perturbations of the
// remaining parameters then re-run only the second stage (bit-identical to the full evaluation).
// =============================================================================================
struct WideLayout {
  int NBI, NBJ, NT, NG, PA, PB, ROW;  // ROW in elements
};
__host__ __device__ constexpr WideLayout wide_layout(int P, int O, int elem_bytes) {
  const int vpe = 16 / elem_bytes;            // elements per 16-byte unit
  const int NBI = (P + 3) / 4;                // 4-row blocks of J^T
  const int NBJ = (P + 1 + 3) / 4;            // 4-column blocks of B = [w C J | w C r]
  int NT = 0;                                 // 4x4 tiles on or above the block diagonal (the b column lives in the last block column)
  for (int bi = 0; bi < NBI; ++bi) NT += NBJ - bi;
  const int NG = 32 / NT;                     // row groups: lane = group * NT + tile, group g takes rows g, g + NG, ...
  const int PA = NBI * 4, PB = NBJ * 4;
  int row = O * PA + O * PB;                  // multiple of vpe
  if (((row / vpe) & 1) == 0) row += vpe;     // odd number of 16-byte units per row: conflict-free 16-byte row stores
  return WideLayout{NBI, NBJ, NT, NG, PA, PB, row};
}
__host__ __device__ constexpr int wide_set_stride(int setn, int elem_bytes) {  // parameter sets padded to 16-byte units
  return ((setn + 16 / elem_bytes - 1) / (16 / elem_bytes)) * (16 / elem_bytes);
}
__host__ __device__ constexpr size_t wide_smem_bytes_rt(int P, int O, int setn, int elem_bytes, int threads) {
  return size_t(elem_bytes) * (size_t(threads / 32) * 32 * wide_layout(P, O, elem_bytes).ROW +
                               size_t(1 + 2 * P) * wide_set_stride(setn, elem_bytes) + P + O * O) + 16;
}

#ifdef __CUDACC__
// Does model M declare a two-stage residual?
template <class M, class = void>
struct WideStage {
  static constexpr int PARAMS = M::P;  // every parameter feeds the whole residual
  static constexpr int NT = 1;
};
template <class M>
struct WideStage<M, decltype(void(M::STAGE1_PARAMS))> {
  static constexpr int PARAMS = M::STAGE1_PARAMS;
  static constexpr int NT = M::STAGE1_VALUES;
};

template <typename CT>
__device__ __forceinline__ void lds16(const CT* p, CT (&v)[16 / sizeof(CT)]);
template <>
__device__ __forceinline__ void lds16<float>(const float* p, float (&v)[4]) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <>
__device__ __forceinline__ void lds16<double>(const double* p, double (&v)[2]) {
  const double2 t = *reinterpret_cast<const double2*>(p);
  v[0] = t.x; v[1] = t.y;
}
template <typename CT>
__device__ __forceinline__ void sts16(CT* p, const CT* v);
template <>
__device__ __forceinline__ void sts16<float>(float* p, const float* v) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
template <>
__device__ __forceinline__ void sts16<double>(double* p, const double* v) {
  *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]);
}

// AFFINE_FD: as in dense_pass_kernel, for models with the affine / finish_diff hooks; parameters that only feed
// the second stage take M::tail_partials (the residual is affine in each of them alone, so the difference quotient
// in that parameter equals the partial derivative).  Used for fp32 compute, where the per-residual difference of
// two rounded ~1e3-pixel projections over h_j = sqrt(eps) |x_j| is mostly rounding noise.
template <class M, typename ST, typename CT, int THREADS, bool NUMERIC = true, bool AFFINE_FD = false>
__global__ void __launch_bounds__(THREADS, (sizeof(CT) == 4 ? 2 : 1)) wide_pass_kernel(const PassArgs a) {
  const int mode = a.mode_override >= 0 ? a.mode_override : *a.mode_ptr;
  if (mode == PASS_SKIP) return;
  if (peer_failed(a)) return;
  constexpr int P = M::P, O = M::O, NS = M::NS;
  constexpr int NRAW = P * (P + 1) / 2 + P + 1;
  constexpr int NCH = (NRAW + 31) / 32;
  constexpr int STRIDE = NCH * 32;              // doubles per warp in s_warp
  constexpr int NW = THREADS / 32;
  constexpr WideLayout L = wide_layout(P, O, int(sizeof(CT)));
  constexpr int NBJ = L.NBJ, NT = L.NT, NG = L.NG, PA = L.PA, PB = L.PB, ROW = L.ROW;
  constexpr int VPE = 16 / int(sizeof(CT));     // elements per 16-byte shared-memory access
  constexpr int NACC = 16;
  constexpr bool kFp32Acc = (sizeof(CT) == 4);
  constexpr int FLUSH_GROUPS = 8;               // fp32 lane partials are folded into fp64 every 8*32 residuals
  constexpr int NSETS = 1 + 2 * P;
  constexpr int SETN = wide_set_stride(M::SETN, int(sizeof(CT)));  // padded: a set is read with 16-byte loads
  constexpr int S1P = WideStage<M>::PARAMS;     // parameters >= S1P only feed the model's second stage
  constexpr int NTMP = WideStage<M>::NT;        // values the first stage hands to the second
  static_assert(NT >= 1 && NT <= 32 && NG >= 1, "wide_pass_kernel: more than 32 tiles of J^T B");

  extern __shared__ __align__(16) unsigned char wide_smem[];
  CT* s_tile = reinterpret_cast<CT*>(wide_smem);                       // [NW][32][ROW]
  CT* s_sets = s_tile + size_t(NW) * 32 * ROW;                         // [NSETS][SETN]
  CT* s_invh = s_sets + NSETS * SETN;                                  // [P]
  CT* s_cov = s_invh + P;                                              // [O*O]
  __shared__ double s_warp[NW * STRIDE];
  __shared__ double s_tot[STRIDE];

  const int jac = a.cost->jacobian;
  const bool central = (jac == MOPT_JAC_CENTRAL);
  const int nsets = !NUMERIC ? 1 : (central ? 1 + 2 * P : 1 + P);
  for (int i = threadIdx.x; i < nsets * SETN; i += THREADS) {
    const int si = i / SETN, k = i % SETN;
    double v = (k < M::SETN) ? a.pb->sets[si][k] : 0.0;
    if (AFFINE_FD && si >= 1 && si <= P && k < M::SETN) {  // D_j = (set(x + h_j e_j) - set_ref) / H_j, in fp64
      const int j = si - 1;
      v = central ? (v - a.pb->sets[1 + P + j][k]) / a.pb->hstep_cen[j] : (v - a.pb->sets[0][k]) / a.pb->hstep_fwd[j];
    }
    s_sets[i] = CT(v);
  }
  if (NUMERIC)
    for (int i = threadIdx.x; i < P; i += THREADS) {
      if (AFFINE_FD) s_invh[i] = CT(central ? a.pb->hstep_cen[i] : a.pb->hstep_fwd[i]);  // H_j itself in this mode
      else s_invh[i] = CT(central ? 1.0 / (2.0 * a.pb->h[i]) : 1.0 / a.pb->h[i]);
    }
  for (int i = threadIdx.x; i < O * O; i += THREADS) s_cov[i] = CT(a.cost->cov[i]);
  for (int i = threadIdx.x; i < NW * STRIDE; i += THREADS) s_warp[i] = 0.0;
  const bool has_cov = a.cost->has_cov != 0;
  const int loss = a.cost->loss;
  const CT lossp = CT(a.cost->loss_param);
  __syncthreads();

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool owner = lane < NT * NG;            // lanes beyond the tile x group grid only take part in phase 1
  const int grp = lane / NT;
  int bi = 0, bj = 0;                           // this lane's tile: block row bi, block column bj >= bi
  {
    int t = lane - grp * NT;
    while (t >= NBJ - bi) { t -= NBJ - bi; ++bi; }
    bj = bi + t;
  }
  CT* tile = s_tile + size_t(warp) * 32 * ROW;
  CT* my_row = tile + lane * ROW;
  const ST* __restrict__ sp[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) sp[s] = static_cast<const ST*>(a.streams.p[s]);

  CT acc[NACC], acc_e2 = CT(0);
  double dacc[NACC], dacc_e2 = 0.0;
#pragma unroll
  for (int c = 0; c < NACC; ++c) { acc[c] = CT(0); dacc[c] = 0.0; }

  // warps stride over groups of 32 consecutive residuals
  const int64_t ngroups = (a.n + 31) / 32;
  const int64_t wstride = int64_t(gridDim.x) * NW;
  int since_flush = 0;
  for (int64_t g = int64_t(blockIdx.x) * NW + warp; g < ngroups; g += wstride) {
    const int64_t i = g * 32 + lane;
    const bool valid = i < a.n;
    // ---- 1. this lane's residual row -------------------------------------------------------------
    CT e[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) e[s] = valid ? CT(sp[s][i]) : CT(0);
    CT r[O];
    CT tmp[NTMP];
    // a parameter set travels shared memory -> registers in 16-byte loads (loads of values the inlined model
    // does not read are dropped by the compiler)
    auto load_set = [&](int idx, CT (&sr)[SETN]) {
#pragma unroll
      for (int k = 0; k < SETN; k += VPE) {
        CT t[VPE];
        lds16<CT>(s_sets + idx * SETN + k, t);
#pragma unroll
        for (int u = 0; u < VPE; ++u) sr[k + u] = t[u];
      }
    };
    {
      CT sr[SETN];
      load_set(0, sr);
      if constexpr (S1P < P) {
        M::template stage1<CT>(sr, e, tmp);
        M::template stage2<CT>(sr, e, tmp, r);
      } else {
        M::template residual<CT>(sr, e, r);
      }
    }
    CT e2 = CT(0);
#pragma unroll
    for (int o = 0; o < O; ++o) e2 = fma(r[o], r[o], e2);
    CT w = valid ? loss_weight<CT>(loss, lossp, e2) : CT(0);
    if (!valid) e2 = CT(0);
    {
      CT s = e2;  // the warp's 32 squared norms
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) s += shfl_xor(s, off);
      acc_e2 += s;  // identical on every lane; lane 0's copy is the one reduced
    }
    if (mode != PASS_COST) {
      CT rowA[O * PA], rowB[O * PB];
#pragma unroll
      for (int k = 0; k < O * PA; ++k) rowA[k] = CT(0);
#pragma unroll
      for (int k = 0; k < O * PB; ++k) rowB[k] = CT(0);
      {
        CT J[O * P];
        if constexpr (NUMERIC && AFFINE_FD) {
          constexpr int NAFF = M::NAFF;
          CT s0[SETN], u0[NAFF];
          load_set(0, s0);
          M::template affine<CT>(s0, e, u0);
#pragma unroll
          for (int j = 0; j < S1P; ++j) {
            CT du[NAFF], d[O];
            {
              CT sr[SETN];
              load_set(1 + j, sr);
              M::template affine<CT>(sr, e, du);
            }
            if (central) {
              CT um[NAFF], sr[SETN];
              load_set(1 + P + j, sr);
              M::template affine<CT>(sr, e, um);
              M::template finish_diff<CT>(s0, um, du, s_invh[j], e, d);
            } else {
              M::template finish_diff<CT>(s0, u0, du, s_invh[j], e, d);
            }
#pragma unroll
            for (int o = 0; o < O; ++o) J[o * P + j] = d[o];
          }
          if constexpr (S1P < P) {
            CT Jt[O * (P - S1P)];
            M::template tail_partials<CT>(s0, tmp, Jt);
#pragma unroll
            for (int o = 0; o < O; ++o)
#pragma unroll
              for (int k = 0; k < P - S1P; ++k) J[o * P + S1P + k] = Jt[o * (P - S1P) + k];
          }
        } else if constexpr (NUMERIC) {
#pragma unroll
          for (int j = 0; j < P; ++j) {
            CT rp[O];
            auto eval = [&](int idx, CT (&out)[O]) {
              CT sr[SETN];
              load_set(idx, sr);
              if constexpr (S1P < P) {
                if (j >= S1P) M::template stage2<CT>(sr, e, tmp, out);
                else M::template residual<CT>(sr, e, out);
              } else {
                M::template residual<CT>(sr, e, out);
              }
            };
            eval(1 + j, rp);
            if (central) {
              CT rm[O];
              eval(1 + P + j, rm);
#pragma unroll
              for (int o = 0; o < O; ++o) J[o * P + j] = (rp[o] - rm[o]) * s_invh[j];
            } else {
#pragma unroll
              for (int o = 0; o < O; ++o) J[o * P + j] = (rp[o] - r[o]) * s_invh[j];
            }
          }
        } else {
          CT ra[O];  // the model's f_df (computeHessian, linearization.h:144); r above is the same f value
          CT sr[SETN];
          load_set(0, sr);
          M::template residual_jacobian<CT>(sr, e, ra, J);
        }
        // B = w C [J | r]   (C is the identity unless setCovariance was called; s_cov holds it)
        if (has_cov) {
#pragma unroll
          for (int o = 0; o < O; ++o) {
            CT cr = CT(0);
#pragma unroll
            for (int k = 0; k < O; ++k) cr = fma(s_cov[o + k * O], r[k], cr);
            rowB[o * PB + P] = w * cr;
#pragma unroll
            for (int p = 0; p < P; ++p) {
              CT cj = CT(0);
#pragma unroll
              for (int k = 0; k < O; ++k) cj = fma(s_cov[o + k * O], J[k * P + p], cj);
              rowA[o * PA + p] = J[o * P + p];
              rowB[o * PB + p] = w * cj;
            }
          }
        } else {
#pragma unroll
          for (int o = 0; o < O; ++o) {
            rowB[o * PB + P] = w * r[o];
#pragma unroll
            for (int p = 0; p < P; ++p) {
              rowA[o * PA + p] = J[o * P + p];
              rowB[o * PB + p] = w * J[o * P + p];
            }
          }
        }
        if (!valid) {  // past the end of the store (last group only): an all-zero row
#pragma unroll
          for (int k = 0; k < O * PA; ++k) rowA[k] = CT(0);
#pragma unroll
          for (int k = 0; k < O * PB; ++k) rowB[k] = CT(0);
        }
      }
#pragma unroll
      for (int k = 0; k < O * PA; k += VPE) sts16<CT>(my_row + k, rowA + k);
#pragma unroll
      for (int k = 0; k < O * PB; k += VPE) sts16<CT>(my_row + O * PA + k, rowB + k);
      __syncwarp();
      // ---- 2. C += J^T B over the 32 rows, register-tiled over the LI x LJ lane grid ----------------
      if (owner) {
#pragma unroll 2
        for (int row = grp; row < 32; row += NG) {
          const CT* rw = tile + row * ROW;
#pragma unroll
          for (int o = 0; o < O; ++o) {
            CT av[4], bv[4];
#pragma unroll
            for (int q = 0; q < 4; q += VPE) {
              CT t[VPE];
              lds16<CT>(rw + o * PA + bi * 4 + q, t);
#pragma unroll
              for (int u = 0; u < VPE; ++u) av[q + u] = t[u];
              lds16<CT>(rw + O * PA + o * PB + bj * 4 + q, t);
#pragma unroll
              for (int u = 0; u < VPE; ++u) bv[q + u] = t[u];
            }
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
              for (int u = 0; u < 4; ++u) acc[q * 4 + u] = fma(av[q], bv[u], acc[q * 4 + u]);
          }
        }
      }
      __syncwarp();
    }
    if (kFp32Acc && ++since_flush >= FLUSH_GROUPS) {
#pragma unroll
      for (int c = 0; c < NACC; ++c) { dacc[c] += double(acc[c]); acc[c] = CT(0); }
      dacc_e2 += double(acc_e2);
      acc_e2 = CT(0);
      since_flush = 0;
    }
  }
#pragma unroll
  for (int c = 0; c < NACC; ++c) dacc[c] += double(acc[c]);
  dacc_e2 += double(acc_e2);

  // merge the row groups of every tile, in group order, into the packed layout (H upper row-major, b, sum) of
  // this warp (s_warp was zeroed at kernel start)
  double* mine = s_warp + warp * STRIDE;
  for (int g = 0; g < NG; ++g) {
    if (owner && grp == g) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int ii = bi * 4 + q;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int jj = bj * 4 + u;
          if (ii < P && jj < P && ii <= jj) mine[tri_index(P, ii, jj)] += dacc[q * 4 + u];
          else if (ii < P && jj == P) mine[P * (P + 1) / 2 + ii] += dacc[q * 4 + u];
        }
      }
    }
    __syncwarp();
  }
  if (lane == 0) mine[NRAW - 1] = dacc_e2;
  __syncthreads();

  if (!grid_reduce_shared<NRAW, STRIDE, THREADS>(a, s_tot, s_warp)) return;
  if (mode == PASS_COST) {
    if (threadIdx.x == 0) a.out->v[NRAW - 1] = a.accumulate ? a.out->v[NRAW - 1] + s_tot[NRAW - 1] : s_tot[NRAW - 1];
  } else {
    for (int i = threadIdx.x; i < NRAW; i += THREADS) a.out->v[i] = a.accumulate ? a.out->v[i] + s_tot[i] : s_tot[i];
  }
  peer_push(a, NRAW);
}

template <class M, typename CT, int THREADS>
constexpr size_t wide_smem_bytes() {
  return wide_smem_bytes_rt(M::P, M::O, M::SETN, int(sizeof(CT)), THREADS);
}

#endif  // __CUDACC__
}  // namespace mopt
