// Score Gram matrix (mopt_covariance_terms): one streaming sweep over a store at x that reduces
//   G = sum_i g_i g_i^T,  g_i = w_i J_i^T C r_i,   wsse = sum_i w_i r_i^T C r_i,   n_valid
// -- the "meat" of the sandwich covariance H^+ G H^+ and the noise level of the scaled one.  H, b and sum r^T r come
// from the pass kernels (mopt_pass.cuh); this kernel forms each residual's Jacobian the way the pass selected for the
// same problem forms it (CovJac below), so that G and H describe the same linearization.
// Raw layout: G upper triangle row-major (P(P+1)/2), wsse, n_valid.  The sums go through the pass kernels' warp ->
// CTA -> last-CTA reduction (grid_reduce, context partials / ticket): fixed order, identical bits from run to run.
// Two tiers: P <= 6 keeps the packed sums in per-thread registers like dense_pass_kernel; larger P stages each
// warp's 32 score rows in shared memory and lanes own 4 x 4 tiles of the upper triangle, like wide_pass_kernel.
// The model is a template parameter and mopt_models.cuh is not included: this header is also compiled by NVRTC
// for run-time compiled user models (mopt_rtc.cu), exactly like mopt_pass.cuh.
#pragma once

#include "mopt_common.cuh"
#include "mopt_pass.cuh"

namespace mopt {

constexpr int kCovThreads = 256;

// How a residual's Jacobian is formed: the form of the linearization pass launch_pass selects for the same problem.
enum CovJac : int {
  COV_JAC_ANALYTICAL = 0,  // the model's residual_jacobian (dense_pass_kernel / wide_pass_kernel with NUMERIC = false)
  COV_JAC_FD = 1,          // per-residual forward or central differences (NUMERIC, AFFINE_FD = false)
  COV_JAC_AFFINE_FD = 2,   // common-denominator differences of a model with an affine first stage (AFFINE_FD)
  COV_JAC_P2P_AFFINE = 3   // point2point: J(q) = J0 + q_x J1 + q_y J2 + q_z J3 from ParamBlock::jaff (moment kernel)
};

__host__ __device__ constexpr int cov_raw(int P) { return P * (P + 1) / 2 + 2; }

struct CovArgs {
  double* out;  // [cov_raw(P)] totals, written by the last CTA
  int qrot;     // COV_JAC_P2P_AFFINE: q = R p (analytical EXACT / LEFT variants) or q = p (the other forms)
};

#ifdef __CUDACC__

template <class M, typename ST, typename CT, int JAC>
__global__ void __launch_bounds__(kCovThreads) score_gram_kernel(const PassArgs a, const CovArgs cv) {
  constexpr int THREADS = kCovThreads, NW = THREADS / 32;
  constexpr int P = M::P, O = M::O, NS = M::NS, NSX = NS > 0 ? NS : 1;
  constexpr int NRAW = cov_raw(P);
  constexpr int VPE = 16 / int(sizeof(CT));
  constexpr int SETN = wide_set_stride(M::SETN > 0 ? M::SETN : 1, int(sizeof(CT)));  // 16-byte aligned sets
  constexpr bool NUMERIC = (JAC == COV_JAC_FD || JAC == COV_JAC_AFFINE_FD);
  constexpr int NSETS = NUMERIC ? 1 + 2 * P : 1;
  constexpr int S1P = WideStage<M>::PARAMS;  // parameters >= S1P only feed the model's second stage
  constexpr int NTMP = WideStage<M>::NT;
  constexpr bool kFp32Acc = (sizeof(CT) == 4);
  static_assert(P >= 1 && P <= kMaxP && NRAW <= kMaxRaw, "score_gram_kernel: parameter count");
  static_assert(JAC != COV_JAC_P2P_AFFINE || (P == 6 && O == 3 && NS == 6), "the affine form is point2point's");

  __shared__ __align__(16) CT s_sets[NSETS * SETN];
  __shared__ CT s_invh[P];
  __shared__ CT s_cov[O * O];
  __shared__ __align__(16) CT s_jaff[JAC == COV_JAC_P2P_AFFINE ? 4 * 3 * 8 : 1];  // [k][row a][col p], rows padded to 8

  // the parameter sets as the pass kernels stage them (dense_pass_kernel / wide_pass_kernel)
  const bool central = (a.cost->jacobian == MOPT_JAC_CENTRAL);
  const int nsets = !NUMERIC ? 1 : (central ? 1 + 2 * P : 1 + P);
  for (int i = threadIdx.x; i < nsets * SETN; i += THREADS) {
    const int si = i / SETN, k = i % SETN;
    double v = (k < M::SETN) ? a.pb->sets[si][k] : 0.0;
    if (JAC == COV_JAC_AFFINE_FD && si >= 1 && si <= P && k < M::SETN) {  // D_j = (set(x + h_j e_j) - set_ref) / H_j
      const int j = si - 1;
      v = central ? (v - a.pb->sets[1 + P + j][k]) / a.pb->hstep_cen[j] : (v - a.pb->sets[0][k]) / a.pb->hstep_fwd[j];
    }
    s_sets[i] = CT(v);
  }
  if (NUMERIC)
    for (int i = threadIdx.x; i < P; i += THREADS) {
      if (JAC == COV_JAC_AFFINE_FD) s_invh[i] = CT(central ? a.pb->hstep_cen[i] : a.pb->hstep_fwd[i]);  // H_j itself
      else s_invh[i] = CT(central ? 1.0 / (2.0 * a.pb->h[i]) : 1.0 / a.pb->h[i]);
    }
  if (JAC == COV_JAC_P2P_AFFINE)
    for (int i = threadIdx.x; i < 4 * 3 * 8; i += THREADS) {
      const int k = i / 24, row = (i / 8) % 3, col = i % 8;
      s_jaff[i] = col < 6 ? CT(a.pb->jaff[k][row * 6 + col]) : CT(0);
    }
  for (int i = threadIdx.x; i < O * O; i += THREADS) s_cov[i] = CT(a.cost->cov[i]);
  const bool has_cov = a.cost->has_cov != 0;
  const int loss = a.cost->loss;
  const CT lossp = CT(a.cost->loss_param);
  const bool masked = a.masked != 0;
  const bool qrot = cv.qrot != 0;
  __syncthreads();

  // a parameter set, shared memory -> registers; the 1 + 2P sets of the larger models are re-read at every use
  // (held across the streaming loop they would be spilled to local memory, see dense_pass_kernel's kReloadSets)
  constexpr bool kReloadSets = NUMERIC && (NSETS * SETN > 32);
  auto load_set = [&](int idx, CT (&sr)[SETN]) {
#pragma unroll
    for (int k = 0; k < SETN; k += VPE) {
      CT t[VPE];
      if constexpr (kReloadSets) lds16_reload(&s_sets[idx * SETN + k], t);
      else lds16<CT>(&s_sets[idx * SETN + k], t);
#pragma unroll
      for (int u = 0; u < VPE; ++u) sr[k + u] = t[u];
    }
  };

  // One element: its score g = w J^T C r and q = w r^T C r.  False for an element without a correspondence.
  auto score = [&](const CT (&e)[NSX], CT (&g)[P], CT& q) -> bool {
    if (NS > 0 && masked) {  // NaN in the first B-group stream: no correspondence, the residual is skipped
      const CT probe = e[(M::NA < NS) ? M::NA : 0];
      if (probe != probe) return false;
    }
    CT r[O], J[O * P];
    if constexpr (JAC == COV_JAC_P2P_AFFINE) {
      // p2p_moments: q = R p, r = (q + t) - y; the Jacobian at a = (QROT ? q : p)
      CT s0[SETN];
      load_set(0, s0);
      CT qv[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        qv[k] = fma(s0[k * 3 + 0], e[0], fma(s0[k * 3 + 1], e[1], s0[k * 3 + 2] * e[2]));
        r[k] = (qv[k] + s0[9 + k]) - e[3 + k];
      }
      const CT a0 = qrot ? qv[0] : e[0], a1 = qrot ? qv[1] : e[1], a2 = qrot ? qv[2] : e[2];
      // the 72 pieces in fp64 do not fit in registers next to the rest: re-read per element (fp32: kept)
#pragma unroll
      for (int row = 0; row < 3; ++row) {
        CT jk[4][8];
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
          for (int c = 0; c < 8; c += VPE) {
            CT t[VPE];
            if constexpr (sizeof(CT) == 8) lds16_reload(&s_jaff[(k * 3 + row) * 8 + c], t);
            else lds16<CT>(&s_jaff[(k * 3 + row) * 8 + c], t);
#pragma unroll
            for (int u = 0; u < VPE; ++u) jk[k][c + u] = t[u];
          }
#pragma unroll
        for (int c = 0; c < 6; ++c) J[row * 6 + c] = fma(a2, jk[3][c], fma(a1, jk[2][c], fma(a0, jk[1][c], jk[0][c])));
      }
    } else {
      CT tmp[NTMP];
      {
        CT s0[SETN];
        load_set(0, s0);
        if constexpr (S1P < P) {
          M::template stage1<CT>(s0, e, tmp);
          M::template stage2<CT>(s0, e, tmp, r);
        } else {
          M::template residual<CT>(s0, e, r);
        }
      }
      if constexpr (JAC == COV_JAC_AFFINE_FD) {
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
      } else if constexpr (JAC == COV_JAC_FD) {
#pragma unroll
        for (int j = 0; j < P; ++j) {
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
        CT ra[O], s0[SETN];
        load_set(0, s0);
        M::template residual_jacobian<CT>(s0, e, ra, J);
        if constexpr (S1P >= P) {  // the dense pass takes r from f_df itself
#pragma unroll
          for (int o = 0; o < O; ++o) r[o] = ra[o];
        }
      }
    }
    CT e2 = CT(0);
#pragma unroll
    for (int o = 0; o < O; ++o) e2 = fma(r[o], r[o], e2);
    const CT w = loss_weight<CT>(loss, lossp, e2);
    CT Cr[O];
#pragma unroll
    for (int o = 0; o < O; ++o) {
      CT s = CT(0);
#pragma unroll
      for (int k = 0; k < O; ++k) s = fma(s_cov[o + k * O], r[k], s);
      Cr[o] = has_cov ? s : r[o];
    }
    CT rc = CT(0);
#pragma unroll
    for (int o = 0; o < O; ++o) rc = fma(r[o], Cr[o], rc);
    q = w * rc;
#pragma unroll
    for (int i = 0; i < P; ++i) {  // the per-element term of b in dense_pass_kernel
      CT s = CT(0);
#pragma unroll
      for (int o = 0; o < O; ++o) s = fma(w * J[o * P + i], Cr[o], s);
      g[i] = s;
    }
    return true;
  };

  const ST* __restrict__ sp[NSX];
#pragma unroll
  for (int s = 0; s < NS; ++s) sp[s] = static_cast<const ST*>(a.streams.p[s]);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  if constexpr (P <= 6) {
    // ---- dense tier: the packed sums in registers, flushed to fp64 on dense_pass_kernel's schedule --------------
    constexpr int VEC = VecOf<ST>::N;
    constexpr int V = next_pow2(NRAW);
    constexpr int FLUSH_ROUNDS = 8;
    static_assert(V <= 32, "dense tier: the sums must fit one transposing-reduce chunk");
    __shared__ double s_warp[NW * V];
    __shared__ double s_tot[V];
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
    auto do_elem = [&](const CT (&e)[NSX]) {
      CT g[P], q;
      if (!score(e, g, q)) return;
      int idx = 0;
#pragma unroll
      for (int i = 0; i < P; ++i)
#pragma unroll
        for (int j = i; j < P; ++j, ++idx) acc[idx] = fma(g[i], g[j], acc[idx]);
      acc[NRAW - 2] += q;
      acc[NRAW - 1] += CT(1);
    };
    auto do_group = [&](int64_t g) {
      CT vals[NSX][VEC];
#pragma unroll
      for (int s = 0; s < NS; ++s) load_vec<ST, CT>(sp[s], g, vals[s]);
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        CT e[NSX];
        e[0] = CT(0);
#pragma unroll
        for (int s = 0; s < NS; ++s) e[s] = vals[s][v];
        do_elem(e);
      }
    };
    if constexpr (NS == 0) {
      // data-free model (Powell): `n` identical residual blocks evaluated by thread 0, as the pass does
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
          CT e[NSX];
#pragma unroll
          for (int s = 0; s < NS; ++s) e[s] = CT(sp[s][i]);
          do_elem(e);
        }
      }
    }
    flush();
    if (!grid_reduce<NRAW, V, 1, THREADS>(dacc, a, s_tot, s_warp)) return;
    for (int i = threadIdx.x; i < NRAW; i += THREADS) cv.out[i] = s_tot[i];
  } else {
    // ---- wide tier: 32 score rows per warp in shared memory, lanes own 4 x 4 tiles of the upper triangle ---------
    static_assert(NS > 0, "wide tier: streamed models only");
    constexpr int NB = (P + 3) / 4;             // 4-row blocks of g
    constexpr int NT = NB * (NB + 1) / 2;       // tiles on or above the block diagonal
    constexpr int NG = 32 / NT;                 // row groups: lane = group * NT + tile, group k takes rows k, k + NG, ...
    constexpr int PA = NB * 4;
    constexpr int ROW = ((PA / VPE) & 1) ? PA : PA + VPE;  // odd number of 16-byte units: conflict-free row stores
    constexpr int STRIDE = (NRAW + 31) / 32 * 32;
    constexpr int NACC = 16;
    constexpr int FLUSH_GROUPS = 8;
    constexpr size_t kTileBytes = sizeof(CT) * size_t(NW) * 32 * ROW;
    constexpr size_t kWarpBytes = sizeof(double) * size_t(NW) * STRIDE;
    // the row tiles and, after the streaming loop, the per-warp totals share one buffer
    __shared__ __align__(16) unsigned char s_buf[kTileBytes > kWarpBytes ? kTileBytes : kWarpBytes];
    __shared__ double s_tot[STRIDE];
    static_assert(NT >= 1 && NT <= 32 && NG >= 1, "wide tier: more than 32 tiles");

    const bool owner = lane < NT * NG;
    const int grp = lane / NT;
    int bi = 0, bj = 0;
    {
      int t = lane - grp * NT;
      while (t >= NB - bi) { t -= NB - bi; ++bi; }
      bj = bi + t;
    }
    CT* tile = reinterpret_cast<CT*>(s_buf) + size_t(warp) * 32 * ROW;
    CT* my_row = tile + lane * ROW;

    CT acc[NACC], acc_q = CT(0), acc_n = CT(0);
    double dacc[NACC], dacc_q = 0.0, dacc_n = 0.0;
#pragma unroll
    for (int c = 0; c < NACC; ++c) { acc[c] = CT(0); dacc[c] = 0.0; }

    const int64_t ngroups = (a.n + 31) / 32;
    const int64_t wstride = int64_t(gridDim.x) * NW;
    int since_flush = 0;
    for (int64_t gi = int64_t(blockIdx.x) * NW + warp; gi < ngroups; gi += wstride) {
      const int64_t i = gi * 32 + lane;
      CT row[PA], q = CT(0);
#pragma unroll
      for (int k = 0; k < PA; ++k) row[k] = CT(0);
      bool ok = false;
      if (i < a.n) {
        CT e[NSX];
#pragma unroll
        for (int s = 0; s < NS; ++s) e[s] = CT(sp[s][i]);
        CT g[P];
        ok = score(e, g, q);
        if (ok) {
#pragma unroll
          for (int k = 0; k < P; ++k) row[k] = g[k];
        } else {
          q = CT(0);
        }
      }
      {
        CT sq = q, sn = ok ? CT(1) : CT(0);  // the warp's 32 values; lane 0's copy is the one reduced
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
          sq += shfl_xor(sq, off);
          sn += shfl_xor(sn, off);
        }
        acc_q += sq;
        acc_n += sn;
      }
#pragma unroll
      for (int k = 0; k < PA; k += VPE) sts16<CT>(my_row + k, row + k);
      __syncwarp();
      if (owner) {
#pragma unroll 2
        for (int rr = grp; rr < 32; rr += NG) {
          const CT* rw = tile + rr * ROW;
          CT av[4], bv[4];
#pragma unroll
          for (int k = 0; k < 4; k += VPE) {
            CT t[VPE];
            lds16<CT>(rw + bi * 4 + k, t);
#pragma unroll
            for (int u = 0; u < VPE; ++u) av[k + u] = t[u];
            lds16<CT>(rw + bj * 4 + k, t);
#pragma unroll
            for (int u = 0; u < VPE; ++u) bv[k + u] = t[u];
          }
#pragma unroll
          for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int u = 0; u < 4; ++u) acc[k * 4 + u] = fma(av[k], bv[u], acc[k * 4 + u]);
        }
      }
      __syncwarp();
      if (kFp32Acc && ++since_flush >= FLUSH_GROUPS) {
#pragma unroll
        for (int c = 0; c < NACC; ++c) { dacc[c] += double(acc[c]); acc[c] = CT(0); }
        dacc_q += double(acc_q);
        dacc_n += double(acc_n);
        acc_q = CT(0);
        acc_n = CT(0);
        since_flush = 0;
      }
    }
#pragma unroll
    for (int c = 0; c < NACC; ++c) dacc[c] += double(acc[c]);
    dacc_q += double(acc_q);
    dacc_n += double(acc_n);

    // every warp is done with its tile: the buffer now holds the per-warp totals, merged tile by tile in group order
    __syncthreads();
    double* s_warp = reinterpret_cast<double*>(s_buf);
    for (int k = threadIdx.x; k < NW * STRIDE; k += THREADS) s_warp[k] = 0.0;
    __syncthreads();
    double* mine = s_warp + warp * STRIDE;
    for (int gg = 0; gg < NG; ++gg) {
      if (owner && grp == gg) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int ii = bi * 4 + k;
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int jj = bj * 4 + u;
            if (ii <= jj && jj < P) mine[tri_index(P, ii, jj)] += dacc[k * 4 + u];
          }
        }
      }
      __syncwarp();
    }
    if (lane == 0) {
      mine[NRAW - 2] = dacc_q;
      mine[NRAW - 1] = dacc_n;
    }
    __syncthreads();
    if (!grid_reduce_shared<NRAW, STRIDE, THREADS>(a, s_tot, s_warp)) return;
    for (int i = threadIdx.x; i < NRAW; i += THREADS) cv.out[i] = s_tot[i];
  }
}

#endif  // __CUDACC__

}  // namespace mopt
