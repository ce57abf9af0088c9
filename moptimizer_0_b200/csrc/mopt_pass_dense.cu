// Instantiations + dispatch of the generic dense pass kernel (mopt_pass.cuh): models with at most 32 packed sums.
#include "mopt_internal.h"
#include "mopt_pass_dense_f2.cuh"

namespace mopt {
namespace {

constexpr int kThreads = 256;

template <class M, typename ST, typename CT, bool NUMERIC, int THREADS, int MINB, bool AFFINE_FD = false>
int launch_shape(const PassLaunch& L, const PassArgs& a) {
  auto kern = dense_pass_kernel<M, ST, CT, NUMERIC, THREADS, MINB, AFFINE_FD>;
  const int64_t groups = (M::NS == 0) ? 1 : a.n / VecOf<ST>::N;
  PassLaunch L2 = L;
  L2.ctas_per_sm = 0;
  const int grid = pick_grid(reinterpret_cast<const void*>(kern), THREADS, L2, groups);
  kern<<<grid, THREADS, 0, L.stream>>>(a);
  MOPT_CUDA_TRY(cudaGetLastError());
  return MOPT_OK;
}

// Second generation for fp32 finite differences of models with an affine first stage (mopt_pass_dense_f2.cuh): two
// observations per thread in packed fp32, 256 threads x 2 CTAs per SM.
template <class M>
int launch_f2(const PassLaunch& L, const PassArgs& a) {
  auto kern = dense_f2_kernel<M, kThreads, 2>;
  PassLaunch L2 = L;
  L2.ctas_per_sm = 0;
  const int grid = pick_grid(reinterpret_cast<const void*>(kern), kThreads, L2, a.n / 4);
  kern<<<grid, kThreads, 0, L.stream>>>(a);
  MOPT_CUDA_TRY(cudaGetLastError());
  return MOPT_OK;
}

template <class M, typename ST, typename CT, bool NUMERIC>
int launch_one(const PassLaunch& L, const PassArgs& a) {
  // Finite-difference kernels of the 6-parameter models want all 1 + 2P parameter sets in registers (247-255
  // registers, one 256-thread CTA per SM, issue slots 34 % busy).  Capping them at 80 registers (3 CTAs per SM)
  // turns the hoisted sets into L1-resident local loads and triples the warps that hide the division / MUFU
  // latency: camera 50 M central 2.55 -> 1.37 ms, forward 2.12 -> 0.96 ms (profiles/r1_tune_dense.txt).
  // fp64 compute: 2 CTAs/SM (128 registers) pays off while the Jacobian is small (camera O x P = 12: 3.88 -> 2.82 ms);
  // with the 3 x 6 point2point Jacobian in doubles the cap spills 400 bytes and loses (3.4 -> 4.6 ms), so that stays at 1.
  constexpr int kMinB = (NUMERIC && M::P >= 4) ? (sizeof(CT) == 4 ? 3 : (M::O * M::P <= 12 ? 2 : 1)) : 1;
  // Finite differences of a model with an affine first stage: common-denominator difference quotient
  // (dense_pass_kernel AFFINE_FD).  launch_pass sets L.affine_fd: on by default with fp32 compute (off with
  // MOPT_FLAG_GENERIC_KERNEL), off by default with fp64 compute — the literal form is the one compared with the
  // reference's fp64 arithmetic — and on with MOPT_FLAG_STABLE_FD.
  if constexpr (NUMERIC && HasAffineStage<M>::value) {
    if constexpr (sizeof(ST) == 4 && sizeof(CT) == 4) {
      // fp32, C = I, no NaN-masked rows: two observations per thread in packed fp32
      // (mopt_ctx_set_launch(.., 1024) keeps dense_pass_kernel for A/B on the same box)
      if (L.affine_fd && L.identity_cov && !a.masked && L.threads != 1024) return launch_f2<M>(L, a);
    }
    if (a.fused_setup) {  // can_fuse_setup (mopt_capi.cu) mirrors the condition above
      set_last_error("internal error: fused set-up requested for a kernel that reads the ParamBlock");
      return MOPT_ERR_CUDA;
    }
    if (L.affine_fd) return launch_shape<M, ST, CT, NUMERIC, kThreads, kMinB, true>(L, a);
  }
  if (a.fused_setup) {
    set_last_error("internal error: fused set-up requested for a kernel that reads the ParamBlock");
    return MOPT_ERR_CUDA;
  }
  return launch_shape<M, ST, CT, NUMERIC, kThreads, kMinB>(L, a);
}

}  // namespace

int launch_dense(const PassLaunch& L, int model, bool numeric, int store_dtype, int compute_dtype, const PassArgs& a) {
  return with_builtin_model(model, [&](auto m) {
    using M = decltype(m);
    if constexpr (is_wide(M::P)) {
      set_last_error("internal error: a wide model on the dense pass");
      return MOPT_ERR_CUDA;
    } else {
      return with_dtypes(store_dtype, compute_dtype, [&](auto st, auto ct) {
        using ST = decltype(st);
        using CT = decltype(ct);
        // cost-only passes of Jacobian-free models still come through here with numeric == false
        if (numeric || !M::HAS_JAC) return launch_one<M, ST, CT, true>(L, a);
        return launch_one<M, ST, CT, false>(L, a);
      });
    }
  });
}

}  // namespace mopt
