// Instantiations + dispatch of the wide pass kernel (mopt_pass.cuh): models with more than 32 packed sums (is_wide).
#include "mopt_internal.h"
#include "mopt_pass_wide_tc.cuh"

namespace mopt {
namespace {

constexpr int kThreads = 256;

template <class M, typename ST, typename CT, bool AFFINE_FD>
int launch_one(const PassLaunch& L, const PassArgs& a) {
  constexpr auto kern = wide_pass_kernel<M, ST, CT, kThreads, true, AFFINE_FD>;
  constexpr size_t smem = wide_smem_bytes<M, CT, kThreads>();
  MOPT_TRY(allow_dyn_smem<kern>(smem));  // the large dynamic shared-memory tile
  PassLaunch L2 = L;
  L2.ctas_per_sm = 0;
  const int grid = pick_grid(reinterpret_cast<const void*>(kern), kThreads, L2, a.n, smem);  // one residual per lane per sweep
  kern<<<grid, kThreads, smem, L.stream>>>(a);
  MOPT_CUDA_TRY(cudaGetLastError());
  return MOPT_OK;
}

// Second generation, fp32 only: packed-fp32 finite differences + Gram matrix on the tensor cores (mopt_pass_wide_tc.cuh).
template <class M>
int launch_tc(const PassLaunch& L, const PassArgs& a) {
  constexpr int kTcThreads = 256;
  constexpr auto kern = wide_tc_kernel<M, kTcThreads, 2>;
  constexpr size_t smem = wide_tc_smem_bytes(M::O, M::SETN, M::P, kTcThreads);
  MOPT_TRY(allow_dyn_smem<kern>(smem));
  // two observations per lane per sweep
  const int grid = pick_grid(reinterpret_cast<const void*>(kern), kTcThreads, L, (a.n + 1) / 2, smem);
  kern<<<grid, kTcThreads, smem, L.stream>>>(a);
  MOPT_CUDA_TRY(cudaGetLastError());
  return MOPT_OK;
}

}  // namespace

int launch_wide(const PassLaunch& L, int model, int store_dtype, int compute_dtype, const PassArgs& a) {
  return with_builtin_model(model, [&](auto m) {
    using M = decltype(m);
    if constexpr (!is_wide(M::P)) {
      set_last_error("internal error: a dense model on the wide pass");
      return MOPT_ERR_CUDA;
    } else {
      return with_dtypes(store_dtype, compute_dtype, [&](auto st, auto ct) {
        using ST = decltype(st);
        using CT = decltype(ct);
        // fp32 store + fp32 compute, common-denominator finite differences, C = I: the tensor-core kernel
        // (mopt_ctx_set_launch(.., 1024) keeps the first-generation kernel for A/B on the same box)
        if constexpr (sizeof(ST) == 4 && sizeof(CT) == 4) {
          if (L.affine_fd && L.identity_cov && !a.masked && L.threads != 1024) return launch_tc<M>(L, a);
        }
        // L.affine_fd (launch_pass): common-denominator finite differences (wide_pass_kernel AFFINE_FD) — the default
        // with fp32 compute unless MOPT_FLAG_GENERIC_KERNEL asks for the per-residual form; fp64 compute is the
        // literal restatement of the reference unless MOPT_FLAG_STABLE_FD opts in
        return L.affine_fd ? launch_one<M, ST, CT, true>(L, a) : launch_one<M, ST, CT, false>(L, a);
      });
    }
  });
}

}  // namespace mopt
