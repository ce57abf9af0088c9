// Instantiations of the hypothesis scoring kernel (mopt_hyp.cuh) for the builtin models with parameters, and the
// batched set-up of the hypotheses, which is the same for every builtin model.
#include "mopt_hyp.cuh"
#include "mopt_internal.h"

namespace mopt {
namespace {

__global__ void hypothesis_setup_kernel(const CostDev* c, const double* xs, int n, double* sets) {
  setup_hypotheses(*c, xs, n, sets);
}

}  // namespace

int launch_hypothesis_setup(cudaStream_t stream, const CostDev* c, const double* xs, int n, double* sets) {
  hypothesis_setup_kernel<<<(n + 31) / 32, 32, 0, stream>>>(c, xs, n, sets);
  MOPT_CUDA_TRY(cudaGetLastError());
  return MOPT_OK;
}

// Models without parameters (point_dist) have nothing to score: mopt_score_hypotheses rejects them.
int hypothesis_score_kernel_desc(int model, int store_dtype, int compute_dtype, KernelDesc* k) {
  return with_builtin_model(model, [&](auto m) {
    using M = decltype(m);
    if constexpr (M::P == 0) {
      set_last_error("internal error: no hypothesis scoring kernel for a model without parameters");
      return MOPT_ERR_CUDA;
    } else {
      return with_dtypes(store_dtype, compute_dtype, [&](auto st, auto ct) {
        *k = builtin_kernel(reinterpret_cast<const void*>(hypothesis_score_kernel<M, decltype(st), decltype(ct)>),
                            kHypThreads);
        return MOPT_OK;
      });
    }
  });
}

}  // namespace mopt
