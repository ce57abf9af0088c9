// Instantiations of the per-residual evaluation kernel (mopt_eval.cuh) for the builtin models.
#include "mopt_eval.cuh"
#include "mopt_internal.h"

namespace mopt {

int evaluate_kernel_desc(int model, int store_dtype, int compute_dtype, bool f64_out, KernelDesc* k) {
  return with_builtin_model(model, [&](auto m) {
    return with_dtypes(store_dtype, compute_dtype, [&](auto st, auto ct) {
      using M = decltype(m);
      using ST = decltype(st);
      using CT = decltype(ct);
      *k = f64_out ? builtin_kernel(reinterpret_cast<const void*>(evaluate_kernel<M, ST, CT, double>), kEvalThreads)
                   : builtin_kernel(reinterpret_cast<const void*>(evaluate_kernel<M, ST, CT, float>), kEvalThreads);
      return MOPT_OK;
    });
  });
}

}  // namespace mopt
