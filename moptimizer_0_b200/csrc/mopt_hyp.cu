// Instantiations + dispatch of the hypothesis scoring kernel (mopt_hyp.cuh) for the builtin models with parameters,
// and the batched set-up of the hypotheses, which is the same for every builtin model.
#include "mopt_hyp.cuh"
#include "mopt_internal.h"

namespace mopt {
namespace {

__global__ void hypothesis_setup_kernel(const CostDev* c, const double* xs, int n, double* sets) {
  setup_hypotheses(*c, xs, n, sets);
}

template <class M, typename ST, typename CT>
int launch_one(const PassLaunch& L, const PassArgs& a, const HypArgs& h) {
  auto k = hypothesis_score_kernel<M, ST, CT>;
  // the grid follows the elements only: the CTA partition of the data, and with it every per-CTA partial, is the
  // same whatever the batch
  const int grid = pick_grid(reinterpret_cast<const void*>(k), kHypThreads, L, h.count / VecOf<ST>::N + 1);
  const dim3 g(unsigned(grid), unsigned((h.n_hyp + kHypTile - 1) / kHypTile));
  k<<<g, kHypThreads, 0, L.stream>>>(a, h);
  MOPT_CUDA_TRY(cudaGetLastError());
  return MOPT_OK;
}

template <class M>
int launch_types(const PassLaunch& L, int store_dtype, int compute_dtype, const PassArgs& a, const HypArgs& h) {
  if (store_dtype == MOPT_F32 && compute_dtype == MOPT_F32) return launch_one<M, float, float>(L, a, h);
  if (store_dtype == MOPT_F32 && compute_dtype == MOPT_F64) return launch_one<M, float, double>(L, a, h);
  if (store_dtype == MOPT_F64 && compute_dtype == MOPT_F64) return launch_one<M, double, double>(L, a, h);
  set_last_error("store dtype f64 with compute dtype f32 is not supported");
  return MOPT_ERR_UNSUPPORTED;
}

}  // namespace

int launch_hypothesis_setup(cudaStream_t stream, const CostDev* c, const double* xs, int n, double* sets) {
  hypothesis_setup_kernel<<<(n + 31) / 32, 32, 0, stream>>>(c, xs, n, sets);
  MOPT_CUDA_TRY(cudaGetLastError());
  return MOPT_OK;
}

// Models without parameters (point_dist) have nothing to score: mopt_score_hypotheses rejects them.
int launch_hypothesis_score(const PassLaunch& L, int model, int store_dtype, int compute_dtype, const PassArgs& a,
                            const HypArgs& h) {
  switch (model) {
    case MOPT_MODEL_POINT2POINT: return launch_types<P2PModel>(L, store_dtype, compute_dtype, a, h);
    case MOPT_MODEL_EXP_CURVE: return launch_types<ExpCurveModel>(L, store_dtype, compute_dtype, a, h);
    case MOPT_MODEL_MICHAELIS_MENTEN: return launch_types<MichaelisMentenModel>(L, store_dtype, compute_dtype, a, h);
    case MOPT_MODEL_PINHOLE: return launch_types<PinholeModel>(L, store_dtype, compute_dtype, a, h);
    case MOPT_MODEL_POWELL: return launch_types<PowellModel>(L, store_dtype, compute_dtype, a, h);
    case MOPT_MODEL_PINHOLE_DISTORT: return launch_types<PinholeDistortModel>(L, store_dtype, compute_dtype, a, h);
    default:
      set_last_error("unknown model kind, or a model without parameters");
      return MOPT_ERR_INVALID_ARGUMENT;
  }
}

}  // namespace mopt
