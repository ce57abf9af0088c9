// Instantiations + dispatch of the per-residual evaluation kernel (mopt_eval.cuh) for the builtin models.
#include "mopt_eval.cuh"
#include "mopt_internal.h"

namespace mopt {
namespace {

template <class M, typename ST, typename CT>
int launch_one(const PassLaunch& L, int out_dtype, const PassArgs& a, const EvalArgs& ev) {
  auto kf = evaluate_kernel<M, ST, CT, float>;
  auto kd = evaluate_kernel<M, ST, CT, double>;
  // One grid for both output dtypes (the smaller of their persistent grids), so that the statistics -- whose
  // summation order follows the grid -- do not depend on which outputs are written or in which dtype.
  const int64_t groups = ev.count / VecOf<ST>::N + 1;
  const int gf = pick_grid(reinterpret_cast<const void*>(kf), kEvalThreads, L, groups);
  const int gd = pick_grid(reinterpret_cast<const void*>(kd), kEvalThreads, L, groups);
  const int grid = gf < gd ? gf : gd;
  if (out_dtype == MOPT_F32) kf<<<grid, kEvalThreads, 0, L.stream>>>(a, ev);
  else kd<<<grid, kEvalThreads, 0, L.stream>>>(a, ev);
  MOPT_CUDA_TRY(cudaGetLastError());
  return MOPT_OK;
}

template <class M>
int launch_types(const PassLaunch& L, int store_dtype, int compute_dtype, int out_dtype, const PassArgs& a,
                 const EvalArgs& ev) {
  if (store_dtype == MOPT_F32 && compute_dtype == MOPT_F32) return launch_one<M, float, float>(L, out_dtype, a, ev);
  if (store_dtype == MOPT_F32 && compute_dtype == MOPT_F64) return launch_one<M, float, double>(L, out_dtype, a, ev);
  if (store_dtype == MOPT_F64 && compute_dtype == MOPT_F64) return launch_one<M, double, double>(L, out_dtype, a, ev);
  set_last_error("store dtype f64 with compute dtype f32 is not supported");
  return MOPT_ERR_UNSUPPORTED;
}

}  // namespace

int launch_evaluate(const PassLaunch& L, int model, int store_dtype, int compute_dtype, int out_dtype,
                    const PassArgs& a, const EvalArgs& ev) {
  switch (model) {
    case MOPT_MODEL_POINT2POINT: return launch_types<P2PModel>(L, store_dtype, compute_dtype, out_dtype, a, ev);
    case MOPT_MODEL_EXP_CURVE: return launch_types<ExpCurveModel>(L, store_dtype, compute_dtype, out_dtype, a, ev);
    case MOPT_MODEL_MICHAELIS_MENTEN:
      return launch_types<MichaelisMentenModel>(L, store_dtype, compute_dtype, out_dtype, a, ev);
    case MOPT_MODEL_PINHOLE: return launch_types<PinholeModel>(L, store_dtype, compute_dtype, out_dtype, a, ev);
    case MOPT_MODEL_POWELL: return launch_types<PowellModel>(L, store_dtype, compute_dtype, out_dtype, a, ev);
    case MOPT_MODEL_POINT_DIST: return launch_types<PointDistModel>(L, store_dtype, compute_dtype, out_dtype, a, ev);
    case MOPT_MODEL_PINHOLE_DISTORT:
      return launch_types<PinholeDistortModel>(L, store_dtype, compute_dtype, out_dtype, a, ev);
    default:
      set_last_error("unknown model kind");
      return MOPT_ERR_INVALID_ARGUMENT;
  }
}

}  // namespace mopt
