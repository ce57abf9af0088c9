// Instantiations + dispatch of the point-to-point moment kernel (mopt_pass.cuh).
#include "mopt_internal.h"

namespace mopt {

namespace {

// Launch shapes (profiles/r1_tune_p2p.txt): the fp32 kernel is bound by bytes in flight, not by its ALU
// work, and does best with the whole SM's 32 warps x 6 outstanding 16-byte loads (64 registers/thread).
struct ShapeF32 {
  static constexpr int THREADS = 1024, MINB = 1, UNROLL = 1, FLUSH = 16;
};
// fp64 compute (the reference's default Scalar): capped at 128 registers so two CTAs stay resident — 16 warps hide the
// DFMA latency that 8 could not.  f32 store 873 -> 622 us per 100 M, f64 store 553 -> 380 us per 50 M (6.3 TB/s)
// (profiles/r1_tune_p2p_f64.txt).
struct ShapeF64 {
  static constexpr int THREADS = 256, MINB = 2, UNROLL = 2, FLUSH = 8;
};

template <typename ST, typename CT, int LOSS, bool QROT, class S, bool FUSED>
int launch_fused(const PassLaunch& L, const PassArgs& a) {
  auto kern = p2p_moment_kernel<ST, CT, LOSS, QROT, S::THREADS, S::MINB, S::UNROLL, S::FLUSH, FUSED>;
  const int64_t groups = a.n / VecOf<ST>::N;
  // small problems: keep CTAs at 256 threads' worth of work granularity by capping the grid, never below 1
  const int grid = pick_grid(reinterpret_cast<const void*>(kern), S::THREADS, L, groups);
  kern<<<grid, S::THREADS, 0, L.stream>>>(a);
  MOPT_CUDA_TRY(cudaGetLastError());
  return MOPT_OK;
}

// PassArgs::fused_setup (host-driven analytical passes): the instantiation that runs model->setup(x) itself
template <typename ST, typename CT, int LOSS, bool QROT, class S>
int launch_one(const PassLaunch& L, const PassArgs& a) {
  return a.fused_setup ? launch_fused<ST, CT, LOSS, QROT, S, true>(L, a) : launch_fused<ST, CT, LOSS, QROT, S, false>(L, a);
}

template <typename ST, typename CT, class S>
int launch_loss(const PassLaunch& L, int loss, bool qrot, const PassArgs& a) {
  switch (loss) {
    case MOPT_LOSS_NONE:
      return qrot ? launch_one<ST, CT, MOPT_LOSS_NONE, true, S>(L, a) : launch_one<ST, CT, MOPT_LOSS_NONE, false, S>(L, a);
    case MOPT_LOSS_GEMAN_MCCLURE:
      return qrot ? launch_one<ST, CT, MOPT_LOSS_GEMAN_MCCLURE, true, S>(L, a)
                  : launch_one<ST, CT, MOPT_LOSS_GEMAN_MCCLURE, false, S>(L, a);
    case MOPT_LOSS_HUBER:
      return qrot ? launch_one<ST, CT, MOPT_LOSS_HUBER, true, S>(L, a) : launch_one<ST, CT, MOPT_LOSS_HUBER, false, S>(L, a);
    default:
      set_last_error("unknown loss kind");
      return MOPT_ERR_INVALID_ARGUMENT;
  }
}

}  // namespace

int launch_p2p_moment(const PassLaunch& L, int store_dtype, int compute_dtype, int loss, bool qrot, const PassArgs& a) {
  return with_dtypes(store_dtype, compute_dtype, [&](auto st, auto ct) {
    using ST = decltype(st);
    using CT = decltype(ct);
    if constexpr (sizeof(CT) == 4) {
      if (L.threads == 1024) return launch_loss<ST, CT, ShapeF32>(L, loss, qrot, a);  // first generation (A/B)
      return launch_p2p_moment_gen2(L, loss, qrot, a);  // mopt_pass_p2p2.cu
    } else {
      return launch_loss<ST, CT, ShapeF64>(L, loss, qrot, a);
    }
  });
}

}  // namespace mopt
