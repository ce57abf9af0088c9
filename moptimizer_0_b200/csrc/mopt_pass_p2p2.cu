// Instantiations + dispatch of the second-generation point-to-point moment kernel (mopt_pass_p2p2.cuh): fp32 store,
// fp32 compute.  Its own translation unit so that the library builds in parallel.
#include "mopt_internal.h"
#include "mopt_pass_p2p2.cuh"

namespace mopt {
namespace {

// Second-generation fp32 kernel (mopt_pass_p2p2.cuh): TMA bulk-copy ring + packed fp32 arithmetic.  Shapes from the
// same-box sustained sweeps (profiles/r2_tune_gen2_*.txt): 384 threads x 2 stages x 2 float4 groups per thread and
// stream (72 KB stages, 144 KB ring) reads within 1 % of the bare read-and-sum ceiling on both boxes measured;
// 512 x 3 x 1 is as fast on one of them (csrc/tune_p2p.cu keeps that shape for A/B).  mopt_ctx_set_launch(.., 1024)
// selects the first-generation kernel (mopt_pass_p2p.cu).
struct ShapeGen2 {
  static constexpr int THREADS = 384, STAGES = 2, U = 2, FLUSH = 16;
};

// ---- second generation (fp32 store, fp32 compute) ----------------------------------------------------------
template <int LOSS, bool QROT, bool MASKED, bool FUSED, class S>
int launch_gen2_one(const PassLaunch& L, const PassArgs& a0) {
  constexpr auto kern = p2p_moment2_kernel<LOSS, QROT, MASKED, FUSED, S::THREADS, 1, S::STAGES, S::U, S::FLUSH>;
  constexpr size_t smem = p2p2_ring_bytes(S::THREADS, S::STAGES, S::U);
  MOPT_TRY(allow_dyn_smem<kern>(smem));
  PassArgs a = a0;
  // the bulk copies need 16-byte aligned sources; anything else streams through the kernel's direct-load path
  for (int k = 0; k < 6; ++k)
    if (reinterpret_cast<uintptr_t>(a.streams.p[k]) & 15u) a.no_ring = 1;
  const int64_t groups = a.n / 4;
  int64_t grid = int64_t(L.ctas_per_sm > 0 ? L.ctas_per_sm : 1) * L.num_sms;  // one CTA per SM owns the whole ring
  if (grid > L.num_sms) grid = L.num_sms;
  const int64_t need = (groups + S::THREADS - 1) / S::THREADS;
  if (need < grid) grid = need;
  if (grid < 1) grid = 1;
  kern<<<int(grid), S::THREADS, smem, L.stream>>>(a);
  MOPT_CUDA_TRY(cudaGetLastError());
  return MOPT_OK;
}

template <int LOSS, bool QROT, class S>
int launch_gen2_flags(const PassLaunch& L, const PassArgs& a) {
  if (a.masked)
    return a.fused_setup ? launch_gen2_one<LOSS, QROT, true, true, S>(L, a) : launch_gen2_one<LOSS, QROT, true, false, S>(L, a);
  return a.fused_setup ? launch_gen2_one<LOSS, QROT, false, true, S>(L, a) : launch_gen2_one<LOSS, QROT, false, false, S>(L, a);
}

template <class S>
int launch_gen2(const PassLaunch& L, int loss, bool qrot, const PassArgs& a) {
  switch (loss) {
    case MOPT_LOSS_NONE:
      return qrot ? launch_gen2_flags<MOPT_LOSS_NONE, true, S>(L, a) : launch_gen2_flags<MOPT_LOSS_NONE, false, S>(L, a);
    case MOPT_LOSS_GEMAN_MCCLURE:
      return qrot ? launch_gen2_flags<MOPT_LOSS_GEMAN_MCCLURE, true, S>(L, a)
                  : launch_gen2_flags<MOPT_LOSS_GEMAN_MCCLURE, false, S>(L, a);
    case MOPT_LOSS_HUBER:
      return qrot ? launch_gen2_flags<MOPT_LOSS_HUBER, true, S>(L, a) : launch_gen2_flags<MOPT_LOSS_HUBER, false, S>(L, a);
    default:
      set_last_error("unknown loss kind");
      return MOPT_ERR_INVALID_ARGUMENT;
  }
}

}  // namespace

int launch_p2p_moment_gen2(const PassLaunch& L, int loss, bool qrot, const PassArgs& a) {
  return launch_gen2<ShapeGen2>(L, loss, qrot, a);
}

}  // namespace mopt
