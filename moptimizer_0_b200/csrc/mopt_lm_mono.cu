// Instantiations + dispatch of the persistent LM kernel for small problems (mopt_lm_mono.cuh).  Its own translation
// unit so that the library builds in parallel.
#include <mutex>

#include "mopt_internal.h"
#include "mopt_lm_mono.cuh"

namespace mopt {
namespace {

struct ShapeMono {  // small CTAs: more of them share a small problem; one per SM so the optimizer step does not spill
  static constexpr int THREADS = 256, MINB = 1, UNROLL = 2, FLUSH = 8;
};

template <typename ST, typename CT>
int launch_mono_loss(const PassLaunch& L, int loss, bool qrot, const PassArgs& a, const MonoArgs& m) {
  using S = ShapeMono;
  if (loss < MOPT_LOSS_NONE || loss > MOPT_LOSS_HUBER) {
    set_last_error("unknown loss kind");
    return MOPT_ERR_INVALID_ARGUMENT;
  }
  auto kern = p2p_lm_mono_kernel<ST, CT, S::THREADS, S::MINB, S::UNROLL, S::FLUSH>;
  const int64_t groups = a.n / VecOf<ST>::N;
  // data CTAs as the pass kernel would size them, plus CTA 0 (the optimizer); all co-resident
  // (the occupancy query behind pick_grid costs microseconds: once per instantiation and launch shape)
  static std::mutex mu;
  static int cached_key = -1, cached_co = 0;
  const int key = L.num_sms * 64 + L.ctas_per_sm;
  int co_resident;
  {
    std::lock_guard<std::mutex> lock(mu);
    if (cached_key != key) {
      cached_co = pick_grid(reinterpret_cast<const void*>(kern), S::THREADS, L, int64_t(1) << 40);
      cached_key = key;
    }
    co_resident = cached_co;
  }
  int64_t need = (groups + S::THREADS - 1) / S::THREADS;
  int data = int(need < co_resident - 1 ? need : co_resident - 1);
  if (data < 1) data = 1;
  const int grid = data + 1;
  PassArgs aa = a;
  MonoArgs mm = m;
  mm.loss = loss;
  mm.qrot = qrot ? 1 : 0;
  void* params[] = {&aa, &mm};
  MOPT_CUDA_TRY(cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(kern), dim3(grid), dim3(S::THREADS), params, 0,
                                            L.stream));
  return MOPT_OK;
}
}  // namespace

int launch_p2p_lm_mono(const PassLaunch& L, int store_dtype, int compute_dtype, int loss, bool qrot, const PassArgs& a,
                       const MonoArgs& m) {
  return with_dtypes(store_dtype, compute_dtype, [&](auto st, auto ct) {
    return launch_mono_loss<decltype(st), decltype(ct)>(L, loss, qrot, a, m);
  });
}


}  // namespace mopt
