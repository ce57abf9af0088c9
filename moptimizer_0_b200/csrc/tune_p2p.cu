// Stand-alone tuning harness (NOT part of libmopt_b200.so): times launch-shape variants of the
// point2point moment kernel and a bare 6-stream read-and-sum kernel (the practical HBM read ceiling)
// on 100 M synthetic correspondences.  Build: python -m moptimizer_0_b200.build --tune
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "mopt_pass.cuh"
#include "mopt_pass_p2p2.cuh"

namespace mopt {
void set_last_error(const std::string&) {}
}
using namespace mopt;

#define CK(x)                                                                    \
  do {                                                                           \
    cudaError_t e = (x);                                                         \
    if (e != cudaSuccess) {                                                      \
      std::printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); \
      std::exit(1);                                                              \
    }                                                                            \
  } while (0)

__global__ void fill_kernel(float* p, int64_t n, unsigned seed) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    unsigned h = unsigned(i) * 2654435761u + seed;
    h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
    p[i] = float(h >> 8) * (10.0f / 16777216.0f);
  }
}

// tgt = R src + t + small noise, 5 % large outliers: the benchmark's data regime (most residuals are inliers)
__global__ void make_targets_kernel(const float* sx, const float* sy, const float* sz, float* tx, float* ty, float* tz,
                                    int64_t n) {
  const float R[12] = {0.99f, -0.08f, 0.05f, 0.08f, 0.99f, -0.1f, -0.05f, 0.1f, 0.99f, 0.5f, -0.3f, 0.2f};
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    unsigned h = unsigned(i) * 747796405u + 2891336453u;
    h ^= h >> 16; h *= 2246822519u; h ^= h >> 13;
    const float noise = (float(h & 0xffff) / 65536.0f - 0.5f) * 0.02f;
    const float out = ((h >> 16) % 20 == 0) ? 0.7f : 0.0f;
    tx[i] = R[0] * sx[i] + R[1] * sy[i] + R[2] * sz[i] + R[9] + noise + out;
    ty[i] = R[3] * sx[i] + R[4] * sy[i] + R[5] * sz[i] + R[10] - noise;
    tz[i] = R[6] * sx[i] + R[7] * sy[i] + R[8] * sz[i] + R[11] + noise * 0.5f;
  }
}

// Bare ceiling: same access pattern (6 planar streams, 16-byte streaming loads), one FADD per value.
template <int THREADS, int UNROLL>
__global__ void __launch_bounds__(THREADS) read_sum_kernel(StreamPtrs sp, int64_t n, float* out) {
  const float4* s[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) s[k] = static_cast<const float4*>(sp.p[k]);
  const int64_t ngroups = n / 4, stride = int64_t(gridDim.x) * THREADS;
  float acc = 0.f;
  int64_t g = int64_t(blockIdx.x) * THREADS + threadIdx.x;
  for (; g + (UNROLL - 1) * stride < ngroups; g += UNROLL * stride) {
    float4 v[UNROLL][6];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u)
#pragma unroll
      for (int k = 0; k < 6; ++k) v[u][k] = ld_stream(s[k] + g + u * stride);
#pragma unroll
    for (int u = 0; u < UNROLL; ++u)
#pragma unroll
      for (int k = 0; k < 6; ++k) acc += (v[u][k].x + v[u][k].y) + (v[u][k].z + v[u][k].w);
  }
  for (; g < ngroups; g += stride)
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const float4 v = ld_stream(s[k] + g);
      acc += (v.x + v.y) + (v.z + v.w);
    }
  for (int o = 16; o >= 1; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

struct Env {
  PassArgs a;
  int num_sms;
  cudaStream_t stream;
  cudaEvent_t e0, e1;
  float* d_out;
};

template <class F>
float time_launch(Env& E, F launch, int reps = 15) {
  for (int i = 0; i < 3; ++i) launch();
  CK(cudaStreamSynchronize(E.stream));
  std::vector<float> ms;
  for (int i = 0; i < reps; ++i) {
    CK(cudaEventRecord(E.e0, E.stream));
    launch();
    CK(cudaEventRecord(E.e1, E.stream));
    CK(cudaEventSynchronize(E.e1));
    float t;
    CK(cudaEventElapsedTime(&t, E.e0, E.e1));
    ms.push_back(t);
  }
  std::sort(ms.begin(), ms.end());
  return ms[ms.size() / 2];
}

// Sustained rate: `warm` untimed launches, then `reps` back-to-back launches between one pair of events (what a
// long-running job sees under the power cap), in ms per launch.
static int g_sustained_reps = 0;
template <class F>
float time_sustained(Env& E, F launch) {
  if (g_sustained_reps <= 0) return 0.f;
  for (int i = 0; i < g_sustained_reps / 4; ++i) launch();
  CK(cudaEventRecord(E.e0, E.stream));
  for (int i = 0; i < g_sustained_reps; ++i) launch();
  CK(cudaEventRecord(E.e1, E.stream));
  CK(cudaEventSynchronize(E.e1));
  float t;
  CK(cudaEventElapsedTime(&t, E.e0, E.e1));
  return t / g_sustained_reps;
}

template <int THREADS, int MINB, int UNROLL, int FLUSH, int LOSS = MOPT_LOSS_HUBER>
void run_variant(Env& E, int ctas_per_sm, int mode = PASS_LINEARIZE) {
  auto kern = p2p_moment_kernel<float, float, LOSS, true, THREADS, MINB, UNROLL, FLUSH>;
  int occ = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, THREADS, 0));
  cudaFuncAttributes fa;
  CK(cudaFuncGetAttributes(&fa, kern));
  const int per_sm = std::min(occ, ctas_per_sm);
  if (per_sm < ctas_per_sm) return;  // shape not reachable
  const int grid = per_sm * E.num_sms;
  PassArgs a = E.a;
  a.mode_override = mode;
  if (mode != PASS_LINEARIZE || LOSS != MOPT_LOSS_HUBER) std::printf("[mode=%d loss=%d] ", mode, LOSS);
  const float ms = time_launch(E, [&] { kern<<<grid, THREADS, 0, E.stream>>>(a); });
  const float sus = time_sustained(E, [&] { kern<<<grid, THREADS, 0, E.stream>>>(a); });
  const double gbs = 24.0 * double(a.n) / (ms * 1e-3) / 1e9;
  std::printf("moment threads=%3d minb=%d unroll=%d flush=%2d ctas/sm=%d regs=%3d occ=%d  %8.1f us  %7.1f GB/s  %6.1f Gres/s",
              THREADS, MINB, UNROLL, FLUSH, per_sm, fa.numRegs, occ, ms * 1e3, gbs, gbs / 24.0);
  if (sus > 0.f) std::printf("   sustained %8.1f us %6.1f Gres/s", sus * 1e3, double(a.n) / (sus * 1e-3) / 1e9);
  std::printf("\n");
  std::fflush(stdout);
}


// second-generation kernel (mopt_pass_p2p2.cuh): packed fp32 + TMA bulk-copy ring
template <int THREADS, int MINB, int STAGES, int U, int FLUSH, int LOSS = MOPT_LOSS_HUBER, bool FUSED = false>
void run_variant2(Env& E, int ctas_per_sm, int mode = PASS_LINEARIZE) {
  auto kern = p2p_moment2_kernel<LOSS, true, false, FUSED, THREADS, MINB, STAGES, U, FLUSH>;
  const size_t smem = p2p2_ring_bytes(THREADS, STAGES, U);
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  int occ = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, THREADS, smem));
  cudaFuncAttributes fa;
  CK(cudaFuncGetAttributes(&fa, kern));
  const int per_sm = std::min(occ, ctas_per_sm);
  if (per_sm < ctas_per_sm) {
    std::printf("moment2 threads=%d stages=%d u=%d: only %d CTAs/SM reachable (regs=%d smem=%zu), skipped\n", THREADS, STAGES, U, occ, fa.numRegs, smem);
    return;
  }
  const int grid = per_sm * E.num_sms;
  PassArgs a = E.a;
  a.mode_override = mode;
  if (mode != PASS_LINEARIZE || LOSS != MOPT_LOSS_HUBER) std::printf("[mode=%d loss=%d] ", mode, LOSS);
  const float ms = time_launch(E, [&] { kern<<<grid, THREADS, smem, E.stream>>>(a); });
  const float sus = time_sustained(E, [&] { kern<<<grid, THREADS, smem, E.stream>>>(a); });
  const double gbs = 24.0 * double(a.n) / (ms * 1e-3) / 1e9;
  std::printf("moment2 threads=%4d minb=%d stages=%d u=%d flush=%2d ctas/sm=%d regs=%3d smem=%6zu  %8.1f us  %7.1f GB/s  %6.1f Gres/s",
              THREADS, MINB, STAGES, U, FLUSH, per_sm, fa.numRegs, smem, ms * 1e3, gbs, gbs / 24.0);
  if (sus > 0.f) std::printf("   sustained %8.1f us %6.1f Gres/s", sus * 1e3, double(a.n) / (sus * 1e-3) / 1e9);
  std::printf("\n");
  std::fflush(stdout);
}

// result of the last launch: the packed (H, b, sum) — to compare kernel generations on the same data
void print_result(Env& E, const char* tag) {
  PassResult h;
  CK(cudaMemcpy(&h, E.a.out, sizeof(h), cudaMemcpyDeviceToHost));
  std::printf("%s: H00=%.9e H05=%.9e H55=%.9e b0=%.9e b5=%.9e sum=%.9e\n", tag, h.v[0], h.v[5], h.v[20], h.v[21], h.v[26], h.v[27]);
}

// fp64-compute variants (the reference's default Scalar is double): ST = float or double streams
template <typename ST, int THREADS, int MINB, int UNROLL, int FLUSH>
void run_variant64(Env& E, const PassArgs& a64, int ctas_per_sm) {
  auto kern = p2p_moment_kernel<ST, double, MOPT_LOSS_HUBER, true, THREADS, MINB, UNROLL, FLUSH>;
  int occ = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, THREADS, 0));
  cudaFuncAttributes fa;
  CK(cudaFuncGetAttributes(&fa, kern));
  const int per_sm = std::min(occ, ctas_per_sm);
  if (per_sm < ctas_per_sm) {
    std::printf("moment64 store=%s threads=%3d minb=%d unroll=%d: only %d CTAs/SM reachable (regs=%d), skipped\n",
                sizeof(ST) == 4 ? "f32" : "f64", THREADS, MINB, UNROLL, occ, fa.numRegs);
    return;
  }
  const int grid = per_sm * E.num_sms;
  PassArgs a = a64;
  a.mode_override = PASS_LINEARIZE;
  const float ms = time_launch(E, [&] { kern<<<grid, THREADS, 0, E.stream>>>(a); });
  const double bytes = 6.0 * sizeof(ST) * double(a.n);
  std::printf("moment64 store=%s threads=%3d minb=%d unroll=%d ctas/sm=%d regs=%3d local=%zu occ=%d  %8.1f us  %7.1f GB/s  %6.1f Gres/s\n",
              sizeof(ST) == 4 ? "f32" : "f64", THREADS, MINB, UNROLL, per_sm, fa.numRegs, (size_t)fa.localSizeBytes, occ, ms * 1e3,
              bytes / (ms * 1e-3) / 1e9, double(a.n) / (ms * 1e-3) / 1e9);
  std::fflush(stdout);
}

__global__ void widen_kernel(const float* in, double* out, int64_t n) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) out[i] = double(in[i]);
}

template <int THREADS, int UNROLL>
void run_ceiling(Env& E, int ctas_per_sm) {
  auto kern = read_sum_kernel<THREADS, UNROLL>;
  int occ = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, THREADS, 0));
  const int per_sm = std::min(occ, ctas_per_sm);
  const int grid = per_sm * E.num_sms;
  const float ms = time_launch(E, [&] { kern<<<grid, THREADS, 0, E.stream>>>(E.a.streams, E.a.n, E.d_out); });
  const float sus = time_sustained(E, [&] { kern<<<grid, THREADS, 0, E.stream>>>(E.a.streams, E.a.n, E.d_out); });
  const double gbs = 24.0 * double(E.a.n) / (ms * 1e-3) / 1e9;
  std::printf("ceiling threads=%3d unroll=%d ctas/sm=%d occ=%d  %8.1f us  %7.1f GB/s", THREADS, UNROLL, per_sm, occ, ms * 1e3, gbs);
  if (sus > 0.f) std::printf("   sustained %8.1f us %7.1f GB/s", sus * 1e3, 24.0 * double(E.a.n) / (sus * 1e-3) / 1e9);
  std::printf("\n");
  std::fflush(stdout);
}

int main(int argc, char** argv) {
  const int64_t n = argc > 1 ? std::atoll(argv[1]) : 100000000LL;
  Env E;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, 0));
  E.num_sms = prop.multiProcessorCount;
  CK(cudaStreamCreate(&E.stream));
  CK(cudaEventCreate(&E.e0));
  CK(cudaEventCreate(&E.e1));
  std::memset(&E.a, 0, sizeof(E.a));
  for (int k = 0; k < 6; ++k) {
    float* p;
    CK(cudaMalloc(&p, size_t(n) * 4 + 512));
    fill_kernel<<<148 * 8, 256, 0, E.stream>>>(p, n, 17u * (k + 1));
    E.a.streams.p[k] = p;
  }
  ParamBlock hpb;
  std::memset(&hpb, 0, sizeof(hpb));
  const double R[12] = {0.99, -0.08, 0.05, 0.08, 0.99, -0.1, -0.05, 0.1, 0.99, 0.5, -0.3, 0.2};
  for (int i = 0; i < 12; ++i) hpb.sets[0][i] = R[i];
  for (int r = 0; r < 3; ++r) hpb.jaff[0][r * 6 + r] = 1.0;
  CostDev hc;
  std::memset(&hc, 0, sizeof(hc));
  hc.model = MOPT_MODEL_POINT2POINT; hc.P = 6; hc.O = 3; hc.loss = MOPT_LOSS_HUBER; hc.loss_param = 0.05;
  ParamBlock* dpb; CostDev* dc; double* dpart; unsigned* dtick; PassResult* dout;
  CK(cudaMalloc(&dpb, sizeof(hpb))); CK(cudaMemcpy(dpb, &hpb, sizeof(hpb), cudaMemcpyHostToDevice));
  CK(cudaMalloc(&dc, sizeof(hc))); CK(cudaMemcpy(dc, &hc, sizeof(hc), cudaMemcpyHostToDevice));
  CK(cudaMalloc(&dpart, sizeof(double) * 32 * kMaxGrid));
  CK(cudaMalloc(&dtick, 4)); CK(cudaMemset(dtick, 0, 4));
  CK(cudaMalloc(&dout, sizeof(PassResult)));
  CK(cudaMalloc(&E.d_out, 4)); CK(cudaMemset(E.d_out, 0, 4));
  E.a.n = n; E.a.pb = dpb; E.a.cost = dc; E.a.partials = dpart; E.a.ticket = dtick; E.a.out = dout;
  E.a.accumulate = 0; E.a.mode_ptr = nullptr; E.a.mode_override = PASS_LINEARIZE;
  if (argc > 2 && std::string(argv[2]) == "realistic")
    make_targets_kernel<<<148 * 8, 256, 0, E.stream>>>((const float*)E.a.streams.p[0], (const float*)E.a.streams.p[1],
                                                       (const float*)E.a.streams.p[2], (float*)E.a.streams.p[3],
                                                       (float*)E.a.streams.p[4], (float*)E.a.streams.p[5], n);
  CK(cudaStreamSynchronize(E.stream));
  std::printf("%s, %d SMs, n = %lld, data = %s\n", prop.name, E.num_sms, (long long)n, argc > 2 ? argv[2] : "random");

  if (argc > 2 && std::string(argv[2]) == "gen2ncu") {  // a few launches of the candidates, for an ncu capture
    make_targets_kernel<<<148 * 8, 256, 0, E.stream>>>((const float*)E.a.streams.p[0], (const float*)E.a.streams.p[1],
                                                       (const float*)E.a.streams.p[2], (float*)E.a.streams.p[3],
                                                       (float*)E.a.streams.p[4], (float*)E.a.streams.p[5], n);
    CK(cudaStreamSynchronize(E.stream));
    PassArgs a = E.a;
    auto k1 = p2p_moment_kernel<float, float, MOPT_LOSS_HUBER, true, 1024, 1, 1, 16>;
    auto k2 = p2p_moment2_kernel<MOPT_LOSS_HUBER, true, false, false, 512, 1, 2, 2, 16>;
    auto k3 = p2p_moment2_kernel<MOPT_LOSS_HUBER, true, false, false, 384, 1, 2, 2, 16>;
    auto k4 = p2p_moment2_kernel<MOPT_LOSS_HUBER, true, false, false, 512, 1, 4, 1, 32>;
    const size_t s2 = p2p2_ring_bytes(512, 2, 2), s3 = p2p2_ring_bytes(384, 2, 2), s4 = p2p2_ring_bytes(512, 4, 1);
    CK(cudaFuncSetAttribute(k2, cudaFuncAttributeMaxDynamicSharedMemorySize, int(s2)));
    CK(cudaFuncSetAttribute(k3, cudaFuncAttributeMaxDynamicSharedMemorySize, int(s3)));
    CK(cudaFuncSetAttribute(k4, cudaFuncAttributeMaxDynamicSharedMemorySize, int(s4)));
    for (int i = 0; i < 2; ++i) {
      k1<<<148, 1024, 0, E.stream>>>(a);
      k2<<<148, 512, s2, E.stream>>>(a);
      k3<<<148, 384, s3, E.stream>>>(a);
      k4<<<148, 512, s4, E.stream>>>(a);
    }
    CK(cudaStreamSynchronize(E.stream));
    std::printf("gen2ncu done\n");
    return 0;
  }
  if (argc > 2 && std::string(argv[2]) == "gen2") {  // packed-fp32 / TMA-ring kernel against the shipped one, realistic data
    make_targets_kernel<<<148 * 8, 256, 0, E.stream>>>((const float*)E.a.streams.p[0], (const float*)E.a.streams.p[1],
                                                       (const float*)E.a.streams.p[2], (float*)E.a.streams.p[3],
                                                       (float*)E.a.streams.p[4], (float*)E.a.streams.p[5], n);
    CK(cudaStreamSynchronize(E.stream));
    const int prewarm = argc > 3 ? std::atoi(argv[3]) : 0;
    {
      auto kern = p2p_moment_kernel<float, float, MOPT_LOSS_HUBER, true, 1024, 1, 1, 16>;
      PassArgs a = E.a;
      for (int i = 0; i < prewarm; ++i) kern<<<148, 1024, 0, E.stream>>>(a);
      CK(cudaStreamSynchronize(E.stream));
    }
    g_sustained_reps = argc > 4 ? std::atoi(argv[4]) : 0;
    for (int rep = 0; rep < 2; ++rep) {
      run_ceiling<256, 4>(E, 3);
      run_variant<1024, 1, 1, 16>(E, 1);  // shipped in round 1
      if (rep == 0) print_result(E, "gen1");
      run_variant2<512, 1, 4, 1, 32>(E, 1);
      if (rep == 0) print_result(E, "gen2");
      run_variant2<512, 1, 3, 1, 32>(E, 1);
      run_variant2<512, 1, 2, 1, 32>(E, 1);
      run_variant2<512, 1, 2, 2, 16>(E, 1);
      run_variant2<512, 1, 2, 2, 8>(E, 1);
      run_variant2<384, 1, 3, 1, 32>(E, 1);
      run_variant2<384, 1, 4, 1, 32>(E, 1);
      run_variant2<384, 1, 2, 2, 16>(E, 1);
      run_variant2<384, 1, 3, 2, 16>(E, 1);
      run_variant2<384, 1, 2, 3, 8>(E, 1);
      run_variant2<448, 1, 2, 2, 16>(E, 1);
      run_variant2<320, 1, 2, 2, 16>(E, 1);
      run_variant2<320, 1, 3, 2, 16>(E, 1);
      run_variant2<256, 1, 2, 4, 8>(E, 1);
      run_variant2<256, 2, 2, 1, 32>(E, 2);
      run_variant2<256, 2, 2, 2, 16>(E, 2);
      run_variant2<192, 2, 2, 2, 16>(E, 2);
      run_variant2<512, 1, 2, 2, 16>(E, 1, PASS_COST);
      run_variant2<384, 1, 2, 2, 16>(E, 1, PASS_COST);
      run_variant2<512, 1, 2, 2, 16, MOPT_LOSS_NONE>(E, 1);
    }
    return 0;
  }
  if (argc > 2 && std::string(argv[2]) == "f64") {  // fp64-compute launch shapes
    make_targets_kernel<<<148 * 8, 256, 0, E.stream>>>((const float*)E.a.streams.p[0], (const float*)E.a.streams.p[1],
                                                       (const float*)E.a.streams.p[2], (float*)E.a.streams.p[3],
                                                       (float*)E.a.streams.p[4], (float*)E.a.streams.p[5], n);
    CK(cudaStreamSynchronize(E.stream));
    PassArgs af = E.a;
    for (int rep = 0; rep < 2; ++rep) {
      run_variant64<float, 256, 1, 2, 8>(E, af, 1);  // shipped
      run_variant64<float, 256, 1, 1, 8>(E, af, 1);
      run_variant64<float, 256, 2, 1, 8>(E, af, 2);
      run_variant64<float, 256, 2, 2, 8>(E, af, 2);
      run_variant64<float, 512, 1, 1, 8>(E, af, 1);
      run_variant64<float, 128, 4, 1, 8>(E, af, 4);
      run_variant64<float, 256, 3, 1, 8>(E, af, 3);
      run_variant64<float, 1024, 1, 1, 8>(E, af, 1);
    }
    // fp64 store: half as many elements so the six double streams fit next to the float ones
    PassArgs ad = E.a;
    ad.n = n / 2;
    for (int k = 0; k < 6; ++k) {
      double* p;
      CK(cudaMalloc(&p, size_t(ad.n) * 8 + 512));
      widen_kernel<<<148 * 8, 256, 0, E.stream>>>((const float*)E.a.streams.p[k], p, ad.n);
      ad.streams.p[k] = p;
    }
    CK(cudaStreamSynchronize(E.stream));
    for (int rep = 0; rep < 2; ++rep) {
      run_variant64<double, 256, 1, 2, 8>(E, ad, 1);  // shipped
      run_variant64<double, 256, 1, 1, 8>(E, ad, 1);
      run_variant64<double, 256, 2, 1, 8>(E, ad, 2);
      run_variant64<double, 256, 2, 2, 8>(E, ad, 2);
      run_variant64<double, 512, 1, 1, 8>(E, ad, 1);
      run_variant64<double, 128, 4, 1, 8>(E, ad, 4);
      run_variant64<double, 256, 3, 1, 8>(E, ad, 3);
    }
    return 0;
  }
  if (argc > 3) {  // sustained-clock experiment: long pre-warm, then the variants that separate ALU from HBM limits
    auto kern = p2p_moment_kernel<float, float, MOPT_LOSS_HUBER, true, 1024, 1, 1, 16>;
    PassArgs a = E.a;
    for (int i = 0; i < std::atoi(argv[3]); ++i) kern<<<148, 1024, 0, E.stream>>>(a);
    CK(cudaStreamSynchronize(E.stream));
    for (int rep = 0; rep < 3; ++rep) {
      run_ceiling<256, 4>(E, 3);
      run_variant<1024, 1, 1, 16>(E, 1);
      run_variant<1024, 1, 1, 16, MOPT_LOSS_NONE>(E, 1);
      run_variant<1024, 1, 1, 16>(E, 1, PASS_COST);
      run_variant<256, 2, 2, 16>(E, 2);
      run_variant<256, 2, 2, 16>(E, 2, PASS_COST);
    }
    return 0;
  }
  run_ceiling<256, 1>(E, 8); run_ceiling<256, 2>(E, 8); run_ceiling<256, 4>(E, 8);
  run_ceiling<256, 2>(E, 4); run_ceiling<256, 4>(E, 4); run_ceiling<256, 4>(E, 2);
  run_ceiling<512, 2>(E, 4); run_ceiling<512, 4>(E, 2); run_ceiling<1024, 2>(E, 2);

  run_variant<256, 2, 2, 8>(E, 2);   // shipped shape
  run_variant<256, 2, 2, 16>(E, 2);
  run_variant<1024, 1, 1, 16>(E, 1);
  return 0;
}
