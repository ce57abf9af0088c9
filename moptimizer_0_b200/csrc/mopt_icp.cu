// Correspondence re-association — `model->update(x)` (SURVEY.md §8f-1).
// The reference calls cost->update(x0) -> model->update(x) before every linearization
// (src/levenberg_marquadt_dyn.cpp:54, include/moptimizer/model.h:24-26 "i.e registration correspondences",
// docs/Cost.puml:14-17 "nearest neighboor search on data") but ships no implementation: every test model
// leaves it empty.  This is the device implementation for point2point: the fixed target cloud lives in a
// uniform grid (cell edge >= the maximum correspondence distance, points counting-sorted by cell; no Thrust),
// and one kernel transforms every source point with T(x), finds its nearest target point in the 27
// surrounding cells and rewrites the store's target streams in place.  Source points with no target within
// the distance get a NaN marker and are skipped by every later pass, which is what `f` returning false
// means in the reference (linearization.h:102,144).
//
// Contract (the brute-force oracle::Point2PointICP restated): ties go to the lowest original index, the radius is
// inclusive (|q - p|^2 <= max_dist^2, in the index dtype), the fp32 index forms the query and the distances in fp32
// from fp32-rounded data and writes fp32-rounded target coordinates, and a target point with a non-finite
// coordinate never matches: it is kept in the index, in one extra cell behind the grid that no query scans.
#include <cmath>
#include <cstring>
#include <vector>

#include "mopt_internal.h"

using namespace mopt;

struct mopt_nn_index {
  mopt_ctx* ctx = nullptr;
  int dtype = MOPT_F64;
  int64_t m = 0;
  double max_dist = 0.0, cell = 0.0;
  double origin[3] = {0, 0, 0};
  int dims[3] = {1, 1, 1};
  int64_t ncells = 1;
  void* d_pts = nullptr;        // sorted by cell: x[m], y[m], z[m] (planar, index dtype)
  int* d_orig = nullptr;        // original index of each sorted point (tie-break => deterministic matches)
  unsigned int* d_start = nullptr;  // [ncells + 2] exclusive prefix of the per-cell counts; cell ncells holds the
                                    // non-finite points
  long long* d_matched = nullptr;
};

namespace {

struct GridDesc {
  double origin[3];
  double inv_cell;
  int dims[3];
};

// Cell of a coordinate along one axis, -1 / dim outside the grid; NaN gives -1 (never int(NaN)).
template <typename T>
__device__ __forceinline__ int cell_coord(T v, double origin, double inv_cell, int dim) {
  const double c = floor((double(v) - origin) * inv_cell);
  return c >= 0.0 ? (c < double(dim) ? int(c) : dim) : -1;
}

template <typename T>
__device__ __forceinline__ bool finite3(const T* p) {
  return isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]);
}

template <typename T>
__global__ void bbox_kernel(const T* __restrict__ aos, int64_t m, double* __restrict__ partial /*[grid][6]*/) {
  // the box of the points whose three coordinates are finite (lo > hi when there is none)
  double lo[3] = {HUGE_VAL, HUGE_VAL, HUGE_VAL}, hi[3] = {-HUGE_VAL, -HUGE_VAL, -HUGE_VAL};
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < m; i += int64_t(gridDim.x) * blockDim.x) {
    if (!finite3(aos + i * 3)) continue;
    for (int k = 0; k < 3; ++k) {
      const double v = double(aos[i * 3 + k]);
      lo[k] = fmin(lo[k], v);
      hi[k] = fmax(hi[k], v);
    }
  }
  __shared__ double s[6][256];
  for (int k = 0; k < 3; ++k) { s[k][threadIdx.x] = lo[k]; s[3 + k][threadIdx.x] = hi[k]; }
  __syncthreads();
  for (int off = blockDim.x / 2; off > 0; off >>= 1) {
    if (int(threadIdx.x) < off)
      for (int k = 0; k < 3; ++k) {
        s[k][threadIdx.x] = fmin(s[k][threadIdx.x], s[k][threadIdx.x + off]);
        s[3 + k][threadIdx.x] = fmax(s[3 + k][threadIdx.x], s[3 + k][threadIdx.x + off]);
      }
    __syncthreads();
  }
  if (threadIdx.x == 0)
    for (int k = 0; k < 6; ++k) partial[blockIdx.x * 6 + k] = s[k][0];
}

// Cell of each target point: the clamped grid cell, or `ncells` (behind the grid, never scanned) for a point with a
// non-finite coordinate.
template <typename T>
__global__ void count_kernel(const T* __restrict__ aos, int64_t m, GridDesc g, unsigned int ncells,
                             unsigned int* __restrict__ counts, unsigned int* __restrict__ cell_of) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < m; i += int64_t(gridDim.x) * blockDim.x) {
    int c[3];
    for (int k = 0; k < 3; ++k) {
      c[k] = cell_coord(aos[i * 3 + k], g.origin[k], g.inv_cell, g.dims[k]);
      c[k] = c[k] < 0 ? 0 : (c[k] >= g.dims[k] ? g.dims[k] - 1 : c[k]);
    }
    const unsigned int cell = finite3(aos + i * 3)
                                  ? (unsigned(c[2]) * g.dims[1] + unsigned(c[1])) * g.dims[0] + unsigned(c[0])
                                  : ncells;
    cell_of[i] = cell;
    atomicAdd(&counts[cell], 1u);
  }
}

// Three-kernel exclusive scan of `n` unsigned counters (in place), 2048 items per block.
constexpr int kScanThreads = 256, kScanItems = 8, kScanTile = kScanThreads * kScanItems;

__global__ void scan_tiles_kernel(unsigned int* __restrict__ data, int64_t n, unsigned int* __restrict__ tile_sums) {
  __shared__ unsigned int s[kScanThreads];
  const int64_t base = int64_t(blockIdx.x) * kScanTile + int64_t(threadIdx.x) * kScanItems;
  unsigned int v[kScanItems], sum = 0;
  for (int k = 0; k < kScanItems; ++k) {
    v[k] = (base + k < n) ? data[base + k] : 0u;
    sum += v[k];
  }
  s[threadIdx.x] = sum;
  __syncthreads();
  for (int off = 1; off < kScanThreads; off <<= 1) {  // Hillis-Steele inclusive scan of the thread sums
    const unsigned int t = (int(threadIdx.x) >= off) ? s[threadIdx.x - off] : 0u;
    __syncthreads();
    s[threadIdx.x] += t;
    __syncthreads();
  }
  unsigned int run = s[threadIdx.x] - sum;  // exclusive prefix of this thread within the tile
  for (int k = 0; k < kScanItems; ++k) {
    if (base + k < n) data[base + k] = run;
    run += v[k];
  }
  if (threadIdx.x == kScanThreads - 1) tile_sums[blockIdx.x] = s[threadIdx.x];
}

__global__ void scan_sums_kernel(unsigned int* __restrict__ tile_sums, int ntiles) {  // one thread: ntiles <= 8193
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    unsigned int run = 0;
    for (int i = 0; i < ntiles; ++i) {
      const unsigned int t = tile_sums[i];
      tile_sums[i] = run;
      run += t;
    }
  }
}

__global__ void scan_add_kernel(unsigned int* __restrict__ data, int64_t n, const unsigned int* __restrict__ tile_sums) {
  const int64_t base = int64_t(blockIdx.x) * kScanTile;
  const unsigned int add = tile_sums[blockIdx.x];
  for (int k = threadIdx.x; k < kScanTile; k += kScanThreads)
    if (base + k < n) data[base + k] += add;
}

template <typename T>
__global__ void scatter_kernel(const T* __restrict__ aos, int64_t m, const unsigned int* __restrict__ cell_of,
                               const unsigned int* __restrict__ start, unsigned int* __restrict__ cursor,
                               T* __restrict__ px, T* __restrict__ py, T* __restrict__ pz, int* __restrict__ orig) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < m; i += int64_t(gridDim.x) * blockDim.x) {
    const unsigned int cell = cell_of[i];
    const unsigned int pos = start[cell] + atomicAdd(&cursor[cell], 1u);
    px[pos] = aos[i * 3 + 0];
    py[pos] = aos[i * 3 + 1];
    pz[pos] = aos[i * 3 + 2];
    orig[pos] = int(i);
  }
}

// model->update(x): tgt_i <- nearest target of T(x) src_i, or the NaN "no correspondence" marker.
// `gate` (may be null) points at {pass_mode, phase, done}-style control words of the device LM: the kernel is
// enqueued in every LM slot and runs only at the start of an outer iteration (levenberg_marquadt_dyn.cpp:54).
template <typename ST, typename T>
__global__ void reassociate_kernel(const ST* __restrict__ sx, const ST* __restrict__ sy, const ST* __restrict__ sz,
                                   ST* __restrict__ tx, ST* __restrict__ ty, ST* __restrict__ tz, int64_t n,
                                   const ParamBlock* __restrict__ pb, GridDesc g, double max_dist,
                                   const T* __restrict__ px, const T* __restrict__ py, const T* __restrict__ pz,
                                   const int* __restrict__ orig, const unsigned int* __restrict__ start,
                                   long long* __restrict__ matched, const LmState* __restrict__ gate) {
  if (gate && (gate->done || gate->phase != LM_PHASE_LIN)) return;
  T R[9], t[3];
  for (int i = 0; i < 9; ++i) R[i] = T(pb->sets[0][i]);
  for (int i = 0; i < 3; ++i) t[i] = T(pb->sets[0][9 + i]);
  const T r2max = T(max_dist * max_dist);
  long long local = 0;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const T p0 = T(sx[i]), p1 = T(sy[i]), p2 = T(sz[i]);
    const T q[3] = {R[0] * p0 + R[1] * p1 + R[2] * p2 + t[0], R[3] * p0 + R[4] * p1 + R[5] * p2 + t[1],
                    R[6] * p0 + R[7] * p1 + R[8] * p2 + t[2]};
    int c[3];
    for (int k = 0; k < 3; ++k) c[k] = cell_coord(q[k], g.origin[k], g.inv_cell, g.dims[k]);
    T best = r2max;
    int best_orig = 0x7fffffff;
    unsigned int best_pos = 0xffffffffu;
    for (int dz = -1; dz <= 1; ++dz) {
      const int cz = c[2] + dz;
      if (cz < 0 || cz >= g.dims[2]) continue;
      for (int dy = -1; dy <= 1; ++dy) {
        const int cy = c[1] + dy;
        if (cy < 0 || cy >= g.dims[1]) continue;
        // the three x-neighbours are contiguous cells: one range
        int x0 = c[0] - 1, x1 = c[0] + 1;
        if (x0 < 0) x0 = 0;
        if (x1 >= g.dims[0]) x1 = g.dims[0] - 1;
        if (x0 > x1) continue;
        const unsigned int row = (unsigned(cz) * g.dims[1] + unsigned(cy)) * g.dims[0];
        const unsigned int b = start[row + x0], e = start[row + x1 + 1];
        for (unsigned int j = b; j < e; ++j) {
          const T d0 = px[j] - q[0], d1 = py[j] - q[1], d2 = pz[j] - q[2];
          const T dd = d0 * d0 + d1 * d1 + d2 * d2;
          const int o = orig[j];
          if (dd < best || (dd == best && dd <= r2max && o < best_orig)) {
            best = dd;
            best_orig = o;
            best_pos = j;
          }
        }
      }
    }
    if (best_pos != 0xffffffffu) {
      tx[i] = ST(px[best_pos]);
      ty[i] = ST(py[best_pos]);
      tz[i] = ST(pz[best_pos]);
      ++local;
    } else {
      const ST no_match = ST(__longlong_as_double(0x7ff8000000000000LL));  // quiet NaN marker
      tx[i] = no_match;
      ty[i] = no_match;
      tz[i] = no_match;
    }
  }
  // warp-aggregated count of matches
  for (int off = 16; off >= 1; off >>= 1) local += __shfl_xor_sync(0xffffffffu, local, off);
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(reinterpret_cast<unsigned long long*>(matched), (unsigned long long)local);
}

template <typename T>
int build_index(mopt_nn_index* ix, const void* host, int host_dtype) {
  mopt_ctx* ctx = ix->ctx;
  const int64_t m = ix->m;
  const size_t esz = sizeof(T);
  T* d_aos = nullptr;
  MOPT_CUDA_TRY(cudaMalloc(&d_aos, esz * 3 * size_t(m > 0 ? m : 1)));
  // host array -> device AoS of the index dtype
  if ((host_dtype == MOPT_F32) == (sizeof(T) == 4)) {
    MOPT_CUDA_TRY(cudaMemcpyAsync(d_aos, host, esz * 3 * size_t(m), cudaMemcpyHostToDevice, ctx->stream));
  } else {
    std::vector<T> tmp(size_t(m) * 3);
    if (host_dtype == MOPT_F32) { const float* h = static_cast<const float*>(host); for (size_t i = 0; i < tmp.size(); ++i) tmp[i] = T(h[i]); }
    else { const double* h = static_cast<const double*>(host); for (size_t i = 0; i < tmp.size(); ++i) tmp[i] = T(h[i]); }
    MOPT_CUDA_TRY(cudaMemcpyAsync(d_aos, tmp.data(), esz * 3 * size_t(m), cudaMemcpyHostToDevice, ctx->stream));
    MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  }
  // bounding box
  const int bb_blocks = 296;
  double* d_part = nullptr;
  MOPT_CUDA_TRY(cudaMalloc(&d_part, sizeof(double) * 6 * bb_blocks));
  bbox_kernel<T><<<bb_blocks, 256, 0, ctx->stream>>>(d_aos, m, d_part);
  MOPT_CUDA_TRY(cudaGetLastError());
  std::vector<double> part(6 * bb_blocks);
  MOPT_CUDA_TRY(cudaMemcpyAsync(part.data(), d_part, sizeof(double) * part.size(), cudaMemcpyDeviceToHost, ctx->stream));
  MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  cudaFree(d_part);
  double lo[3] = {HUGE_VAL, HUGE_VAL, HUGE_VAL}, hi[3] = {-HUGE_VAL, -HUGE_VAL, -HUGE_VAL};
  for (int b = 0; b < bb_blocks; ++b)
    for (int k = 0; k < 3; ++k) {
      lo[k] = std::fmin(lo[k], part[b * 6 + k]);
      hi[k] = std::fmax(hi[k], part[b * 6 + 3 + k]);
    }
  if (!(lo[0] <= hi[0])) for (int k = 0; k < 3; ++k) lo[k] = hi[k] = 0.0;  // no finite point (or m == 0)
  // An axis whose points span more than DBL_MAX (e.g. -1e308 and 1e308): hi - lo is inf, and the axis becomes one
  // slab that every query scans whole.
  double ext[3];
  for (int k = 0; k < 3; ++k) ext[k] = hi[k] - lo[k];
  // cell edge: the search radius, grown until the grid has at most 2^24 cells.  The extents are finite (or one slab)
  // and the radius is finite: a radius of at least every extent fits on the first pass, and otherwise the edge grows
  // until it exceeds every extent / 255 (< DBL_MAX / 200), so the loop ends.
  double cell = ix->max_dist;
  for (;;) {
    double dims[3], total = 1.0;  // in double until the total is known to be small: a tiny radius over a wide
    for (int k = 0; k < 3; ++k) {  // cloud gives per-axis counts far beyond INT_MAX
      dims[k] = std::isfinite(ext[k]) ? std::floor(ext[k] / cell) + 1.0 : 1.0;
      total *= dims[k];
    }
    if (total <= double(1 << 24)) {
      for (int k = 0; k < 3; ++k) ix->dims[k] = int(dims[k]);
      break;
    }
    cell *= 1.26;
  }
  ix->cell = cell;
  ix->ncells = int64_t(ix->dims[0]) * ix->dims[1] * ix->dims[2];
  for (int k = 0; k < 3; ++k) ix->origin[k] = lo[k];
  GridDesc g;
  for (int k = 0; k < 3; ++k) { g.origin[k] = ix->origin[k]; g.dims[k] = ix->dims[k]; }
  g.inv_cell = 1.0 / cell;

  unsigned int *d_cell_of = nullptr, *d_cursor = nullptr, *d_tiles = nullptr;
  const int64_t nstart = ix->ncells + 2;  // the grid's cells, the cell of the non-finite points, the end
  const int ntiles = int((nstart + kScanTile - 1) / kScanTile);
  MOPT_CUDA_TRY(cudaMalloc(&ix->d_start, sizeof(unsigned int) * size_t(nstart)));
  MOPT_CUDA_TRY(cudaMalloc(&d_cursor, sizeof(unsigned int) * size_t(ix->ncells + 1)));
  MOPT_CUDA_TRY(cudaMalloc(&d_cell_of, sizeof(unsigned int) * size_t(m > 0 ? m : 1)));
  MOPT_CUDA_TRY(cudaMalloc(&d_tiles, sizeof(unsigned int) * size_t(ntiles)));
  MOPT_CUDA_TRY(cudaMemsetAsync(ix->d_start, 0, sizeof(unsigned int) * size_t(nstart), ctx->stream));
  MOPT_CUDA_TRY(cudaMemsetAsync(d_cursor, 0, sizeof(unsigned int) * size_t(ix->ncells + 1), ctx->stream));
  int blocks = int(std::min<int64_t>((m + 255) / 256, 148 * 16));
  if (blocks < 1) blocks = 1;
  count_kernel<T><<<blocks, 256, 0, ctx->stream>>>(d_aos, m, g, unsigned(ix->ncells), ix->d_start, d_cell_of);
  MOPT_CUDA_TRY(cudaGetLastError());
  scan_tiles_kernel<<<ntiles, kScanThreads, 0, ctx->stream>>>(ix->d_start, nstart, d_tiles);
  scan_sums_kernel<<<1, 32, 0, ctx->stream>>>(d_tiles, ntiles);
  scan_add_kernel<<<ntiles, kScanThreads, 0, ctx->stream>>>(ix->d_start, nstart, d_tiles);
  MOPT_CUDA_TRY(cudaGetLastError());
  T* pts = nullptr;
  MOPT_CUDA_TRY(cudaMalloc(&pts, esz * 3 * size_t(m > 0 ? m : 1)));
  MOPT_CUDA_TRY(cudaMalloc(&ix->d_orig, sizeof(int) * size_t(m > 0 ? m : 1)));
  ix->d_pts = pts;
  scatter_kernel<T><<<blocks, 256, 0, ctx->stream>>>(d_aos, m, d_cell_of, ix->d_start, d_cursor, pts, pts + m, pts + 2 * m,
                                                     ix->d_orig);
  MOPT_CUDA_TRY(cudaGetLastError());
  MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  cudaFree(d_aos); cudaFree(d_cell_of); cudaFree(d_cursor); cudaFree(d_tiles);
  MOPT_CUDA_TRY(cudaMalloc(&ix->d_matched, sizeof(long long)));
  return MOPT_OK;
}

template <typename ST, typename T>
void launch_reassoc(mopt_store* st, mopt_nn_index* ix, const ParamBlock* pb, const LmState* gate) {
  GridDesc g;
  for (int k = 0; k < 3; ++k) { g.origin[k] = ix->origin[k]; g.dims[k] = ix->dims[k]; }
  g.inv_cell = 1.0 / ix->cell;
  const T* pts = static_cast<const T*>(ix->d_pts);
  int blocks = int(std::min<int64_t>((st->n + 255) / 256, 148 * 32));
  if (blocks < 1) blocks = 1;
  reassociate_kernel<ST, T><<<blocks, 256, 0, st->ctx->stream>>>(
      static_cast<const ST*>(st->streams[0]), static_cast<const ST*>(st->streams[1]), static_cast<const ST*>(st->streams[2]),
      static_cast<ST*>(st->streams[3]), static_cast<ST*>(st->streams[4]), static_cast<ST*>(st->streams[5]), st->n, pb, g,
      ix->max_dist, pts, pts + ix->m, pts + 2 * ix->m, ix->d_orig, ix->d_start, ix->d_matched, gate);
}

}  // namespace

namespace mopt {

// Enqueue model->update for `st` on its context stream; `gate` != null makes it conditional on the LM state.
int enqueue_reassociate(mopt_store* st, const ParamBlock* pb, const LmState* gate) {
  mopt_nn_index* ix = st->index;
  if (!ix) return MOPT_OK;
  MOPT_CUDA_TRY(cudaMemsetAsync(ix->d_matched, 0, sizeof(long long), st->ctx->stream));
  if (st->dtype == MOPT_F32 && ix->dtype == MOPT_F32) launch_reassoc<float, float>(st, ix, pb, gate);
  else if (st->dtype == MOPT_F32 && ix->dtype == MOPT_F64) launch_reassoc<float, double>(st, ix, pb, gate);
  else if (st->dtype == MOPT_F64 && ix->dtype == MOPT_F32) launch_reassoc<double, float>(st, ix, pb, gate);
  else launch_reassoc<double, double>(st, ix, pb, gate);
  MOPT_CUDA_TRY(cudaGetLastError());
  st->may_have_invalid = true;
  return MOPT_OK;
}

}  // namespace mopt

extern "C" {

int mopt_nn_index_create(mopt_ctx* ctx, const void* host_xyz, int host_dtype, int index_dtype, int64_t m,
                         double max_distance, mopt_nn_index** out) try {
  MOPT_REQUIRE(ctx && out && (host_xyz || m == 0), "null argument");
  MOPT_REQUIRE(m >= 0 && m < (int64_t(1) << 31), "target cloud size must be below 2^31");
  MOPT_REQUIRE(max_distance > 0.0 && std::isfinite(max_distance), "max_distance must be positive");
  MOPT_REQUIRE((host_dtype == MOPT_F32 || host_dtype == MOPT_F64) && (index_dtype == MOPT_F32 || index_dtype == MOPT_F64),
               "bad dtype");
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  mopt_nn_index* ix = new mopt_nn_index();
  ix->ctx = ctx;
  ix->dtype = index_dtype;
  ix->m = m;
  ix->max_dist = max_distance;
  const int s = index_dtype == MOPT_F32 ? build_index<float>(ix, host_xyz, host_dtype) : build_index<double>(ix, host_xyz, host_dtype);
  if (s != MOPT_OK) {
    mopt_nn_index_destroy(ix);
    return s;
  }
  *out = ix;
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_nn_index_destroy(mopt_nn_index* ix) try {
  if (!ix) return MOPT_OK;
  cudaSetDevice(ix->ctx->device);
  cudaStreamSynchronize(ix->ctx->stream);
  cudaFree(ix->d_pts); cudaFree(ix->d_orig); cudaFree(ix->d_start); cudaFree(ix->d_matched);
  delete ix;
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_store_set_target(mopt_store* store, mopt_nn_index* index) try {
  MOPT_REQUIRE(store, "null store");
  MOPT_REQUIRE(store->model == MOPT_MODEL_POINT2POINT, "correspondence re-association is defined for point2point stores");
  MOPT_REQUIRE(!index || index->ctx == store->ctx, "index and store live on different contexts");
  store->index = index;
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_store_reassociate(mopt_store* store, const double* x, int64_t* matched) try {
  MOPT_REQUIRE(store && x, "null argument");
  MOPT_REQUIRE(store->index, "no target index attached (mopt_store_set_target)");
  mopt_ctx* ctx = store->ctx;
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  mopt_problem p;
  std::memset(&p, 0, sizeof(p));
  p.model = MOPT_MODEL_POINT2POINT; p.num_parameters = 6; p.num_outputs = 3; p.jacobian = MOPT_JAC_ANALYTICAL;
  p.compute_dtype = MOPT_F64;
  MOPT_TRY(mopt::setup_slot(ctx, 0, &p, x));
  MOPT_TRY(enqueue_reassociate(store, &ctx->d_slots[0].pb, nullptr));
  long long h = 0;
  MOPT_CUDA_TRY(cudaMemcpyAsync(&h, store->index->d_matched, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  if (matched) *matched = int64_t(h);
  return MOPT_OK;
}
MOPT_ABI_CATCH

}  // extern "C"
