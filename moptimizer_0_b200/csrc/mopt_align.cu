// Closed-form rigid alignment: the point2point instantiations of align_terms_kernel (mopt_align.cuh) and its launch,
// mopt_align_terms (device), mopt_align_terms_merge and mopt_align_from_terms (host only: Horn's quaternion solve).
#include <cmath>
#include <cstring>

#include "mopt_align.cuh"
#include "mopt_internal.h"

namespace mopt {

int align_kernel_desc(int store_dtype, int compute_dtype, KernelDesc* k) {
  return with_dtypes(store_dtype, compute_dtype, [&](auto st, auto ct) {
    *k = builtin_kernel(reinterpret_cast<const void*>(align_terms_kernel<P2PModel, decltype(st), decltype(ct)>),
                        kAlignThreads);
    return MOPT_OK;
  });
}

}  // namespace mopt

using namespace mopt;

namespace {

static_assert(sizeof(AlignAcc) <= sizeof(PassResult), "the terms must fit the pinned bounce buffer");

// The terms of cost slot 0 (staged by setup_slot) into ctx->d_align.  The grid follows the elements of the range by
// the rule of every streaming kernel (persistent_grid), so the order of the merges is fixed for a launch setting.
int launch_align(mopt_ctx* ctx, const mopt_store* st, const mopt_problem* p, const AlignArgs& al) {
  KernelDesc k;
  MOPT_TRY(align_kernel_desc(st->dtype, p->compute_dtype, &k));
  const int grid = persistent_grid(k.occupancy, k.threads, pass_launch(ctx, p), al.count / store_vec(st->dtype) + 1);
  PassArgs a = make_args(ctx, st, 0, 0, PASS_COST);
  AlignArgs aa = al;
  void* params[] = {&a, &aa};
  MOPT_CUDA_TRY(cudaLaunchKernel(k.fn, dim3(unsigned(grid)), dim3(unsigned(k.threads)), params, 0, ctx->stream));
  return MOPT_OK;
}

AlignAcc acc_of(const mopt_align_moments& t) {
  AlignAcc a{};
  a.w = t.w;
  for (int k = 0; k < 3; ++k) a.mean_src[k] = t.mean_src[k], a.mean_tgt[k] = t.mean_tgt[k];
  for (int k = 0; k < 9; ++k) a.cross[k] = t.cross[k];
  a.var_src = t.var_src;
  a.var_tgt = t.var_tgt;
  return a;
}

// The terms of `a` (counts left to the caller): each mean rounded to one double.
mopt_align_moments terms_of(const AlignAcc& a) {
  mopt_align_moments t;
  std::memset(&t, 0, sizeof(t));
  t.w = a.w;
  for (int k = 0; k < 3; ++k) t.mean_src[k] = a.mean_src[k], t.mean_tgt[k] = a.mean_tgt[k];
  for (int k = 0; k < 9; ++k) t.cross[k] = a.cross[k];
  t.var_src = a.var_src;
  t.var_tgt = a.var_tgt;
  return t;
}

bool terms_finite(const mopt_align_moments& t) {
  bool ok = std::isfinite(t.w) && std::isfinite(t.var_src) && std::isfinite(t.var_tgt);
  for (int k = 0; k < 3; ++k) ok = ok && std::isfinite(t.mean_src[k]) && std::isfinite(t.mean_tgt[k]);
  for (int k = 0; k < 9; ++k) ok = ok && std::isfinite(t.cross[k]);
  return ok;
}

}  // namespace

extern "C" {

int mopt_align_terms(mopt_ctx* ctx, mopt_store* store, const mopt_problem* problem, const double* x, int64_t first,
                     int64_t count, double inlier_threshold, mopt_align_moments* out) try {
  MOPT_REQUIRE(ctx && store && store->ctx == ctx, "store does not belong to this context");
  MOPT_REQUIRE(store->model == MOPT_MODEL_POINT2POINT, "closed-form alignment needs a point2point store");
  MOPT_TRY(validate_problem(store, problem, false));
  MOPT_REQUIRE(first >= 0 && count >= 0 && first <= store->n && count <= store->n - first,
               "the range [first, first + count) must lie inside the store");
  MOPT_REQUIRE(inlier_threshold >= 0.0, "inlier_threshold must not be negative or NaN");
  MOPT_REQUIRE(x && out, "null x or out");
  if (count == 0) {
    std::memset(out, 0, sizeof(*out));
    return MOPT_OK;
  }
  MOPT_CUDA_TRY(cudaSetDevice(ctx->device));
  MOPT_TRY(setup_slot(ctx, 0, problem, x));
  AlignArgs al;
  al.first = first;
  al.count = count;
  al.thr2 = inlier_threshold * inlier_threshold;  // as mopt_evaluate forms it
  al.out = ctx->d_align;
  MOPT_TRY(launch_align(ctx, store, problem, al));
  double* h = ctx->h_result->v;  // pinned bounce buffer (idle between calls)
  MOPT_CUDA_TRY(cudaMemcpyAsync(h, ctx->d_align, sizeof(AlignAcc), cudaMemcpyDeviceToHost, ctx->stream));
  MOPT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  AlignAcc acc;
  std::memcpy(&acc, h, sizeof(acc));
  mopt_align_moments t = terms_of(acc);  // mean + lo rounds to mean: the two-sum pairs are normalised
  t.n_valid = int64_t(acc.n_valid);
  t.n_used = int64_t(acc.n_used);
  *out = t;
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_align_terms_merge(const mopt_align_moments* a, const mopt_align_moments* b, mopt_align_moments* out) try {
  MOPT_REQUIRE(a && b && out, "null argument");
  AlignAcc m;
  align_merge(acc_of(*a), acc_of(*b), m);
  mopt_align_moments t = terms_of(m);
  t.n_valid = a->n_valid + b->n_valid;  // exact in int64, whatever the counts
  t.n_used = a->n_used + b->n_used;
  *out = t;
  return MOPT_OK;
}
MOPT_ABI_CATCH

int mopt_align_from_terms(const mopt_align_moments* terms, double* x_out, mopt_align_report* report) try {
  MOPT_REQUIRE(terms && x_out, "null terms or x_out");
  MOPT_REQUIRE(terms_finite(*terms), "the terms are not finite");
  MOPT_REQUIRE(terms->w > 0.0, "the terms have no weight (w <= 0)");
  // Horn's N from S = cross (source a, target b): max over unit quaternions q of q^T N q = max sum w q'.(R p')
  const double* S = terms->cross;
  const double xx = S[0], xy = S[1], xz = S[2], yx = S[3], yy = S[4], yz = S[5], zx = S[6], zy = S[7], zz = S[8];
  const double N[16] = {xx + yy + zz, yz - zy,       zx - xz,       xy - yx,        // column-major, symmetric
                        yz - zy,      xx - yy - zz,  xy + yx,       zx + xz,
                        zx - xz,      xy + yx,       -xx + yy - zz, yz + zy,
                        xy - yx,      zx + xz,       yz + zy,       -xx - yy + zz};
  double A[16], V[16];
  std::memcpy(A, N, sizeof(A));
  jacobi_eigen(4, A, V);
  int order[4] = {0, 1, 2, 3};  // eigenvalues descending (stable among equal ones)
  for (int i = 1; i < 4; ++i)
    for (int j = i; j > 0 && A[order[j] * 5] > A[order[j - 1] * 5]; --j) {
      const int o = order[j];
      order[j] = order[j - 1];
      order[j - 1] = o;
    }
  const double* v = V + 4 * order[0];
  double q0 = v[0], qx = v[1], qy = v[2], qz = v[3];
  const double qn = std::sqrt(q0 * q0 + qx * qx + qy * qy + qz * qz);
  const double sgn = q0 < 0.0 ? -1.0 : 1.0;  // q and -q are the same rotation: take w >= 0
  q0 *= sgn / qn, qx *= sgn / qn, qy *= sgn / qn, qz *= sgn / qn;
  const double R[9] = {q0 * q0 + qx * qx - qy * qy - qz * qz, 2.0 * (qx * qy - q0 * qz), 2.0 * (qx * qz + q0 * qy),
                       2.0 * (qy * qx + q0 * qz), q0 * q0 - qx * qx + qy * qy - qz * qz, 2.0 * (qy * qz - q0 * qx),
                       2.0 * (qz * qx - q0 * qy), 2.0 * (qz * qy + q0 * qx), q0 * q0 - qx * qx - qy * qy + qz * qz};
  double x[6];
  for (int i = 0; i < 3; ++i)
    x[i] = terms->mean_tgt[i] -
           (R[3 * i] * terms->mean_src[0] + R[3 * i + 1] * terms->mean_src[1] + R[3 * i + 2] * terms->mean_src[2]);
  // omega = angle * axis with angle = 2 atan2(|v|, w): well conditioned near 0 and near pi
  const double vn = std::sqrt(qx * qx + qy * qy + qz * qz);
  const double f = vn > 0.0 ? 2.0 * std::atan2(vn, q0) / vn : 2.0;  // the limit 2 / w with w = 1 at vn = 0
  x[3] = f * qx;
  x[4] = f * qy;
  x[5] = f * qz;
  std::memcpy(x_out, x, sizeof(x));
  if (report) {
    mopt_align_report r;
    std::memset(&r, 0, sizeof(r));
    for (int i = 0; i < 4; ++i) r.eig[i] = A[order[i] * 5];
    r.cost = std::fmax(0.0, terms->var_src + terms->var_tgt - 2.0 * r.eig[0]);
    r.rms = std::sqrt(r.cost / terms->w);
    r.degenerate = (r.eig[0] - r.eig[1] <= 1e-12 * std::fabs(r.eig[0])) ? 1 : 0;
    *report = r;
  }
  return MOPT_OK;
}
MOPT_ABI_CATCH

}  // extern "C"
