// The snippet of INTEGRATION.md §1 as a program: rigid registration of two clouds through the C++ mirror of the
// reference API (same class names and call sequence as tst/point2point.cpp:142-160), whole LM loop on the GPU.
//
//   g++ -std=c++17 -Iinclude examples/point2point_registration.cpp -Lmoptimizer_0_b200 -lmopt_b200
//       -Wl,-rpath,$PWD/moptimizer_0_b200 -o /tmp/p2p_example && /tmp/p2p_example [n]
//
// Exits 77 with a message when no CUDA device is usable: there is no CPU fallback.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>

#include <moptimizer/cost_function_analytical_dyn.h>
#include <moptimizer/levenberg_marquadt_dyn.h>
#include <moptimizer/loss_function/huber.h>
#include <moptimizer/device/models.h>
#include <moptimizer/so3.h>

int main(int argc, char** argv) {
  const long n = argc > 1 ? std::atol(argv[1]) : 1000000;
  // synthetic clouds: tgt = T_gt src + noise, 5 % outliers (what bench.py generates on the device)
  const double x_gt[6] = {0.5, -0.3, 0.2, 0.10, -0.05, 0.08};
  double T[16];
  so3::convert6DOFParameterToMatrix<double>(x_gt, T);
  std::mt19937_64 rng(2);
  std::uniform_real_distribution<double> box(0.0, 10.0), out(-1.0, 1.0), u01(0.0, 1.0);
  std::normal_distribution<double> noise(0.0, 0.01);
  std::vector<double> src(3 * n), tgt(3 * n);
  for (long i = 0; i < n; ++i) {
    double* p = &src[3 * i];
    for (int k = 0; k < 3; ++k) p[k] = box(rng);
    const bool outlier = u01(rng) < 0.05;
    for (int k = 0; k < 3; ++k)
      tgt[3 * i + k] = T[k * 4] * p[0] + T[k * 4 + 1] * p[1] + T[k * 4 + 2] * p[2] + T[k * 4 + 3] + noise(rng) +
                       (outlier ? out(rng) : 0.0);
  }
  try {
    auto ctx = moptimizer::device::Context::create(0);
    // fp32 planar streams in HBM (24 B per correspondence), fp64 LM arithmetic: the benchmark configuration
    auto model = std::make_shared<moptimizer::device::Point2Point<double>>(ctx, src.data(), tgt.data(), n,
                                                                          MOPT_P2P_EXACT, MOPT_F32);
    moptimizer::CostFunctionAnalyticalDynamic<double> cost(model, 6, 3, int(n));
    cost.setLossFunction(std::make_shared<moptimizer::loss::Huber<double>>(0.05));
    moptimizer::LevenbergMarquadtDynamic<double> lm(6);
    lm.setMaximumIterations(50);
    lm.addCost(&cost);
    double x0[6] = {0, 0, 0, 0, 0, 0};
    const auto status = lm.minimize(x0);
    double err = 0;
    for (int i = 0; i < 6; ++i) err = std::fmax(err, std::fabs(x0[i] - x_gt[i]));
    std::printf("status %d after %d iterations, x = (%.5f %.5f %.5f %.5f %.5f %.5f), max |x - x_gt| = %.2e\n", int(status),
                lm.getExecutedIterations(), x0[0], x0[1], x0[2], x0[3], x0[4], x0[5], err);
    // registration quality at the solution: correspondences within 3 noise sigmas (0.03) of their target
    const mopt_eval_stats fit = cost.evaluateStatistics(x0, 0.03);
    std::printf("fitness %.4f (%lld of %ld residuals within 0.03), inlier RMSE %.5f\n", double(fit.n_inliers) / double(n),
                (long long)fit.n_inliers, n, fit.n_inliers ? std::sqrt(fit.inlier_sum_sq / double(fit.n_inliers)) : 0.0);
    // the distribution of the correspondence distances |r| and the robust noise scale, which outliers do not inflate
    const mopt_quantiles qd = cost.residualQuantiles(x0, {0.5, 0.9});
    std::printf("correspondence distance: median %.5f, 90th percentile %.5f, robust sigma %.5f\n", std::sqrt(qd.value[0]),
                std::sqrt(qd.value[1]), qd.robust_sigma);
    // hypothesis scoring (the RANSAC step): the solution against the start, scored in one pass over the data
    double hyps[12] = {0, 0, 0, 0, 0, 0};
    for (int i = 0; i < 6; ++i) hyps[6 + i] = x0[i];
    const std::vector<mopt_eval_stats> sc = cost.scoreHypotheses(hyps, 2, 0.03);
    std::printf("inliers within 0.03: %lld at x = 0, %lld at the solution\n", (long long)sc[0].n_inliers,
                (long long)sc[1].n_inliers);
    // how certain the pose is: standard deviations from s^2 H^-1, s^2 estimated from the fit
    double cov[36];
    mopt_cov_report rep;
    lm.computeCovariance(x0, MOPT_COV_SCALED, cov, &rep);
    std::printf("std (t, omega) = (%.2e %.2e %.2e %.2e %.2e %.2e), rank %d, sigma^2 %.3e\n", std::sqrt(cov[0]),
                std::sqrt(cov[7]), std::sqrt(cov[14]), std::sqrt(cov[21]), std::sqrt(cov[28]), std::sqrt(cov[35]),
                rep.rank, rep.sigma2);
    return err < 1e-3 ? 0 : 1;
  } catch (const moptimizer::Exception& e) {
    std::printf("moptimizer::Exception: %s\n", e.what());
    return 77;
  }
}
