"""Throughput of hypothesis scoring (mopt_score_hypotheses) on one GPU: prints one JSON line.

    python scripts/bench_hypotheses.py [--calls 10] [--warmup 2] [--out FILE]

Cases (every working set is larger than the 126 MB L2 of a B200, so each tile's pass streams from HBM):
  p2p_K       point2point, 100 M, fp32 store + compute, K = 1, 8, 32, 256, 1024     (RANSAC on correspondences)
  pnp_256     pinhole P = 6, 50 M, fp32, K = 256                                    (PnP-RANSAC)
  curve_64    exp curve, 10 M, fp64 store + compute, K = 64                         (multi-start)
Each case reports ms per call, hypothesis-element evaluations per second (K n / t), and the time of K back-to-back
statistics-only mopt_evaluate calls at the same hypotheses, measured in the same run, with the ratio of the two.
Milliseconds come from CUDA events on the context stream around back-to-back calls after warm-up calls; every call
synchronises the stream, so the figure includes the host side of the call (the K evaluate calls: K host round trips).
GPU name, power limit and max SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from scripts.bench_evaluate import gpu_info, time_calls  # noqa: E402


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    assert args.calls >= 3, "time at least 3 calls"
    from moptimizer_0_b200 import capi
    from tests.common import camera_consts

    info = gpu_info()
    ctx = capi.Context(0)
    cases = {}
    rng = np.random.default_rng(0)

    def record(name, st, prob, x, n, K, thr):
        xs = x + rng.normal(0, 1, (K, len(x))) * (0.01 * np.abs(x) + 1e-3)
        ms = time_calls(ctx, lambda: ctx.score_hypotheses(st, prob, xs, thr), args.calls, args.warmup)

        def evaluate_all():
            for xk in xs:
                ctx.evaluate(st, prob, xk, inlier_threshold=thr, residuals=False, weights=False)
        ev = time_calls(ctx, evaluate_all, max(3, args.calls * 8 // K), 1)
        sc = ctx.score_hypotheses(st, prob, xs, thr)
        cases[name] = {"n": n, "K": K, "ms_per_call": round(ms, 4), "hyp_elem_per_s": float(f"{K * n / (ms * 1e-3):.4g}"),
                       "evaluate_k_calls_ms": round(ev, 4), "speedup_over_evaluate": round(ev / ms, 2),
                       "best_n_inliers": int(sc.n_inliers.max()), "n_valid": int(sc.n_valid[0])}

    # point2point, 100 M, fp32
    n = 100_000_000
    x = np.array([0.5, -0.3, 0.2, 0.1, -0.05, 0.08])
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    st.generate(seed=1, gt=x, noise_sigma=0.01, outlier_fraction=0.05, outlier_range=1.0)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32)
    for K in (1, 8, 32, 256, 1024):
        record(f"p2p_{K}", st, prob, x, n, K, 0.03)
    st.close()

    # pinhole P = 6, 50 M, fp32
    n = 50_000_000
    x = np.array([-0.01, 0.02, -0.06, 0.018, -0.0013, 0.027])
    cam = camera_consts()
    M = cam[:12].reshape(3, 4) @ capi.so3_convert6dof(x) @ cam[12:].reshape(4, 4)
    st = capi.Store(ctx, capi.MODEL_PINHOLE, n, capi.F32)
    st.generate(seed=3, gt=M.reshape(-1), lo=(2.0, -1.0, -0.5), hi=(5.0, 1.0, 1.0), noise_sigma=0.5)
    prob = capi.make_problem(capi.MODEL_PINHOLE, capi.JAC_CENTRAL, capi.F32, consts=cam)
    record("pnp_256", st, prob, x, n, 256, 2.0)
    st.close()

    # exp curve, 10 M, fp64
    n = 10_000_000
    x = np.array([0.3, 0.1])
    st = capi.Store(ctx, capi.MODEL_EXP_CURVE, n, capi.F64)
    st.generate(seed=2, gt=x, lo=(0, 0, 0), hi=(5, 0, 0), n_total=n, noise_sigma=0.2)
    prob = capi.make_problem(capi.MODEL_EXP_CURVE, capi.JAC_FORWARD, capi.F64)
    record("curve_64", st, prob, x, n, 64, 0.4)
    st.close()
    ctx.close()

    line = json.dumps({"bench": "hypotheses", **info, "calls": args.calls, "warmup": args.warmup, "cases": cases})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
