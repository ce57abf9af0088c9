"""Throughput of closed-form alignment terms (mopt_align_terms) on one GPU: prints one JSON line.

    python scripts/bench_align.py [--calls 50] [--warmup 5] [--rounds 3] [--out FILE]

Cases, all on one point2point store of 100 M pairs in fp32 (2.4 GB: larger than the 126 MB L2 of a B200, so each call
streams from HBM and reads 24 B per element):
  none_inf      fp32 compute, loss NONE, inlier_threshold = +inf (every pair is used)
  huber_thr     fp32 compute, Huber k = 0.05, inlier_threshold = 0.05 (95 % inliers, 5 % outliers)
  f64_compute   fp64 compute, loss NONE, inlier_threshold = +inf
and, for each, mopt_evaluate statistics-only on the same store and problem, timed in the same run: `--rounds` rounds
alternate the two calls, `--calls` back-to-back calls each after `--warmup` calls.  Milliseconds per call come from CUDA
events on the context stream; every call synchronises the stream, so the figure includes the host side of the call
(mopt_align_terms: set-up kernel, terms kernel, one 208-byte copy back).  Bytes are algorithmic (24 B per element);
the HBM read ceiling is mopt_measure_peaks' read-only stream, measured in the same run.  GPU name, power limit and max
SM clock are read in the same run.
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
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    assert args.calls >= 50, "time at least 50 calls"
    from moptimizer_0_b200 import capi

    info = gpu_info()
    ctx = capi.Context(0)
    hbm = ctx.measure_peaks()["hbm_read_gbs"]
    n = 100_000_000
    x = np.array([0.5, -0.3, 0.2, 0.1, -0.05, 0.08])
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    st.generate(seed=1, gt=x, noise_sigma=0.01, outlier_fraction=0.05, outlier_range=1.0)
    cases = {}
    for name, cdt, loss, k, thr in (("none_inf", capi.F32, capi.LOSS_NONE, 0.0, np.inf),
                                    ("huber_thr", capi.F32, capi.LOSS_HUBER, 0.05, 0.05),
                                    ("f64_compute", capi.F64, capi.LOSS_NONE, 0.0, np.inf)):
        prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, cdt, loss=loss, loss_param=k)
        align_ms, eval_ms = [], []
        for _ in range(args.rounds):
            align_ms.append(time_calls(ctx, lambda: ctx.align_terms(st, prob, x, thr), args.calls, args.warmup))
            eval_ms.append(time_calls(ctx, lambda: ctx.evaluate(st, prob, x, inlier_threshold=thr, residuals=False,
                                                                weights=False), args.calls, args.warmup))
        t = ctx.align_terms(st, prob, x, thr)
        a = capi.align_from_terms(t)
        best = min(align_ms)
        gbs = n * 24 / (best * 1e-3) / 1e9
        cases[name] = {"n": n, "n_used": t.n_used, "align_ms_per_call": [round(v, 4) for v in align_ms],
                       "evaluate_ms_per_call": [round(v, 4) for v in eval_ms],
                       "align_over_evaluate": round(best / min(eval_ms), 3), "bytes": n * 24,
                       "gb_per_s": round(gbs, 1), "fraction_of_hbm_read": round(gbs / hbm, 3),
                       "max_abs_x_minus_gt": float(np.max(np.abs(a.x - x)))}
    st.close()
    ctx.close()

    line = json.dumps({"bench": "align", **info, "hbm_read_gbs_measured": round(hbm, 1), "calls": args.calls,
                       "warmup": args.warmup, "rounds": args.rounds, "cases": cases})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
