"""Throughput of exact residual quantiles (mopt_residual_quantiles) on one GPU: prints one JSON line.

    python scripts/bench_quantiles.py [--calls 20] [--warmup 3] [--out FILE]

Cases (every working set is larger than the 126 MB L2 of a B200, so each sweep streams from HBM):
  p2p       point2point, 100 M, fp32 store + compute, q = (0.5, 0.9, 0.99)   (4 sweeps of 24 B per element)
  camera    pinhole + distortion, 50 M, fp32, q = (0.5, 0.9, 0.99)           (4 sweeps of 20 B per element)
  curve     exp curve, 10 M, fp64 store + compute, q = (0.5, 0.9, 0.99)      (8 sweeps of 16 B per element)
For comparison each case also times mopt_evaluate with statistics only on the same store: one sweep over the same
bytes.  Milliseconds per call come from CUDA events on the context stream around `--calls` back-to-back calls after
`--warmup` calls; every call synchronises the stream, so the figure includes the host side of the call.  ms per
sweep is ms per call over the number of sweeps (the one-CTA steps between sweeps included).  Bytes are algorithmic
(read streams, from shapes); the HBM read ceiling is mopt_measure_peaks' read-only stream, measured in the same run.
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
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    assert args.calls >= 20, "time at least 20 calls"
    from moptimizer_0_b200 import capi
    from tests.common import camera_consts

    info = gpu_info()
    ctx = capi.Context(0)
    hbm = ctx.measure_peaks()["hbm_read_gbs"]
    cases = {}
    q = (0.5, 0.9, 0.99)

    def record(name, st, prob, x, n, read_b):
        sweeps = 4 if prob.compute_dtype == capi.F32 else 8
        ms = time_calls(ctx, lambda: ctx.quantiles(st, prob, x, q), args.calls, args.warmup)
        ev = time_calls(ctx, lambda: ctx.evaluate(st, prob, x, residuals=False, weights=False), args.calls,
                        args.warmup)
        nbytes = n * read_b * sweeps
        gbs = nbytes / (ms * 1e-3) / 1e9
        ev_gbs = n * read_b / (ev * 1e-3) / 1e9
        r = ctx.quantiles(st, prob, x, q)
        cases[name] = {"n": n, "q": list(q), "sweeps": sweeps, "ms_per_call": round(ms, 4),
                       "ms_per_sweep": round(ms / sweeps, 4), "bytes": nbytes, "gb_per_s": round(gbs, 1),
                       "fraction_of_hbm_read": round(gbs / hbm, 3), "evaluate_stats_ms": round(ev, 4),
                       "evaluate_stats_fraction_of_hbm_read": round(ev_gbs / hbm, 3),
                       "sweep_over_evaluate": round(ms / sweeps / ev, 3),
                       "median": r.median, "robust_sigma": r.robust_sigma}

    # point2point, 100 M, fp32
    n = 100_000_000
    x = np.array([0.5, -0.3, 0.2, 0.1, -0.05, 0.08])
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    st.generate(seed=1, gt=x, noise_sigma=0.01, outlier_fraction=0.05, outlier_range=1.0)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32, loss=capi.LOSS_HUBER, loss_param=0.05)
    record("p2p", st, prob, x, n, 24)
    st.close()

    # pinhole + distortion, 50 M, fp32
    n = 50_000_000
    x = np.array([-0.01, 0.02, -0.06, 0.018, -0.0013, 0.027, 586.0, 722.0, 638.0, 323.0, -0.12, 0.05, 0.001, -0.0007,
                  0.01])
    cm = camera_consts()[12:]
    st = capi.Store(ctx, capi.MODEL_PINHOLE_DISTORT, n, capi.F32)
    st.generate(seed=3, gt=x, lo=(2.0, -1.0, -0.5), hi=(5.0, 1.0, 1.0), noise_sigma=0.3, consts=cm)
    prob = capi.make_problem(capi.MODEL_PINHOLE_DISTORT, capi.JAC_CENTRAL, capi.F32, consts=cm)
    record("camera", st, prob, x, n, 20)
    st.close()

    # exp curve, 10 M, fp64
    n = 10_000_000
    x = np.array([0.3, 0.1])
    st = capi.Store(ctx, capi.MODEL_EXP_CURVE, n, capi.F64)
    st.generate(seed=2, gt=x, lo=(0, 0, 0), hi=(5, 0, 0), n_total=n, noise_sigma=0.2)
    prob = capi.make_problem(capi.MODEL_EXP_CURVE, capi.JAC_FORWARD, capi.F64)
    record("curve", st, prob, x, n, 16)
    st.close()
    ctx.close()

    line = json.dumps({"bench": "quantiles", **info, "hbm_read_gbs_measured": round(hbm, 1), "calls": args.calls,
                       "warmup": args.warmup, "cases": cases})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
