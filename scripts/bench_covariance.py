"""Time of the covariance terms (mopt_covariance_terms) on one GPU: prints one JSON line.

    python scripts/bench_covariance.py [--calls 50] [--warmup 5] [--out FILE]

Cases (every working set is larger than the 126 MB L2 of a B200, so each sweep streams from HBM):
  p2p           point2point, 100 M, fp32 store + compute, analytical Jacobian, Huber     (24 B per element)
  camera_p6     pinhole, 50 M, fp32, central differences                                 (20 B per element)
  camera_p15    pinhole + distortion, 50 M, fp32, central differences                    (20 B per element)
For each case the same run times mopt_covariance_terms (set-up, the linearization pass that gives H / b / sum, the
score Gram pass, one synchronisation) and mopt_linearize of the same problem (set-up, the same linearization pass,
one synchronisation); their difference is the score Gram pass.  Milliseconds per call come from CUDA events on the
context stream around `--calls` back-to-back calls after `--warmup` calls.  The score Gram pass's rate is over the
bytes it reads (from shapes).  GPU name, power limit and max SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_evaluate import gpu_info, time_calls  # noqa: E402


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    assert args.calls >= 50, "time at least 50 calls"
    from moptimizer_0_b200 import capi
    from tests.common import camera_consts

    info = gpu_info()
    ctx = capi.Context(0)
    hbm = ctx.measure_peaks()["hbm_read_gbs"]
    cases = {}

    def record(name, st, prob, x, n, read_b):
        ms_cov = time_calls(ctx, lambda: ctx.covariance_terms([st], [prob], x), args.calls, args.warmup)
        ms_lin = time_calls(ctx, lambda: ctx.linearize(st, prob, x), args.calls, args.warmup)
        g_ms = ms_cov - ms_lin
        gbs = n * read_b / (g_ms * 1e-3) / 1e9
        cases[name] = {"n": n, "covariance_terms_ms": round(ms_cov, 4), "linearize_ms": round(ms_lin, 4),
                       "g_pass_ms": round(g_ms, 4), "g_pass_gb_per_s": round(gbs, 1),
                       "g_pass_fraction_of_hbm_read": round(gbs / hbm, 3)}

    n = 100_000_000
    x = np.array([0.5, -0.3, 0.2, 0.1, -0.05, 0.08])
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    st.generate(seed=1, gt=x, noise_sigma=0.01, outlier_fraction=0.05, outlier_range=1.0)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32, loss=capi.LOSS_HUBER, loss_param=0.05)
    record("p2p", st, prob, x, n, 24)
    st.close()

    # the camera workloads of bench.py
    n = 50_000_000
    consts = camera_consts()
    x6 = np.array([-0.01, 0.02, -0.06, 0.018, -0.0013, 0.027])
    M = consts[:12].reshape(3, 4) @ capi.so3_convert6dof(x6) @ consts[12:].reshape(4, 4)
    st = capi.Store(ctx, capi.MODEL_PINHOLE, n, capi.F32)
    st.generate(seed=3, gt=M.reshape(-1), lo=(2.0, -1.0, -0.5), hi=(5.0, 1.0, 1.0), noise_sigma=0.5)
    prob = capi.make_problem(capi.MODEL_PINHOLE, capi.JAC_CENTRAL, capi.F32, consts=consts)
    record("camera_p6", st, prob, x6, n, 20)
    st.close()
    x15 = np.concatenate([x6, [600.0, 600.0, 320.0, 240.0, 0.05, -0.02, 0.001, -0.001, 0.005]])
    C44 = consts[12:]
    st = capi.Store(ctx, capi.MODEL_PINHOLE_DISTORT, n, capi.F32)
    st.generate(seed=3, gt=x15, lo=(2.0, -1.0, -0.5), hi=(5.0, 1.0, 1.0), noise_sigma=0.5, consts=C44)
    prob = capi.make_problem(capi.MODEL_PINHOLE_DISTORT, capi.JAC_CENTRAL, capi.F32, consts=C44)
    record("camera_p15", st, prob, x15, n, 20)
    st.close()
    ctx.close()

    line = json.dumps({"bench": "covariance", **info, "hbm_read_gbs_measured": round(hbm, 1), "calls": args.calls,
                       "warmup": args.warmup, "cases": cases})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
