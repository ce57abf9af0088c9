"""Throughput of per-residual evaluation (mopt_evaluate) on one GPU: prints one JSON line.

    python scripts/bench_evaluate.py [--calls 50] [--warmup 5] [--out FILE]

Cases (every working set is larger than the 126 MB L2 of a B200, so each call streams from HBM):
  p2p_stats     point2point, 100 M, fp32 store + compute, statistics only          (reads 24 B per element)
  p2p_outputs   the same, also writing fp32 residuals (12 B) and weights (4 B)
  cost_pass     mopt_compute_cost on the same store: the pass that reads the same 24 B per element
  camera        pinhole + distortion, 50 M, fp32, fp32 residuals + weights         (reads 20 B, writes 12 B)
  curve         exp curve, 10 M, fp64 store + compute + outputs                    (reads 16 B, writes 16 B: 320 MB;
                an fp32 store of 10 M would be 80 MB and fit in L2)
Milliseconds per call come from CUDA events on the context stream around `--calls` back-to-back calls after
`--warmup` calls; every call synchronises the stream, so the figure includes the host side of the call.  Bytes are
algorithmic (read streams + written outputs, from shapes); the HBM read ceiling is mopt_measure_peaks' read-only
stream, measured in the same run.  GPU name, power limit and max SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True)
    name, power, clock = [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def time_calls(ctx, fn, calls: int, warmup: int) -> float:
    import torch
    for _ in range(warmup):
        fn()
    stream = torch.cuda.ExternalStream(ctx.stream())
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(calls):
        fn()
    t1.record(stream)
    t1.synchronize()
    return t0.elapsed_time(t1) / calls


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    assert args.calls >= 50, "time at least 50 calls"
    import torch
    from moptimizer_0_b200 import capi
    from tests.common import camera_consts

    info = gpu_info()
    ctx = capi.Context(0)
    hbm = ctx.measure_peaks()["hbm_read_gbs"]
    dev = torch.device("cuda", 0)
    cases = {}

    def record(name, fn, n, read_b, write_b):
        ms = time_calls(ctx, fn, args.calls, args.warmup)
        nbytes = n * (read_b + write_b)
        gbs = nbytes / (ms * 1e-3) / 1e9
        cases[name] = {"n": n, "ms_per_call": round(ms, 4), "bytes": nbytes, "gb_per_s": round(gbs, 1),
                       "fraction_of_hbm_read": round(gbs / hbm, 3)}

    # point2point, 100 M, fp32
    n = 100_000_000
    x = np.array([0.5, -0.3, 0.2, 0.1, -0.05, 0.08])
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    st.generate(seed=1, gt=x, noise_sigma=0.01, outlier_fraction=0.05, outlier_range=1.0)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32, loss=capi.LOSS_HUBER, loss_param=0.05)
    record("p2p_stats", lambda: ctx.evaluate(st, prob, x, inlier_threshold=0.05, residuals=False, weights=False),
           n, 24, 0)
    out = (torch.empty((n, 3), dtype=torch.float32, device=dev), torch.empty((n,), dtype=torch.float32, device=dev))
    record("p2p_outputs", lambda: ctx.evaluate(st, prob, x, inlier_threshold=0.05, out=out), n, 24, 16)
    record("cost_pass", lambda: ctx.compute_cost(st, prob, x), n, 24, 0)
    del out
    st.close()

    # pinhole + distortion, 50 M, fp32
    n = 50_000_000
    x = np.array([-0.01, 0.02, -0.06, 0.018, -0.0013, 0.027, 586.0, 722.0, 638.0, 323.0, -0.12, 0.05, 0.001, -0.0007,
                  0.01])
    cm = camera_consts()[12:]
    st = capi.Store(ctx, capi.MODEL_PINHOLE_DISTORT, n, capi.F32)
    st.generate(seed=3, gt=x, lo=(2.0, -1.0, -0.5), hi=(5.0, 1.0, 1.0), noise_sigma=0.3, consts=cm)
    prob = capi.make_problem(capi.MODEL_PINHOLE_DISTORT, capi.JAC_CENTRAL, capi.F32, consts=cm)
    out = (torch.empty((n, 2), dtype=torch.float32, device=dev), torch.empty((n,), dtype=torch.float32, device=dev))
    record("camera", lambda: ctx.evaluate(st, prob, x, inlier_threshold=1.0, out=out), n, 20, 12)
    del out
    st.close()

    # exp curve, 10 M, fp64
    n = 10_000_000
    x = np.array([0.3, 0.1])
    st = capi.Store(ctx, capi.MODEL_EXP_CURVE, n, capi.F64)
    st.generate(seed=2, gt=x, lo=(0, 0, 0), hi=(5, 0, 0), n_total=n, noise_sigma=0.2)
    prob = capi.make_problem(capi.MODEL_EXP_CURVE, capi.JAC_FORWARD, capi.F64)
    out = (torch.empty((n, 1), dtype=torch.float64, device=dev), torch.empty((n,), dtype=torch.float64, device=dev))
    record("curve", lambda: ctx.evaluate(st, prob, x, inlier_threshold=0.4, out=out, out_dtype=capi.F64), n, 16, 16)
    del out
    st.close()
    ctx.close()

    line = json.dumps({"bench": "evaluate", **info, "hbm_read_gbs_measured": round(hbm, 1), "calls": args.calls,
                       "warmup": args.warmup, "cases": cases})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
