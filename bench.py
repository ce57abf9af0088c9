#!/usr/bin/env python
"""bench.py — point2point linearization throughput (Gres/s) on B200, the BASELINE.json metric.

Headline workload (BASELINE.json configs[2], SURVEY.md §8d C3): point-to-point rigid registration,
100 M correspondences per GPU, analytical Jacobian + Huber loss, fp32 planar streams resident in
HBM (24 B per correspondence), fp32 residual math with fp64 accumulation.  A "step" is one
linearization pass (H, b, sum r^T r) over every rank's shard plus, for N > 1, the exchange of the 28
packed fp64 values (NVLink peer exchange fused into the pass kernel; `--collective nccl` for the
NCCL all-reduce baseline).  Weak scaling: every rank holds `--n` correspondences.

The same JSON line also carries (under "configs") the other BASELINE.json configurations, each with its own
roofline: curve fitting 10 M (central differences), camera calibration 50 M with 6 and 15 parameters, the
small-problem LM (tst/point2point's 29 310-point cloud) and, for N > 1, the 1 B-correspondence strong-scaling split
of configs[3]; "peaks" holds the fp32 FMA / issue / HBM-read / host-to-device ceilings measured in this run with
the library's micro-kernels; for N > 1 "check.vs_single_gpu" compares the exchanged result with the sum of every
shard's result recomputed on rank 0's GPU alone.

  python bench.py [--gpus N] [--steps K] [--warmup W]          # our CUDA path
  python bench.py --impl reference ...                         # CPU restatement of the reference, same workload
  python bench.py ... --dump-outputs DIR                       # also save the last timed step's H, b, sum as DIR/*.npy
Multi-GPU: python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "point2point_linearized_residuals_per_sec"
UNIT = "Gres/s"
BYTES_PER_RES = 24  # src xyz + tgt xyz, fp32 (SURVEY.md §8d)
X_GT = [0.5, -0.3, 0.2, 0.10, -0.05, 0.08]
HUBER_K = 0.05
SEED = 2
NOISE_SIGMA, OUTLIER_FRACTION, OUTLIER_RANGE = 0.01, 0.05, 1.0
GEN = dict(lo=(0, 0, 0), hi=(10, 10, 10), noise_sigma=NOISE_SIGMA, outlier_fraction=OUTLIER_FRACTION,
           outlier_range=OUTLIER_RANGE)
INST_COUNTS = os.path.join(ROOT, "profiles", "kernel_inst_counts.json")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", "--per-gpu", dest="n", type=int, default=100_000_000, help="correspondences per GPU")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-sample", type=int, default=20_000_000,
                    help="correspondences in the cpu_baseline sample of the GPU arm (the reference arm uses --n)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--ref-budget-s", type=float, default=240.0,
                    help="--impl reference: shrink the per-step sample only if (W + K) steps of --n would exceed this")
    ap.add_argument("--prewarm-steps", type=int, default=2000, help="untimed steps before the W warm-up steps")
    ap.add_argument("--ctas-per-sm", type=int, default=0)
    ap.add_argument("--threads", type=int, default=0,
                    help="launch-shape override (0 = default; 512 = second ring shape; 1024 = first-generation kernel)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-balance-threshold", type=float, default=1.1,
                    help="N > 1: add the e2e leg with shards proportional to the ranks' host-link rates when the fastest "
                         "link is this many times the slowest")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configurations")
    ap.add_argument("--no-check", action="store_true", help="N>1: skip the comparison with the single-GPU sums")
    ap.add_argument("--no-peaks", action="store_true")
    ap.add_argument("--lm", dest="lm", action="store_true", default=True,
                    help="also time a device-resident LM solve (LM iters/s, the second half of BASELINE.json's metric)")
    ap.add_argument("--no-lm", dest="lm", action="store_false")
    ap.add_argument("--collective", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: how the 28 packed doubles are combined per step")
    ap.add_argument("--strong-total", type=int, default=-1,
                    help="N>1: second timed region, this many correspondences in total sharded contiguously over the "
                         "ranks (BASELINE configs[3]); default 1e9 when N>1, 0 disables")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (H, b, sum r^T r of the headline workload) as "
                         "DIR/H.npy, DIR/b.npy, DIR/sum_rtr.npy (float64), so that two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(directory, H, b, s):
    """--dump-outputs: the arrays a caller of the timed path receives from its last step.  The inputs are the seeded
    generator's rows, so the same arguments give the same inputs in every run."""
    os.makedirs(directory, exist_ok=True)
    for name, v in (("H", H), ("b", b), ("sum_rtr", s)):
        np.save(os.path.join(directory, name + ".npy"), np.asarray(v, dtype=np.float64))


def workload_config(n_per_gpu: int, n_total: int) -> dict:
    """The keys that define the workload: identical in the GPU arm and in `--impl reference`."""
    return {"workload": f"point2point {n_per_gpu / 1e6:.0f}M correspondences/GPU, analytical Jacobian + Huber(k=0.05), x0=0",
            "n_per_gpu": n_per_gpu, "n_total": n_total,
            "generator": f"counter-based (splitmix64), seed {SEED}, src uniform in [0,10]^3, tgt = T_gt src + N(0,0.01^2), "
                         "5% outliers U(-1,1); identical rows on the device and on the host (tests/test_gpu_generator.py)",
            "l2": "inputs per step (2.4 GB fp32 / 4.8 GB fp64 per 100M) exceed every cache: no flush needed"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def inst_counts() -> dict:
    """Warp instructions per residual of each kernel, from the committed ncu captures (profiles/kernel_inst_counts.json,
    written by scripts/ncu_inst_counts.py): a property of the binary, used for the issue-slot rooflines."""
    try:
        return json.load(open(INST_COUNTS))
    except Exception:
        return {}


# ------------------------------------------------------------------------- clocks ----
class ClockSampler:
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self._stop = [], set(), threading.Event()
        self.times, self.window = [], None
        self.sm_max = None
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.times.append(time.perf_counter())
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.0005)

    def start(self):
        if self.nv is not None:
            self._stop.clear()
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        if self._t is not None:
            self._stop.set()
            self._t.join()
            self._t = None

    def mark(self):
        """Start (first call) / end (second call) of the timed region on the host clock."""
        t = time.perf_counter()
        self.window = (t, None) if self.window is None else (self.window[0], t)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": 0}
        pairs = list(zip(self.times, self.samples))
        where = "whole run"
        if self.window and self.window[1]:
            inside = [c for t, c in pairs if self.window[0] <= t <= self.window[1]]
            if len(inside) >= 5:
                pairs, where = [(0, c) for c in inside], "timed region"
            else:  # a short timed region: add the samples of the identical back-to-back steps just before it
                upto = [c for t, c in pairs if t <= self.window[1]]
                pairs, where = [(0, c) for c in upto[-max(10, len(inside)):]], "timed region + the warm-up steps before it"
        vals = [c for _, c in pairs]
        return {"sm_mhz": float(np.median(vals)), "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(vals), "window": where}


def bind_host_thread(index: int, local_rank: int, local_world: int):
    """Pin this process BEFORE any pinned host buffer is allocated: to the CPUs NVML reports as local to GPU `index`
    and, when several ranks share that set (a single-NUMA box reports every CPU for every GPU), to this rank's own
    contiguous 1/local_world slice of it, so the ranks' staging copies and first-touched pages do not compete for the
    same cores.  Returns a short note for the JSON line."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
        local = allowed
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(index)
            ncpu = os.cpu_count() or 1
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
            cpus = [w * 64 + b for w, mask in enumerate(words) for b in range(64) if (int(mask) >> b) & 1 and w * 64 + b < ncpu]
            local = sorted(set(cpus) & set(allowed)) or allowed
        except Exception:
            pass
        mine = local
        if local_world > 1 and len(local) >= local_world:
            per = len(local) // local_world
            mine = local[local_rank * per:(local_rank + 1) * per]
        os.sched_setaffinity(0, mine)
        return f"{len(mine)} of {len(local)} CPUs local to GPU {index} (CPUs {mine[0]}-{mine[-1]})"
    except Exception as e:  # containers without the syscall, ...
        return f"unavailable ({type(e).__name__})"


# ------------------------------------------------------------------ CPU (oracle) arm ----
def oracle_cost(src, tgt):
    from oracle import oracle_py as orc
    return orc.Cost(orc.P2P, 6, 3, src.shape[0], a=src, b=tgt, jac_mode=orc.JAC_ANALYTICAL, variant=orc.P2P_EXACT,
                    loss=orc.LOSS_HUBER, loss_param=HUBER_K)


def time_oracle(src, tgt, nthreads: int, budget_s: float):
    """-> (Gres/s, reps, seconds) for fp64 linearizations of the sample, at least one rep."""
    from oracle import oracle_py as orc
    cost = oracle_cost(src, tgt)
    x0 = [0.0] * 6
    t1, _, _, _ = orc.time_linearize(cost, x0, nthreads=nthreads, reps=1)
    reps = max(1, int(budget_s / max(t1, 1e-9)) - 1)
    reps = min(reps, 200)
    t, _, _, _ = orc.time_linearize(cost, x0, nthreads=nthreads, reps=reps)
    return src.shape[0] * reps / t / 1e9, reps, t


def run_reference(args):
    """`--impl reference`: the CPU restatement of the reference path (oracle port; the reference itself cannot be
    built in this image — no Eigen3/oneTBB) on all host threads, on the SAME workload as the GPU arm: the rows of
    rank 0's shard come from the host restatement of the device generator (bit-identical, tests/test_gpu_generator.py),
    W warm-up and K timed steps of one full linearization each.  Only if (W + K) full steps would not fit
    --ref-budget-s is the per-step sample shrunk, and the line says so."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle_py as orc
    cores = orc.hardware_concurrency() or (os.cpu_count() or 1)
    n_full = args.n
    steps, warmup = args.steps, max(0, args.warmup)
    # a quick probe decides whether the full per-GPU workload fits the time budget
    probe_n = min(n_full, 2_000_000)
    ps, pt = orc.generate_p2p(SEED, probe_n, X_GT, **GEN)
    t_probe, _, _, _ = orc.time_linearize(oracle_cost(ps, pt), [0.0] * 6, nthreads=cores, reps=1)
    est_step = t_probe * n_full / probe_n
    n = n_full
    if est_step * (steps + warmup) > args.ref_budget_s:
        n = max(probe_n, int(n_full * args.ref_budget_s / (est_step * (steps + warmup))))
    del ps, pt
    src, tgt = orc.generate_p2p(SEED, n, X_GT, **GEN)
    cost = oracle_cost(src, tgt)
    x0 = [0.0] * 6
    if warmup:
        orc.time_linearize(cost, x0, nthreads=cores, reps=warmup)
    t, H, b, s = orc.time_linearize(cost, x0, nthreads=cores, reps=steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, H, b, s)
    ms = t / steps * 1e3
    value = n / (t / steps) / 1e9
    sample = (f"{n} correspondences per step (fp64 AoS, the first rows of rank 0's shard"
              + ("" if n == n_full else f"; shrunk from {n_full} to fit --ref-budget-s {args.ref_budget_s:.0f}")
              + "), threaded linearization with thread-local H/b on all host threads (the reference's own loop is "
                "serial, linearization.h:142)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(n_full, n_full * max(1, args.gpus)),
        "cpu_sample_per_step": n,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "check": {"sum_rtr": s, "H00": float(H[0, 0]), "b0": float(b[0]), "rows": n},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------- GPU arm ----
class Timer:
    """CUDA-event timing of back-to-back asynchronous passes on the context's stream."""

    def __init__(self, torch, ctx, stream):
        self.torch, self.ctx, self.stream = torch, ctx, stream

    def ms_per_pass(self, store, prob, x, steps, warm):
        x = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
        for _ in range(warm):
            self.ctx.linearize_async(store, prob, x)
        self.ctx.synchronize()
        e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(steps):
            self.ctx.linearize_async(store, prob, x)
        e1.record(self.stream)
        self.ctx.synchronize()
        return e0.elapsed_time(e1) / steps


def alu_roofline(key, n, ms, bytes_per, pk, counts, hbm_peak):
    """Roofline of an ALU-bound pass: warp instructions issued per second against the measured issue peak
    (one instruction per clock per scheduler = the FFMA-only rate of csrc/mopt_peaks.cu), next to the HBM fraction."""
    out = {"bound": "fp32_issue", "hbm_gbs": n * bytes_per / (ms * 1e-3) / 1e9,
           "hbm_frac": n * bytes_per / (ms * 1e-3) / 1e9 / hbm_peak}
    c = counts.get(key)
    if c and pk:
        issue_peak = pk["fp32_fma_tflops"] * 1e12 / 64.0 / 1e9  # G warp-instructions/s: one FFMA = 64 flop per warp
        ach = c["warp_inst_per_residual"] * n / (ms * 1e-3) / 1e9
        out.update({"achieved": ach, "peak": issue_peak, "unit": "G warp-inst/s", "frac": ach / issue_peak,
                    "warp_inst_per_residual": c["warp_inst_per_residual"], "inst_source": c.get("source"),
                    "peak_source": "FFMA-only issue rate measured in this run (mopt_measure_peaks)"})
        if c.get("fma_pipe_inst_per_residual"):
            f = c["fma_pipe_inst_per_residual"] * n / (ms * 1e-3) / 1e9
            out["fma_pipe"] = {"achieved": f, "peak": issue_peak, "frac": f / issue_peak,
                               "note": "FMA-pipe warp instructions per second against the same peak (an FFMA2 is one instruction "
                                       "and occupies the pipe for two cycles)"}
        if c.get("tensor_pipe_inst_per_residual"):
            out["tensor_pipe"] = {"mma_per_residual": c["tensor_pipe_inst_per_residual"],
                                  "busy_pct_in_capture": c.get("tensor_pipe_pct"),
                                  "note": "mma.sync m16n8k4 TF32 (3xTF32 Gram matrix); share of cycles from the ncu capture"}
    else:
        out.update({"achieved": None, "peak": None, "unit": "G warp-inst/s", "frac": None})
    return out


def camera_consts():
    """K (3x4 row-major) ++ C (4x4 row-major) of tst/camera_calibration.cpp:22-30 (K from the golden fixtures)."""
    fx = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_fixtures.json")))
    K = np.array(fx["camera"]["K"], dtype=np.float64)
    c, s = np.cos(np.pi / 2), np.sin(np.pi / 2)
    rx = np.array([[1, 0, 0], [0, c, -s], [0, s, c]])
    rz = np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]])
    Cm = np.eye(4)
    Cm[:3, :3] = rx @ rz
    return np.concatenate([K, Cm.reshape(-1)])


def run_other_configs(capi, ctx, timer, pk, hbm_peak):
    """BASELINE.json configs[1], configs[4] (6 and 15 parameters) and configs[0]-sized LM, on this GPU."""
    counts = inst_counts()
    out = {}
    # configs[1]: curve fitting, 10 M samples, central differences, fp32 compute
    n = 10_000_000
    st = capi.Store(ctx, capi.MODEL_EXP_CURVE, n, capi.F32)
    st.generate(seed=1, gt=[0.3, 0.1], lo=(0, 0, 0), hi=(5, 0, 0), n_total=n, noise_sigma=0.2)
    prob = capi.make_problem(capi.MODEL_EXP_CURVE, capi.JAC_CENTRAL, capi.F32)
    ms = timer.ms_per_pass(st, prob, [0.25, 0.15], steps=200, warm=200)
    out["curve_10M_central"] = {
        "workload": "exp curve y = exp(m t + c), 10M samples, numerical central-difference Jacobian, fp32 (BASELINE configs[1])",
        "n": n, "ms": ms, "Gres_per_s": n / ms / 1e6, "l2": "80 MB of streams: L2-resident between passes (126 MB L2)",
        "roofline": alu_roofline("curve_central_f32", n, ms, 8, pk, counts, hbm_peak)}
    r64 = capi.make_problem(capi.MODEL_EXP_CURVE, capi.JAC_CENTRAL, capi.F64)
    t0 = time.perf_counter()
    r = ctx.lm_minimize([st], [r64], [0.0, 0.0], max_iterations=50)
    dt = time.perf_counter() - t0
    out["curve_10M_central"]["lm_f64"] = {"status": r.status, "iterations": r.executed_iterations, "passes": r.num_passes,
                                          "seconds": dt, "x": [float(v) for v in r.x]}
    st.close()
    # configs[4]: camera calibration, 50 M observations, numerical Jacobian; 6 extrinsics, then the n x n case (P = 15)
    n = 50_000_000
    consts = camera_consts()
    x6 = np.array([-0.01, 0.02, -0.06, 0.018, -0.0013, 0.027])
    T = capi.so3_convert6dof(x6)
    M = consts[:12].reshape(3, 4) @ T @ consts[12:].reshape(4, 4)
    st = capi.Store(ctx, capi.MODEL_PINHOLE, n, capi.F32)
    st.generate(seed=3, gt=M.reshape(-1), lo=(2.0, -1.0, -0.5), hi=(5.0, 1.0, 1.0), noise_sigma=0.5)
    prob = capi.make_problem(capi.MODEL_PINHOLE, capi.JAC_CENTRAL, capi.F32, consts=consts)
    ms = timer.ms_per_pass(st, prob, [0.0] * 6, steps=30, warm=30)
    out["camera_50M_P6_central"] = {
        "workload": "pinhole reprojection, 50M observations, 6 extrinsics, numerical central differences, fp32 (BASELINE configs[4], the reference's own test model)",
        "n": n, "ms": ms, "Gres_per_s": n / ms / 1e6,
        "roofline": alu_roofline("camera6_central_f32", n, ms, 20, pk, counts, hbm_peak)}
    st.close()
    x15 = np.concatenate([x6, [600.0, 600.0, 320.0, 240.0, 0.05, -0.02, 0.001, -0.001, 0.005]])
    C44 = consts[12:]
    st = capi.Store(ctx, capi.MODEL_PINHOLE_DISTORT, n, capi.F32)
    st.generate(seed=3, gt=x15, lo=(2.0, -1.0, -0.5), hi=(5.0, 1.0, 1.0), noise_sigma=0.5, consts=C44)
    prob = capi.make_problem(capi.MODEL_PINHOLE_DISTORT, capi.JAC_CENTRAL, capi.F32, consts=C44)
    ms = timer.ms_per_pass(st, prob, x15 * 0.999, steps=15, warm=15)
    entry = {
        "workload": "pinhole + distortion, 50M observations, 15 parameters (n x n device solve), numerical central differences, fp32 (BASELINE configs[4])",
        "n": n, "ms": ms, "Gres_per_s": n / ms / 1e6,
        "roofline": alu_roofline("camera15_central_f32", n, ms, 20, pk, counts, hbm_peak)}
    p64 = capi.make_problem(capi.MODEL_PINHOLE_DISTORT, capi.JAC_CENTRAL, capi.F64, consts=C44)
    x0 = x15.copy()
    x0[:6] = 0.0
    x0[6:10] *= 1.02
    x0[10:] = 0.0
    t0 = time.perf_counter()
    r = ctx.lm_minimize([st], [p64], x0, max_iterations=50)
    dt = time.perf_counter() - t0
    entry["lm_f64"] = {"status": r.status, "iterations": r.executed_iterations, "passes": r.num_passes, "seconds": dt,
                       "x_err_extrinsics": float(np.max(np.abs(r.x[:6] - x15[:6]))),
                       "x_err_focal_rel": float(np.max(np.abs(r.x[6:10] / x15[6:10] - 1.0)))}
    out["camera_50M_P15_central"] = entry
    st.close()
    # configs[0]: the small-problem LM — tst/point2point's cloud (29 310 points), fp64 Scalar, LM iterations per second
    try:
        src = np.fromfile(os.path.join(ROOT, "tests", "golden", "fachada_xyz.f64"), dtype="<f8").reshape(-1, 3)
        fx = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_fixtures.json")))["fachada"]
        ex, ey, ez = fx["gt_euler_xyz"]

        def rot(axis, a):
            c, s = np.cos(a), np.sin(a)
            return {"x": np.array([[1, 0, 0], [0, c, -s], [0, s, c]]), "y": np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]]),
                    "z": np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]])}[axis]
        R = rot("x", ex) @ rot("y", ey) @ rot("z", ez)
        tgt = src @ R.T + np.array(fx["gt_translation"])
        n = src.shape[0]
        st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F64)
        st.upload(0, src)
        st.upload(1, tgt)
        prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64, variant=capi.P2P_EXACT)
        ctx.lm_minimize([st], [prob], [0.0] * 6, max_iterations=50)
        times, r = [], None
        for _ in range(30):
            ctx.synchronize()
            t0 = time.perf_counter()
            r = ctx.lm_minimize([st], [prob], [0.0] * 6, max_iterations=50)
            times.append(time.perf_counter() - t0)
        dt = float(np.median(times))
        out["fachada_lm"] = {
            "workload": "tst/point2point cloud (29 310 correspondences), analytical Jacobian, fp64, LM from x0 = 0 "
                        "(BASELINE configs[0]); wall clock of mopt_lm_minimize, median of 30 solves",
            "n": n, "status": r.status, "iterations": r.executed_iterations, "passes": r.num_passes, "sequence": r.sequence,
            "seconds": dt, "lm_iters_per_s": r.executed_iterations / dt, "us_per_pass": dt / max(r.num_passes, 1) * 1e6,
            "roofline": {"bound": "latency", "note": "launch- and dependency-bound: a pass over 0.7 MB takes microseconds; "
                                                     "the figure of merit is microseconds per pass + optimizer step"}}
        st.close()
    except Exception as e:  # the fixture travels with the repo; never fail the headline line over it
        out["fachada_lm"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from moptimizer_0_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the CUDA path is the only implementation (no CPU fallback)")
    torch.cuda.set_device(local)
    numa_note = bind_host_thread(local, local, local_world) if world > 1 else "not bound (single rank)"
    from moptimizer_0_b200 import sharding
    collective, collective_note = "none", ""
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        ctx, collective, collective_note = sharding.make_sharded_context(local, rank, world, args.collective)
    else:
        ctx = capi.Context(local)
    if args.ctas_per_sm or args.threads:
        ctx.set_launch(args.ctas_per_sm, args.threads)
    n, first, n_total = args.n, rank * args.n, args.n * world
    store = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    store.generate(seed=SEED, gt=X_GT, first_index=first, **GEN)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32, loss=capi.LOSS_HUBER,
                             loss_param=HUBER_K, variant=capi.P2P_EXACT)
    x0 = np.zeros(6, dtype=np.float64)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.synchronize()

    def timed_steps(st, steps):
        """K lock-step passes between two events on the context's stream; max over ranks, ms per step."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            ctx.linearize_async(st, prob, x0)
        e1.record(stream)
        barrier()
        mine = e0.elapsed_time(e1)
        t = torch.tensor([mine], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps, mine / steps

    # Untimed pre-warm: the B200's clocks/power state take a few hundred ms of load to settle (measured:
    # the same kernel moves between 347 and 380 us during the first ~0.3 s), so a 20 ms timed region right
    # after an idle GPU does not measure the sustained rate.  Fixed step count => identical on every rank.
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.prewarm_steps):
        ctx.linearize_async(store, prob, x0)
    for _ in range(max(args.warmup, 3)):
        ctx.linearize_async(store, prob, x0)
    barrier()
    sampler.mark()
    ms_step, ms_mine = timed_steps(store, args.steps)
    sampler.mark()
    sampler.stop()
    H, b, s = ctx.result(6)
    if rank == 0 and args.dump_outputs:  # every rank holds the same exchanged result
        dump_outputs(args.dump_outputs, H, b, s)
    # diagnostics for N > 1: every rank's own pass time with the exchange switched off (no lock-step coupling);
    # the gap between max(local) and the coupled step is what the collective + straggling cost
    local_ms = None
    if world > 1:
        ctx.set_exchange_enabled(False)
        _, mine = timed_steps(store, args.steps)
        ctx.set_exchange_enabled(True)
        mt = torch.tensor([mine], dtype=torch.float64, device="cuda")
        allv = [torch.zeros_like(mt) for _ in range(world)]
        dist.all_gather(allv, mt)
        local_ms = [float(v.item()) for v in allv]
    value = n_total / (ms_step * 1e-3) / 1e9
    peak, peak_kind = peaks()
    achieved = BYTES_PER_RES * n / (ms_mine * 1e-3) / 1e9  # this rank's kernel, GB/s

    # ---- N > 1: the exchanged result against every shard recomputed on ONE GPU (rank 0's) -------------------
    vs_single = None
    if world > 1 and not args.no_check:
        barrier()
        if rank == 0:
            solo = capi.Context(local)  # a plain single-GPU context: no exchange, no peers
            if args.ctas_per_sm or args.threads:
                solo.set_launch(args.ctas_per_sm, args.threads)
            tmp = capi.Store(solo, capi.MODEL_POINT2POINT, n, capi.F32)
            tot = np.zeros(28)
            for r_ in range(world):  # the exchange sums the ranks' slots in rank order, starting from 0.0
                tmp.generate(seed=SEED, gt=X_GT, first_index=r_ * n, **GEN)
                Hr, br, sr = solo.linearize(tmp, prob, x0)
                tot = tot + sharding.pack(Hr, br, sr)
            got = sharding.pack(H, b, s)
            Hs, bs, ss = sharding.unpack(tot, 6)
            vs_single = {"H_rel": float(np.max(np.abs(H - Hs)) / np.max(np.abs(Hs))),
                         "b_rel": float(np.max(np.abs(b - bs)) / np.max(np.abs(bs))),
                         "sum_rel": float(abs(s - ss) / abs(ss)), "bit_identical": bool(np.array_equal(got, tot)),
                         "how": f"rank 0 regenerated all {world} shards on its own GPU with a single-GPU context, "
                                "linearized each and added the packed results in rank order"}
            tmp.close()
            solo.close()
        barrier()

    # ---- measured ceilings of this box ----------------------------------------------------------------------
    pk = None
    pk_rates = None  # every rank's concurrent pinned host->device rate, known to every rank
    if not args.no_peaks:
        pk = ctx.measure_peaks() if rank == 0 else None
        barrier()
        h2d = ctx.measure_h2d(1 << 30, 1.0)  # every rank at the same time: the N-way concurrent ceiling
        ht = torch.tensor([h2d], dtype=torch.float64, device="cuda")
        if world > 1:
            allh = [torch.zeros_like(ht) for _ in range(world)]
            dist.all_gather(allh, ht)
            h2d_all = [float(v.item()) for v in allh]
        else:
            h2d_all = [h2d]
        pk_rates = h2d_all
        if rank == 0:
            pk["h2d_pinned_gbs_per_rank"] = h2d_all
            pk["h2d_pinned_gbs_total"] = float(sum(h2d_all))
            pk["how"] = ("csrc/mopt_peaks.cu micro-kernels on rank 0's GPU: 8 independent FFMA / FFMA2 chains per thread, "
                         "2048 threads per SM; 2 GiB read-only stream; pinned host->device copies of 1 GiB in 64 MB "
                         "cudaMemcpyAsync chunks for >= 1 s on all ranks at once")

    # ---- e2e: host (pinned) AoS buffers -> upload -> linearize -> H, b back, every step -------------
    e2e = None
    if not args.no_e2e:
        ha = torch.empty((n, 3), dtype=torch.float32, pin_memory=True)
        hb = torch.empty((n, 3), dtype=torch.float32, pin_memory=True)
        ha.numpy()[:] = store.download(0, np.float32)
        hb.numpy()[:] = store.download(1, np.float32)
        e_store = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
        ctx.upload_and_linearize(e_store, prob, ha.numpy(), hb.numpy(), x0)  # warm-up (allocates staging)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            He, be, se = ctx.upload_and_linearize(e_store, prob, ha.numpy(), hb.numpy(), x0)
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        e2e = {"host_affinity": numa_note, "value": n_total * args.e2e_steps / dt / 1e9, "unit": UNIT,
               "h2d_bytes_per_step": int(BYTES_PER_RES * n), "d2h_bytes_per_step": 8 * 28,
               "steps": args.e2e_steps, "ms_per_step": dt / args.e2e_steps * 1e3,
               "h2d_gbs_total": BYTES_PER_RES * n_total * args.e2e_steps / dt / 1e9,
               "matches_resident": bool(np.array_equal(He, H) and np.array_equal(be, b) and se == s)}
        if pk is not None:
            # two ceilings, both measured in this run with every rank copying at once: the sum of the ranks' rates, and
            # what equal shards can reach (every rank moves the same bytes, so the slowest link sets the step time)
            rates = pk["h2d_pinned_gbs_per_rank"]
            e2e["h2d_ceiling_gbs_total"] = pk["h2d_pinned_gbs_total"]
            e2e["frac_of_h2d_ceiling"] = e2e["h2d_gbs_total"] / pk["h2d_pinned_gbs_total"]
            e2e["h2d_ceiling_gbs_equal_shards"] = world * min(rates)
            e2e["frac_of_h2d_ceiling_equal_shards"] = e2e["h2d_gbs_total"] / (world * min(rates))
        e_store.close()
        del ha, hb
        # ---- N > 1, unequal host links: shards in proportion to each rank's measured copy rate -----------------
        # (8-GPU boxes of this pool give GPUs 0-3 about 22 GB/s and GPUs 4-7 about 38 GB/s when all copy at once:
        # with equal shards the step ends with the slowest link.)  Same rows in total, same exchange, one more leg.
        if world > 1 and pk_rates is not None and max(pk_rates) > args.e2e_balance_threshold * min(pk_rates):
            tot_rate = float(sum(pk_rates))
            bounds = [0]
            for r_ in range(world):
                nxt = n_total if r_ == world - 1 else min(n_total, bounds[-1] + int(n_total * pk_rates[r_] / tot_rate) // 64 * 64)
                bounds.append(nxt)
            my0, my1 = bounds[rank], bounds[rank + 1]
            nb = my1 - my0
            b_store = capi.Store(ctx, capi.MODEL_POINT2POINT, nb, capi.F32)
            b_store.generate(seed=SEED, gt=X_GT, first_index=my0, **GEN)  # the same global rows, cut differently
            ha = torch.empty((nb, 3), dtype=torch.float32, pin_memory=True)
            hb = torch.empty((nb, 3), dtype=torch.float32, pin_memory=True)
            ha.numpy()[:] = b_store.download(0, np.float32)
            hb.numpy()[:] = b_store.download(1, np.float32)
            ctx.upload_and_linearize(b_store, prob, ha.numpy(), hb.numpy(), x0)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                Hb, bb, sb = ctx.upload_and_linearize(b_store, prob, ha.numpy(), hb.numpy(), x0)
            barrier()
            dtb = time.perf_counter() - t0
            tt = torch.tensor([dtb], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dtb = float(tt.item())
            bal = {"value": n_total * args.e2e_steps / dtb / 1e9, "unit": UNIT, "ms_per_step": dtb / args.e2e_steps * 1e3,
                   "rows_per_rank": [bounds[i + 1] - bounds[i] for i in range(world)],
                   "h2d_gbs_total": BYTES_PER_RES * n_total * args.e2e_steps / dtb / 1e9,
                   "frac_of_h2d_ceiling": BYTES_PER_RES * n_total * args.e2e_steps / dtb / 1e9 / tot_rate,
                   "H_rel_vs_equal_shards": float(np.max(np.abs(Hb - H)) / np.max(np.abs(H))),
                   "sum_rel_vs_equal_shards": float(abs(sb - s) / abs(s)),
                   "how": "the same N x n rows, rank r takes a contiguous range proportional to its measured pinned "
                          "host->device rate (peaks.h2d_pinned_gbs_per_rank); same exchange of the packed result"}
            e2e["equal_shards"] = {k: e2e[k] for k in ("value", "ms_per_step", "h2d_gbs_total", "h2d_bytes_per_step")}
            e2e["balanced_shards"] = bal
            if bal["value"] > e2e["value"]:  # the headline is the better partition of the same rows
                e2e["value"], e2e["ms_per_step"], e2e["h2d_gbs_total"] = bal["value"], bal["ms_per_step"], bal["h2d_gbs_total"]
                e2e["h2d_bytes_per_step"] = int(BYTES_PER_RES * max(bal["rows_per_rank"]))
                e2e["frac_of_h2d_ceiling"] = bal["frac_of_h2d_ceiling"]
                e2e["partition"] = "balanced_shards"
            b_store.close()
            del ha, hb

    # ---- optional: device-resident LM solve (LM iters/s) --------------------------------------------
    lm = None
    if args.lm:
        ctx.lm_minimize([store], [prob], x0, max_iterations=2)  # untimed: first launches of the optimizer kernels
        barrier()
        t0 = time.perf_counter()
        r = ctx.lm_minimize([store], [prob], x0, max_iterations=50)
        barrier()
        dt = time.perf_counter() - t0
        lm = {"status": r.status, "executed_iterations": r.executed_iterations, "passes": r.num_passes,
              "seconds": dt, "lm_iters_per_s": (r.executed_iterations or 1) / dt, "sequence": r.sequence,
              "x_err_inf": float(np.max(np.abs(r.x - np.array(X_GT))))}

    # ---- N > 1: BASELINE configs[3] as stated — 1 B correspondences in total, strong split ------------------
    strong = None
    strong_total = args.strong_total if args.strong_total >= 0 else (1_000_000_000 if world > 1 else 0)
    if world > 1 and strong_total > 0:
        store.close()
        store = None
        f0, f1 = sharding.shard_range(strong_total, rank, world)
        sst = capi.Store(ctx, capi.MODEL_POINT2POINT, f1 - f0, capi.F32)
        sst.generate(seed=SEED, gt=X_GT, first_index=f0, **GEN)
        for _ in range(max(args.warmup, 3) + 200):
            ctx.linearize_async(sst, prob, x0)
        sms, _ = timed_steps(sst, args.steps)
        Hs_, bs_, ss_ = ctx.result(6)
        ctx.lm_minimize([sst], [prob], x0, max_iterations=2)
        barrier()
        t0 = time.perf_counter()
        r = ctx.lm_minimize([sst], [prob], x0, max_iterations=50)
        barrier()
        dt = time.perf_counter() - t0
        ach = BYTES_PER_RES * strong_total / (sms * 1e-3) / 1e9
        strong = {"workload": f"point2point {strong_total / 1e9:.0f}B correspondences in total, contiguous shards over {world} GPUs, "
                              "one exchange of 28 packed doubles per step (BASELINE configs[3])",
                  "n_total": strong_total, "n_per_gpu": f1 - f0, "scaling": "strong", "ms_per_step": sms,
                  "Gres_per_s": strong_total / (sms * 1e-3) / 1e9,
                  "roofline": {"bound": "hbm", "achieved": ach, "peak": peak * world, "unit": "GB/s",
                               "frac": ach / (peak * world), "note": "aggregate over all ranks against N x the measured copy peak"},
                  "check": {"sum_rtr": ss_, "H00": float(Hs_[0, 0])},
                  "lm": {"status": r.status, "executed_iterations": r.executed_iterations, "passes": r.num_passes,
                         "seconds": dt, "lm_iters_per_s": (r.executed_iterations or 1) / dt, "sequence": r.sequence,
                         "x_err_inf": float(np.max(np.abs(r.x - np.array(X_GT))))}}
        sst.close()

    # ---- the other BASELINE configurations (single-GPU workloads: rank 0 of an N = 1 run) ------------------------
    configs = None
    if world == 1 and not args.no_configs:
        configs = run_other_configs(capi, ctx, Timer(torch, ctx, stream), pk, peak)
    if strong is not None:
        configs = configs or {}
        configs["p2p_1B_strong"] = strong

    # ---- CPU baseline: oracle port on a bounded sample of the same data (rank 0, N=1 only) ----------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle_py as orc
        m = min(args.cpu_sample, n)
        src = store.download(0, np.float64, 0, m)
        tgt = store.download(1, np.float64, 0, m)
        v1, reps1, t1 = time_oracle(src, tgt, 1, args.cpu_seconds)
        cores = orc.hardware_concurrency() or (os.cpu_count() or 1)
        vt, repst, tt_ = time_oracle(src, tgt, cores, args.cpu_seconds / 2)
        # the reference's one multithreaded piece: parallelComputeCost (linearization.h:49-63, tst/parallel.cpp)
        pc = oracle_cost(src, tgt)
        pc.cost_threads = cores
        orc.compute_cost(pc, [0.0] * 6, parallel=True)
        t0, reps_pc = time.perf_counter(), 0
        while reps_pc < 50 and time.perf_counter() - t0 < args.cpu_seconds / 4:
            orc.compute_cost(pc, [0.0] * 6, parallel=True)
            reps_pc += 1
        t_pc = time.perf_counter() - t0
        cpu = {"value": v1, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": f"first {m} correspondences of the same synthetic set, {reps1} serial fp64 linearizations "
                         f"in {t1:.1f} s (the reference's linearization loop is single-threaded, linearization.h:142)",
               "threaded": {"value": vt, "cores": cores, "reps": repst, "seconds": tt_,
                            "note": "thread-local H/b on all host cores; the reference has no such variant"},
               "parallel_cost": {"value": m * reps_pc / t_pc / 1e9, "cores": cores, "reps": reps_pc, "seconds": t_pc,
                                 "note": "cost-only pass (sum r^T r), the reference's TBB parallel_reduce variant "
                                         "(tst/parallel.cpp) restated with std::thread"}}

    if rank == 0:
        counts = inst_counts()
        tr = counts.get("p2p_gen2_f32", {})
        traffic = tr.get("dram_bytes_per_launch") if n == 100_000_000 else None
        gen1 = args.threads == 1024
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(n, n_total),
            "impl_detail": {"store": "fp32 planar (SoA) streams, 24 B/correspondence",
                            "kernel": "first generation (register-direct loads, scalar fp32)" if gen1 else
                                      "TMA bulk-copy ring (cp.async.bulk + mbarrier) + packed fp32 (FFMA2), one CTA per SM",
                            "accumulate": "fp32 partials folded into fp64 every 64 residuals per accumulator lane",
                            "prewarm_steps": args.prewarm_steps,
                            "collective": {"none": "none",
                                           "p2p": "NVLink peer exchange of 28 x f64, pushed and reduced by the pass kernel's last CTA"
                                                  + (" (separate consumer kernel)" if os.environ.get("MOPT_PEER_CONSUMER") == "kernel" else ""),
                                           "nccl": "ncclAllReduce(28 x f64) per step"}[collective]
                                          + (f" (p2p unavailable: {collective_note})" if collective_note else "")},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic,
                         "traffic_source": (tr.get("source", "") + " — ncu --set full capture of this kernel on this workload, "
                                            "committed; not re-measured in this run") if traffic else None,
                         "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})",
                         "frac_of_read_stream": (achieved / pk["hbm_read_gbs"]) if pk else None,
                         "achieved_from": "24 B x n_per_gpu / (CUDA-event time of the K timed steps / K) on the "
                                          "context's stream; a step = this kernel alone (model->setup(x) and, for N > 1, the exchange of "
                                          "the packed result run inside it)",
                         "kernel": "p2p_moment_kernel<float,float,HUBER,QROT,...,FUSED>" if gen1 else
                                   "p2p_moment2_kernel<HUBER,QROT,...> (csrc/mopt_pass_p2p2.cuh)",
                         "algorithmic_bytes_per_launch": BYTES_PER_RES * n},
            "clocks": sampler.summary(),
            # per step: the pass kernel with setup(x) and, for N > 1, the peer exchange fused in
            # (+ the setup kernel with MOPT_FUSED_SETUP=0, + NCCL's kernel or the separate consumer kernel when selected)
            "gpu_launches": ((2 if os.environ.get("MOPT_FUSED_SETUP", "")[:1] == "0" else 1) + (1 if world > 1 and (collective == "nccl" or os.environ.get("MOPT_PEER_CONSUMER") == "kernel") else 0)) * args.steps,
            "check": {"sum_rtr": s, "H00": float(H[0, 0]), "b0": float(b[0])},
        }
        if vs_single is not None:
            line["check"]["vs_single_gpu"] = vs_single
        if local_ms is not None:
            line["per_rank_uncoupled_ms_per_step"] = local_ms
        if pk is not None:
            line["peaks"] = pk
        if e2e is not None:
            line["e2e"] = e2e
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if lm is not None:
            line["lm"] = lm
        if configs is not None:
            line["configs"] = configs
        print(json.dumps(line), flush=True)
    if store is not None:
        store.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on stdout at
    # N > 1): file descriptor 1 is pointed at stderr for the duration of the run and the line goes to the real stdout.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)
    finally:
        sys.stdout.flush()


if __name__ == "__main__":
    main()
