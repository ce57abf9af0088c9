"""n x n calibration case, 50 M observations: the tensor-core Gram kernel against the first-generation kernel and the
fp64-compute path — time per pass and error of H, b in the scale sqrt(H_ii H_jj)."""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from moptimizer_0_b200 import capi
from tests.common import camera_consts

ctx = capi.Context(0)
stream = torch.cuda.ExternalStream(ctx.stream())
n = 50_000_000
Cm = camera_consts()[12:]
x_gt = np.array([-0.01, 0.02, -0.06, 0.018, -0.0013, 0.027, 600.0, 600.0, 320.0, 240.0, 0.05, -0.02, 0.001, -0.001, 0.005])
st = capi.Store(ctx, capi.MODEL_PINHOLE_DISTORT, n, capi.F32)
st.generate(seed=3, gt=x_gt, lo=(2.0, -1.0, -0.5), hi=(5.0, 1.0, 1.0), noise_sigma=0.5, consts=Cm)
x = x_gt * (1.0 + 0.002 * np.cos(np.arange(15)))
H, b, s = ctx.linearize(st, capi.make_problem(capi.MODEL_PINHOLE_DISTORT, capi.JAC_CENTRAL, capi.F64, consts=Cm), x)
d = np.sqrt(np.diag(H))
def run(tag, threads, loss=capi.LOSS_NONE, lp=0.0):
    ctx.set_launch(0, threads)
    prob = capi.make_problem(capi.MODEL_PINHOLE_DISTORT, capi.JAC_CENTRAL, capi.F32, consts=Cm, loss=loss, loss_param=lp)
    H32, b32, s32 = ctx.linearize(st, prob, x)
    xs = np.ascontiguousarray(x)
    for _ in range(10): ctx.linearize_async(st, prob, xs)
    ctx.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(20): ctx.linearize_async(st, prob, xs)
    e1.record(stream); ctx.synchronize()
    ms = e0.elapsed_time(e1) / 20
    if loss == capi.LOSS_NONE:
        eH = np.max(np.abs(H32 - H) / np.outer(d, d)); eb = np.max(np.abs(b32 - b) / (d * np.sqrt(s)))
        print(f"{tag}: {ms:.3f} ms  H {eH:.2e} b {eb:.2e} sum {abs(s32 - s) / s:.1e}", flush=True)
    else:
        print(f"{tag}: {ms:.3f} ms (Huber)", flush=True)
    return H32, b32
run("tensor-core kernel", 0)
run("first-generation kernel", 1024)
h1, b1 = run("tensor-core kernel, Huber(2 px)", 0, capi.LOSS_HUBER, 2.0)
h2, b2 = run("first-generation kernel, Huber(2 px)", 1024, capi.LOSS_HUBER, 2.0)
dd = np.sqrt(np.diag(h2))
print("Huber: tensor-core vs first generation  H %.2e  b %.2e" % (np.max(np.abs(h1 - h2) / np.outer(dd, dd)), np.max(np.abs(b1 - b2)) / np.max(np.abs(b2))))
