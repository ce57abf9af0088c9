"""Camera calibration, 6 extrinsics, 50 M observations, central / forward fp32: dense_f2_kernel against
dense_pass_kernel (set_launch(.., 1024)) — time per pass and H, b against fp64 compute."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from moptimizer_0_b200 import capi
from tests.common import camera_consts
from oracle import oracle_py as orc

ctx = capi.Context(0)
stream = torch.cuda.ExternalStream(ctx.stream())
n = 50_000_000
consts = camera_consts()
x_gt = np.array([-0.01, 0.02, -0.06, 0.018, -0.0013, 0.027])
M = consts[:12].reshape(3, 4) @ orc.so3_convert6dof(x_gt) @ consts[12:].reshape(4, 4)
st = capi.Store(ctx, capi.MODEL_PINHOLE, n, capi.F32)
st.generate(seed=3, gt=M.reshape(-1), lo=(2.0, -1.0, -0.5), hi=(5.0, 1.0, 1.0), noise_sigma=0.5)
x = np.array([0.01, -0.01, 0.02, 0.005, 0.003, -0.004])
for jac, jn in ((capi.JAC_CENTRAL, "central"), (capi.JAC_FORWARD, "forward")):
    H, b, s = ctx.linearize(st, capi.make_problem(capi.MODEL_PINHOLE, jac, capi.F64, consts=consts, flags=capi.FLAG_STABLE_FD), x)
    for tag, threads in (("dense_f2", 0), ("dense_pass", 1024)):
        ctx.set_launch(0, threads)
        prob = capi.make_problem(capi.MODEL_PINHOLE, jac, capi.F32, consts=consts)
        H32, b32, s32 = ctx.linearize(st, prob, x)
        xs = np.ascontiguousarray(x)
        for _ in range(20): ctx.linearize_async(st, prob, xs)
        ctx.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(30): ctx.linearize_async(st, prob, xs)
        e1.record(stream); ctx.synchronize()
        ms = e0.elapsed_time(e1) / 30
        print(f"{jn} {tag}: {ms:.3f} ms  H {np.max(np.abs(H32 - H)) / np.max(np.abs(H)):.2e}  b {np.max(np.abs(b32 - b)) / np.max(np.abs(b)):.2e}  sum {abs(s32 - s) / s:.1e}", flush=True)
