"""Exp-curve fit, 10 M samples, central / forward fp32: dense_f2_kernel with the model's series-form difference quotient
against the literal form (MOPT_FLAG_GENERIC_KERNEL) — time per pass and H, b against fp64 compute with the analytical
Jacobian."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from moptimizer_0_b200 import capi

ctx = capi.Context(0)
stream = torch.cuda.ExternalStream(ctx.stream())
n = 10_000_000
st = capi.Store(ctx, capi.MODEL_EXP_CURVE, n, capi.F32)
st.generate(seed=1, gt=[0.3, 0.1], lo=(0, 0, 0), hi=(5, 0, 0), n_total=n, noise_sigma=0.2)
x = np.array([0.25, 0.15])
H, b, s = ctx.linearize(st, capi.make_problem(capi.MODEL_EXP_CURVE, capi.JAC_ANALYTICAL, capi.F64), x)
for jac, jn in ((capi.JAC_CENTRAL, "central"), (capi.JAC_FORWARD, "forward")):
    for tag, flags in (("series form", 0), ("literal form", capi.FLAG_GENERIC_KERNEL)):
        prob = capi.make_problem(capi.MODEL_EXP_CURVE, jac, capi.F32, flags=flags)
        H32, b32, s32 = ctx.linearize(st, prob, x)
        for _ in range(20): ctx.linearize_async(st, prob, x)
        ctx.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(50): ctx.linearize_async(st, prob, x)
        e1.record(stream); ctx.synchronize()
        ms = e0.elapsed_time(e1) / 50
        print(f"{jn} {tag}: {ms * 1e3:.1f} us  H {np.max(np.abs(H32 - H)) / np.max(np.abs(H)):.2e}  b {np.max(np.abs(b32 - b)) / np.max(np.abs(b)):.2e}  sum {abs(s32 - s) / s:.1e}", flush=True)
