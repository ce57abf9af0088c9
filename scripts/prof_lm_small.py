"""tst/point2point's cloud (29 310 points, fp64): a few device LM solves, for ncu (launch list / lm_step_kernel source
page); prints the wall time of every solve."""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from moptimizer_0_b200 import capi
from tests.common import fachada
ctx = capi.Context(0)
src, tgt, _, _ = fachada()
st = capi.Store(ctx, capi.MODEL_POINT2POINT, src.shape[0], capi.F64)
st.upload(0, src); st.upload(1, tgt)
prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64, variant=capi.P2P_EXACT)
ts = []
for _ in range(int(sys.argv[1]) if len(sys.argv) > 1 else 2):
    ctx.synchronize(); t0 = time.perf_counter()
    r = ctx.lm_minimize([st], [prob], [0.0] * 6, max_iterations=50)
    ts.append((time.perf_counter() - t0) * 1e6)
print("us per solve:", " ".join(f"{t:.0f}" for t in ts))
print(r.status, r.sequence, r.x)
