"""Worker of tests/test_gpu_fp32_boundaries.py (run with MOPT_FUSED_SETUP=0, which the library reads once per process):
the exact point2point data of the test at n = argv[1], linearized with the set-up kernel in front of the pass.  Prints
the bits of H, b, the sum and compute_cost per Jacobian variant."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from moptimizer_0_b200 import capi  # noqa: E402
from tests import test_gpu_fp32_boundaries as t  # noqa: E402

t.capi = capi
n = int(sys.argv[1])
ctx = capi.Context(0)
src, tgt = t.exact_p2p(n)
st = t.p2p_store(ctx, src, tgt)
out = {v: {"H": [float(x).hex() for x in H.reshape(-1)], "b": [float(x).hex() for x in b], "s": float(s).hex(),
           "c": float(c).hex()} for v, (H, b, s, c) in t.exact_results(ctx, st).items()}
st.close()
ctx.close()
print(json.dumps(out))
