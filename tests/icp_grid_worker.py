"""Worker of tests/test_icp_grid.py: builds an index of every non-finite target cloud of the test (in both index and host
dtypes), re-associates, and saves [matched; targets downloaded] per case under argv[1].  Runs in its own process so
that a build that never returns fails the test through a timeout."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from moptimizer_0_b200 import capi  # noqa: E402
from tests import test_icp_grid as t  # noqa: E402

ctx = capi.Context(0)
for name in t.NONFINITE_CASES:
    for it in (t.F32, t.F64):
        for ht in (t.F32, t.F64):
            matched, got = t.run_nonfinite_case(capi, ctx, name, it, ht)
            head = np.full((1, 3), float(matched))
            np.save(os.path.join(sys.argv[1], f"{name}_{it}_{ht}.npy"), np.vstack([head, got]))
ctx.close()
