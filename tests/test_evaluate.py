"""Per-residual evaluation, CPU side: the mopt_eval_stats ABI mirror, and the oracle's per-element loop
(tests/oracle_evaluate.cpp: the reference's computeCost loop with each element kept) against a numpy restatement."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_py as orc
from tests import oracle_evaluate as oev
from tests.common import curve_cost

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_eval_stats_size_matches_ctypes_mirror(tmp_path):
    from moptimizer_0_b200 import capi
    c = tmp_path / "s.c"
    c.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mopt_capi.h"\nint main(void) { printf("%zu %zu %zu\\n", '
                 "sizeof(mopt_eval_stats), offsetof(mopt_eval_stats, sum_sq), offsetof(mopt_eval_stats, max_sq)); "
                 "return 0; }\n")
    exe = str(tmp_path / "s")
    subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(c),
                    "-o", exe], check=True)
    size, off_sum, off_max = [int(v) for v in subprocess.run([exe], capture_output=True, text=True,
                                                             check=True).stdout.split()]
    assert size == ctypes.sizeof(capi.EvalStats) == 64
    assert off_sum == capi.EvalStats.sum_sq.offset and off_max == capi.EvalStats.max_sq.offset


def np_weight(loss, k, e2):
    if loss == orc.LOSS_NONE:
        return np.ones_like(e2)
    if loss == orc.LOSS_GM:
        return (k * k) / ((e2 + k) * (e2 + k))
    return np.where(e2 <= k * k, 1.0, k / np.sqrt(e2))


@pytest.mark.parametrize("loss,k", [(orc.LOSS_NONE, 0.0), (orc.LOSS_GM, 0.02), (orc.LOSS_HUBER, 0.05)])
def test_oracle_evaluate_point2point_matches_numpy(loss, k):
    rng = np.random.default_rng(1)
    n = 1001
    src = rng.uniform(0, 10, (n, 3))
    x = np.array([0.5, -0.3, 0.2, 0.1, -0.05, 0.08])
    T = orc.so3_convert6dof(x)
    tgt = src @ T[:3, :3].T + T[:3, 3] + rng.normal(0, 0.05, (n, 3))
    cost = orc.Cost(orc.P2P, 6, 3, n, a=src, b=tgt, jac_mode=orc.JAC_ANALYTICAL, loss=loss, loss_param=k)
    r, w, valid = oev.evaluate(cost, x)
    r_np = src @ T[:3, :3].T + T[:3, 3] - tgt
    assert valid.all()
    assert np.max(np.abs(r - r_np)) <= 1e-14 * np.max(np.abs(tgt))
    # the weight is the loss of the element's own r^T r (a 1e-15 change of a 0.05 residual moves e2 by 1e-13 relative)
    assert np.max(np.abs(w - np_weight(loss, k, np.sum(r ** 2, axis=1)))) <= 1e-14
    # a sub-range is the same elements
    r2, w2, _ = oev.evaluate(cost, x, first=100, count=37)
    assert np.array_equal(r2, r[100:137]) and np.array_equal(w2, w[100:137])
    # its statistics: sum r^T r is computeCost's value
    st = oev.eval_stats(r, valid)
    assert st["n_valid"] == n and st["sum_sq"] == pytest.approx(orc.compute_cost(cost, x, parallel=False), rel=1e-14)


def test_oracle_evaluate_exp_curve_matches_numpy():
    cost = curve_cost(loss=orc.LOSS_HUBER, loss_param=0.2)
    x = [0.3, 0.1]
    r, w, valid = oev.evaluate(cost, x)
    r_np = cost.b - np.exp(x[0] * cost.a + x[1])
    assert valid.all() and r.shape == (cost.n, 1)
    assert np.max(np.abs(r[:, 0] - r_np)) <= 1e-14 * np.max(np.abs(cost.b))
    assert np.max(np.abs(w - np_weight(orc.LOSS_HUBER, 0.2, r[:, 0] ** 2))) <= 1e-14
    st = oev.eval_stats(r, valid, inlier_threshold=0.2)
    inl = r_np ** 2 <= 0.04
    assert st["n_inliers"] == int(inl.sum()) and st["inlier_sum_sq"] == pytest.approx(np.sum(r_np[inl] ** 2), rel=1e-14)
    assert st["max_sq"] == pytest.approx(np.max(r_np ** 2), rel=1e-14)


def test_oracle_evaluate_marks_unmatched_icp_elements():
    from tests.test_icp import X_TRUE, clouds, icp_cost
    src, tgt = clouds()
    r, w, valid = oev.evaluate(icp_cost(src, tgt), X_TRUE)
    assert 0 < valid.sum() < src.shape[0]
    assert np.isnan(r[~valid]).all() and not np.isnan(r[valid]).any() and (w[~valid] == 0).all()
