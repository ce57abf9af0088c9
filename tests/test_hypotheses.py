"""CPU-only checks of the hypothesis-scoring ABI (mopt_score_hypotheses): MOPT_MAX_HYPOTHESES and the
mopt_eval_stats layout against the ctypes binding, the host rule behind the fp32 inlier test (csrc/mopt_hyp_rule.h:
the largest float <= thr^2) compiled with the host compiler and compared with numpy, HypothesisScores.msac, and the
shape check of Context.score_hypotheses."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "moptimizer_0_b200", "csrc")

DRIVER = r'''
#include <cstdio>
#include <cstdlib>
#include "mopt_hyp_rule.h"
// stdin: one double per line (hex float, inf or nan) -> the largest float <= it, as a hex float
int main() {
  char a[64];
  while (std::scanf("%63s", a) == 1) std::printf("%a\n", double(mopt::largest_float_le(std::strtod(a, nullptr))));
  return 0;
}
'''


def _hex(v):
    v = float(v)
    if np.isnan(v):
        return "nan"
    if np.isinf(v):
        return "inf" if v > 0 else "-inf"
    return v.hex()


@pytest.fixture(scope="module")
def rule(tmp_path_factory):
    d = tmp_path_factory.mktemp("hyp_rule")
    src, exe = d / "rule.cpp", str(d / "rule")
    src.write_text(DRIVER)
    subprocess.run(["g++", "-std=c++17", "-O2", "-I", CSRC, str(src), "-o", exe], check=True)

    def run(values):
        out = subprocess.run([exe], input="\n".join(_hex(v) for v in values) + "\n", capture_output=True, text=True,
                             check=True).stdout.split()
        return np.array([float(s) if s in ("inf", "-inf", "nan", "-nan") else float.fromhex(s) for s in out])
    return run


def expected_largest_float_le(t):
    """np.float32(t) rounds to nearest; step down once with np.nextafter when that went above t."""
    if np.isnan(t):
        return np.nan
    if t >= np.inf:
        return np.inf
    f = np.float32(min(t, float(np.finfo(np.float32).max)))
    if float(f) > t:
        f = np.nextafter(f, np.float32(-np.inf))
    return float(f)


def test_max_hypotheses_and_struct_size_match_the_binding(tmp_path):
    from moptimizer_0_b200 import capi
    c = tmp_path / "s.c"
    c.write_text('#include <stdio.h>\n#include "mopt_capi.h"\nint main(void) { printf("%zu %d\\n", '
                 'sizeof(mopt_eval_stats), (int)MOPT_MAX_HYPOTHESES); return 0; }\n')
    exe = str(tmp_path / "s")
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(c), "-o", exe], check=True)
    size, cap = map(int, subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split())
    assert size == C.sizeof(capi.EvalStats)
    assert cap == capi.MAX_HYPOTHESES == 1024


def test_largest_float_le(rule):
    f32 = np.finfo(np.float32)
    tiny_sub = float(np.nextafter(np.float32(0), np.float32(1)))  # smallest positive float subnormal
    rng = np.random.default_rng(0)
    cases = [0.0, 0.25, 1e-3, 0.5 ** 2, 0.03 ** 2, 1.0 / 3.0, 2.0 / 3.0, 1e10, 1e-30,
             tiny_sub, tiny_sub / 2, tiny_sub * 1.5, 1e-320, 5e-324, float(f32.tiny), float(f32.tiny) * (1 - 2 ** -30),
             float(f32.max), float(f32.max) * (1 + 2 ** -30), float(f32.max) * 2, 1e300, np.inf, np.nan]
    cases += list(rng.uniform(0, 100, 200)) + list(10.0 ** rng.uniform(-45, 38, 200))
    got = rule(cases)
    for t, g in zip(cases, got):
        e = expected_largest_float_le(t)
        if np.isnan(t):
            assert np.isnan(g)
            continue
        assert g == e, (t, g, e)
        assert np.float32(g) == g and g <= t  # a float, not above t ...
        if g < np.inf:  # ... and the next float up is above t
            with np.errstate(over="ignore"):
                assert float(np.nextafter(np.float32(g), np.float32(np.inf))) > t


def test_largest_float_le_is_the_fp64_test(rule):
    """For float keys e2: e2 <= f exactly when double(e2) <= thr2, f the largest float <= thr2."""
    rng = np.random.default_rng(1)
    thr2 = np.concatenate([rng.uniform(0, 1, 64), [0.0, 0.25, np.inf, float(np.finfo(np.float32).max) * 3]])
    fs = rule(thr2)
    for t, f in zip(thr2, fs):
        base = np.float32(min(t, 1.0))
        e2 = np.concatenate([
            np.array([np.nextafter(base, np.float32(0)), base, np.nextafter(base, np.float32(2)), 0.0, np.inf, np.nan],
                     dtype=np.float32),
            rng.uniform(0, 1.5, 64).astype(np.float32)])
        with np.errstate(invalid="ignore"):
            assert np.array_equal(e2 <= np.float32(f), e2.astype(np.float64) <= t), t


def test_msac_matches_numpy():
    from moptimizer_0_b200 import capi
    rng = np.random.default_rng(2)
    K = 17
    raw = (capi.EvalStats * K)()
    nv = rng.integers(100, 1000, K)
    ni = (nv * rng.uniform(0, 1, K)).astype(np.int64)
    isum = rng.uniform(0, 5, K)
    for k in range(K):
        raw[k].n_valid, raw[k].n_inliers, raw[k].inlier_sum_sq = int(nv[k]), int(ni[k]), float(isum[k])
        raw[k].sum_sq, raw[k].max_sq = float(isum[k] + 7.0), 0.5
    thr = 0.03
    sc = capi.HypothesisScores(raw, thr)
    assert np.array_equal(sc.n_valid, nv) and np.array_equal(sc.n_inliers, ni)
    assert np.array_equal(sc.inlier_sum_sq, isum) and np.array_equal(sc.sum_sq, isum + 7.0)
    assert np.array_equal(sc.msac, isum + (nv - ni) * thr ** 2)
    assert sc.n_valid.shape == sc.msac.shape == (K,)


@pytest.mark.parametrize("shape", [(6,), (0, 6), (4, 5), (4, 7), (2, 3, 6)])
def test_bad_hypothesis_shape_raises_before_the_call(shape):
    from moptimizer_0_b200 import capi
    ctx = object.__new__(capi.Context)  # never reaches the library: no device needed
    prob = capi.make_problem(capi.MODEL_POINT2POINT)
    with pytest.raises(ValueError):
        capi.Context.score_hypotheses(ctx, None, prob, np.zeros(shape), 0.1)
