"""CPU-only checks of the residual-quantile ABI (mopt_residual_quantiles): the mopt_quantiles layout and
MOPT_MAX_QUANTILES against the ctypes binding, and the host rule the library uses (csrc/mopt_quant_rule.h:
numpy's method="linear" ranks and interpolation, the chi-square medians of the robust scale) compiled with the host
compiler and compared with numpy and scipy."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "moptimizer_0_b200", "csrc")

DRIVER = r'''
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "mopt_quant_rule.h"
// stdin: "R n q" -> "j j1 t" (quantile_rank), "L lo hi t" -> "v" (quantile_lerp), "C dof" -> "m" (chi2_median)
int main() {
  char op[4], a[64], b[64], c[64];
  while (std::scanf("%3s", op) == 1) {
    if (op[0] == 'R' && std::scanf("%63s %63s", a, b) == 2) {
      const mopt::QuantRank r = mopt::quantile_rank(std::strtoll(a, nullptr, 10), std::strtod(b, nullptr));
      std::printf("%lld %lld %a\n", (long long)r.j, (long long)r.j1, r.t);
    } else if (op[0] == 'L' && std::scanf("%63s %63s %63s", a, b, c) == 3) {
      std::printf("%a\n", mopt::quantile_lerp(std::strtod(a, nullptr), std::strtod(b, nullptr), std::strtod(c, nullptr)));
    } else if (op[0] == 'C' && std::scanf("%63s", a) == 1) {
      std::printf("%a\n", mopt::chi2_median(std::atoi(a)));
    }
  }
  return 0;
}
'''


@pytest.fixture(scope="module")
def rule(tmp_path_factory):
    d = tmp_path_factory.mktemp("quant_rule")
    src, exe = d / "rule.cpp", str(d / "rule")
    src.write_text(DRIVER)
    subprocess.run(["g++", "-std=c++17", "-O2", "-I", CSRC, str(src), "-o", exe], check=True)

    def run(lines):
        out = subprocess.run([exe], input="\n".join(lines) + "\n", capture_output=True, text=True, check=True).stdout
        return out.split("\n")[:len(lines)]
    return run


def _hex(v):
    v = float(v)
    if np.isnan(v):
        return "nan"
    if np.isinf(v):
        return "inf" if v > 0 else "-inf"
    return v.hex()


def _unhex(s):
    return float.fromhex(s) if s not in ("inf", "-inf", "nan", "-nan") else float(s.replace("-nan", "nan"))


def library_quantiles(rule, e_sorted, qs):
    """lo, hi, value as mopt_residual_quantiles forms them from the order statistics of e."""
    n = len(e_sorted)
    ranks = [r.split() for r in rule([f"R {n} {_hex(q)}" for q in qs])]
    lo = np.array([e_sorted[int(r[0])] for r in ranks])
    hi = np.array([e_sorted[int(r[1])] for r in ranks])
    t = np.array([_unhex(r[2]) for r in ranks])
    vals = np.array([_unhex(v) for v in rule([f"L {_hex(a)} {_hex(b)} {_hex(c)}" for a, b, c in zip(lo, hi, t)])])
    return lo, hi, t, vals


def test_struct_size_and_max_quantiles_match_the_binding(tmp_path):
    import ctypes
    from moptimizer_0_b200 import capi
    c = tmp_path / "s.c"
    c.write_text('#include <stdio.h>\n#include "mopt_capi.h"\nint main(void) { printf("%zu %d\\n", '
                 'sizeof(mopt_quantiles), (int)MOPT_MAX_QUANTILES); return 0; }\n')
    exe = str(tmp_path / "s")
    subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(c),
                    "-o", exe], check=True)
    size, mq = (int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split())
    assert size == ctypes.sizeof(capi.QuantilesStruct) == 8 * (2 + 3 * mq + 2 + 4)
    assert mq == capi.MAX_QUANTILES


def test_chi2_medians_match_scipy(rule):
    from scipy.stats import chi2
    got = [_unhex(v) for v in rule([f"C {k}" for k in (1, 2, 3, 4)])]
    for k, m in zip((1, 2, 3, 4), got):
        assert m == pytest.approx(chi2.median(k), rel=1e-14), k
    assert got[1] == pytest.approx(2 * np.log(2), rel=1e-15)
    # O = 1: sqrt(median r^2 / m_1) = 1.4826 median |r|
    assert 1.0 / np.sqrt(got[0]) == pytest.approx(1.4826, abs=1e-4)


QS = np.array([0.0, 0.1, 0.25, 0.5, 0.5 + 1e-12, 0.9, 0.99, 0.999, 1.0, 1 / 3, 2 / 3, 0.7, 0.3])


@pytest.mark.parametrize("kind", ["uniform", "lognormal", "ties", "zeros", "inf", "all_inf", "fp32"])
@pytest.mark.parametrize("n", [1, 2, 3, 31, 1000, 100_003])
def test_host_rule_matches_numpy(rule, kind, n):
    rng = np.random.default_rng(n)
    if kind == "uniform":
        e = rng.uniform(0, 1, n)
    elif kind == "lognormal":
        e = rng.lognormal(0, 4, n)
    elif kind == "ties":
        e = rng.integers(0, 4, n).astype(np.float64) * 0.25
    elif kind == "zeros":
        e = np.where(rng.random(n) < 0.9, 0.0, rng.uniform(0, 1, n))
    elif kind == "inf":
        e = np.where(rng.random(n) < 0.2, np.inf, rng.uniform(0, 1, n))
        e[-1] = np.inf
    elif kind == "all_inf":
        e = np.full(n, np.inf)
    else:
        e = rng.uniform(0, 10, n).astype(np.float32).astype(np.float64)
    es = np.sort(e)
    lo, hi, t, vals = library_quantiles(rule, es, QS)
    with np.errstate(invalid="ignore"):
        ref = np.quantile(e, QS)
    # the order statistics np.quantile interpolates between
    h = (n - 1) * QS
    j = np.floor(h).astype(np.int64)
    assert np.array_equal(lo, es[j]) and np.array_equal(hi, es[np.minimum(j + 1, n - 1)])
    assert np.array_equal(t, h - j)
    # numpy's value, bit for bit (NaN where numpy gives NaN), except value = lo where t = 0
    exact = t == 0
    assert np.array_equal(vals[exact], lo[exact])
    assert np.array_equal(vals[~exact], ref[~exact], equal_nan=True)
    assert np.array_equal(vals[exact & np.isfinite(ref)], ref[exact & np.isfinite(ref)])
