"""Closed-form rigid alignment, CPU side: the mopt_align_moments / mopt_align_report ABI mirrors, Horn's solve
(mopt_align_from_terms, host only) against a weighted fp64 SVD Kabsch, and the pairwise merge
(mopt_align_terms_merge) against one-shot centred moments, with terms built in numpy."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def capi():
    from moptimizer_0_b200 import build
    build.build()
    from moptimizer_0_b200 import capi as c
    return c


def terms_of(capi, p, q, w=None, n_valid=None):
    """Centred moments of the pairs (p_i, q_i) with weights w, as mopt_align_terms defines them."""
    p, q = np.asarray(p, dtype=np.float64), np.asarray(q, dtype=np.float64)
    w = np.ones(len(p)) if w is None else np.asarray(w, dtype=np.float64)
    t = capi.AlignMomentsStruct()
    t.n_used = len(p)
    t.n_valid = len(p) if n_valid is None else n_valid
    W = float(np.sum(w))
    t.w = W
    if W > 0:
        ms, mt = w @ p / W, w @ q / W
        ms, mt = ms + w @ (p - ms) / W, mt + w @ (q - mt) / W  # a second pass: the means to rounding far from 0
        dp, dq = p - ms, q - mt
        np.ctypeslib.as_array(t.mean_src)[:] = ms
        np.ctypeslib.as_array(t.mean_tgt)[:] = mt
        np.ctypeslib.as_array(t.cross)[:] = ((w[:, None] * dp).T @ dq).reshape(-1)
        t.var_src, t.var_tgt = float(np.sum(w * np.sum(dp * dp, 1))), float(np.sum(w * np.sum(dq * dq, 1)))
    return capi.AlignTerms(t)


def kabsch(p, q, w=None):
    """R, t minimising sum w |R p + t - q|^2: weighted SVD with the determinant fix-up."""
    w = np.ones(len(p)) if w is None else w
    W = np.sum(w)
    pc, qc = w @ p / W, w @ q / W
    pc, qc = pc + w @ (p - pc) / W, qc + w @ (q - qc) / W
    U, _, Vt = np.linalg.svd((w[:, None] * (p - pc)).T @ (q - qc))
    R = Vt.T @ np.diag([1.0, 1.0, np.sign(np.linalg.det(Vt.T @ U.T))]) @ U.T
    return R, qc - R @ pc


def solve(capi, p, q, w=None):
    a = capi.align_from_terms(terms_of(capi, p, q, w))
    return a, Rotation.from_rotvec(a.x[3:]).as_matrix(), a.x[:3]


def test_structs_match_ctypes_mirrors(tmp_path, capi):
    fields = [("mopt_align_moments", f) for f in ("n_valid", "n_used", "w", "mean_src", "mean_tgt", "cross",
                                                  "var_src", "var_tgt", "reserved")] + \
             [("mopt_align_report", f) for f in ("cost", "rms", "eig", "degenerate", "reserved")]
    c = tmp_path / "s.c"
    c.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mopt_capi.h"\nint main(void) { printf("%zu %zu'
                 + " %zu" * len(fields) + '\\n", sizeof(mopt_align_moments), sizeof(mopt_align_report), '
                 + ", ".join(f"offsetof({s}, {f})" for s, f in fields) + "); return 0; }\n")
    exe = str(tmp_path / "s")
    subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(c),
                    "-o", exe], check=True)
    vals = [int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    assert vals[0] == ctypes.sizeof(capi.AlignMomentsStruct) and vals[1] == ctypes.sizeof(capi.AlignReport)
    mirrors = {"mopt_align_moments": capi.AlignMomentsStruct, "mopt_align_report": capi.AlignReport}
    assert vals[2:] == [getattr(mirrors[s], f).offset for s, f in fields]


# ---- Horn's solve against the SVD oracle ---------------------------------------------------------------------------
def cloud(rng, n=200, spread=(3.0, 2.0, 1.0)):
    return rng.normal(0, 1, (n, 3)) * np.array(spread) + rng.uniform(-5, 5, 3)


def check_solve(capi, p, q, w=None, tol=1e-12):
    a, R, t = solve(capi, p, q, w)
    Ro, to = kabsch(p, q, w)
    assert np.max(np.abs(R - Ro)) <= tol, np.max(np.abs(R - Ro))
    assert np.max(np.abs(t - to)) <= tol * max(1.0, np.max(np.abs(to))), np.max(np.abs(t - to))
    assert np.linalg.norm(a.x[3:]) <= np.pi * (1 + 1e-15)
    assert np.linalg.det(R) == pytest.approx(1.0, abs=1e-13)
    wv = np.ones(len(p)) if w is None else w
    cost = float(np.sum(wv * np.sum((p @ Ro.T + to - q) ** 2, 1)))
    assert a.cost == pytest.approx(cost, rel=1e-9, abs=1e-12 * (a.eig[0] + 1.0))
    assert a.rms == pytest.approx(np.sqrt(a.cost / np.sum(wv)), rel=1e-15)
    assert np.all(np.diff(a.eig) <= 0) and not a.degenerate
    return a


@pytest.mark.parametrize("seed", range(8))
def test_random_rotations(capi, seed):
    rng = np.random.default_rng(seed)
    p = cloud(rng)
    R = Rotation.random(random_state=seed).as_matrix()
    q = p @ R.T + rng.uniform(-10, 10, 3) + rng.normal(0, 0.1, p.shape)
    check_solve(capi, p, q)


@pytest.mark.parametrize("angle", [0.0, 1e-12, 1e-9, 1e-6, np.pi - 1e-6, np.pi - 1e-9, np.pi])
def test_angles_near_zero_and_pi(capi, angle):
    rng = np.random.default_rng(3)
    p = cloud(rng)
    axis = rng.normal(0, 1, 3)
    axis /= np.linalg.norm(axis)
    R = Rotation.from_rotvec(angle * axis).as_matrix()
    q = p @ R.T + np.array([0.3, -0.2, 0.1])
    a = check_solve(capi, p, q)
    # noise free: R itself, whatever omega's sign convention at pi
    Rs = Rotation.from_rotvec(a.x[3:]).as_matrix()
    assert np.max(np.abs(Rs - R)) <= 1e-12


def test_weighted_points(capi):
    rng = np.random.default_rng(4)
    p = cloud(rng, 500)
    R = Rotation.random(random_state=4).as_matrix()
    q = p @ R.T + 1.0 + rng.normal(0, 0.05, p.shape)
    q[:100] += rng.uniform(-3, 3, (100, 3))  # down-weighted outliers move the weighted optimum
    w = np.where(np.arange(500) < 100, 1e-3, 1.0) * rng.uniform(0.5, 2.0, 500)
    check_solve(capi, p, q, w)
    _, R1, _ = solve(capi, p, q, w)
    _, R2, _ = solve(capi, p, q)
    assert np.max(np.abs(R1 - R2)) > 1e-6  # the weights matter


def test_reflection_gives_the_proper_rotation(capi):
    rng = np.random.default_rng(5)
    p = cloud(rng, 300)
    q = p @ np.diag([1.0, 1.0, -1.0]) + rng.normal(0, 0.01, p.shape)  # a mirror image: the plain SVD has det < 0
    pc, qc = p - p.mean(0), q - q.mean(0)
    U, _, Vt = np.linalg.svd(pc.T @ qc)
    assert np.linalg.det(Vt.T @ U.T) < 0
    check_solve(capi, p, q)


def test_degenerate_configurations(capi):
    rng = np.random.default_rng(6)
    s = rng.uniform(-2, 2, 50)
    d = np.array([1.0, 2.0, -0.5])
    p = np.outer(s, d) + 1.0                     # collinear
    R = Rotation.from_rotvec([0.1, 0.2, -0.3]).as_matrix()
    a = capi.align_from_terms(terms_of(capi, p, p @ R.T + 0.5))
    assert a.degenerate
    Rs = Rotation.from_rotvec(a.x[3:]).as_matrix()
    assert np.max(np.abs(p @ Rs.T + a.x[:3] - (p @ R.T + 0.5))) <= 1e-12  # one of the minimisers
    assert capi.align_from_terms(terms_of(capi, p[:1], p[:1] + 1.0)).degenerate  # one point


def test_invalid_terms_write_nothing(capi):
    rng = np.random.default_rng(7)
    p = cloud(rng, 20)
    good = terms_of(capi, p, p + 1.0)
    x = np.full(6, -7.25)
    rep = capi.AlignReport()
    rep.cost = -3.0
    sentinel = (x.tobytes(), bytes(rep))

    def call(t):
        return capi.lib().mopt_align_from_terms(ctypes.byref(t.raw), capi._dp(x), ctypes.byref(rep))

    bad = []
    for field, v in (("w", 0.0), ("w", -1.0), ("w", np.nan), ("var_src", np.inf), ("var_tgt", np.nan)):
        t = terms_of(capi, p, p + 1.0)
        setattr(t.raw, field, v)
        bad.append(t)
    for arr in ("mean_src", "mean_tgt", "cross"):
        t = terms_of(capi, p, p + 1.0)
        getattr(t.raw, arr)[1] = np.nan
        bad.append(t)
    bad.append(terms_of(capi, p, p, w=np.zeros(len(p))))
    for t in bad:
        assert call(t) == 1  # MOPT_ERR_INVALID_ARGUMENT
        assert (x.tobytes(), bytes(rep)) == sentinel
    assert capi.lib().mopt_align_from_terms(ctypes.byref(good.raw), None, None) == 1
    assert capi.lib().mopt_align_from_terms(ctypes.byref(good.raw), capi._dp(x), None) == 0  # report may be NULL
    assert np.allclose(x, [1, 1, 1, 0, 0, 0], atol=1e-12)


# ---- the merge ---------------------------------------------------------------------------------------------------
FIELDS = ("w", "mean_src", "mean_tgt", "cross", "var_src", "var_tgt")


def as_vec(t):
    return np.concatenate([np.atleast_1d(np.asarray(getattr(t, f), dtype=np.float64)).ravel() for f in FIELDS])


def assert_moments_close(a, b, rel):
    assert a.n_valid == b.n_valid and a.n_used == b.n_used
    assert a.w == pytest.approx(b.w, rel=rel)
    for f in ("mean_src", "mean_tgt"):
        assert np.max(np.abs(getattr(a, f) - getattr(b, f))) <= rel * np.max(np.abs(getattr(b, f))), f
    scale = max(b.var_src, b.var_tgt)
    for f in ("cross", "var_src", "var_tgt"):
        assert np.max(np.abs(np.asarray(getattr(a, f)) - np.asarray(getattr(b, f)))) <= rel * scale, f


def chunks(rng, n, k):
    cuts = np.sort(rng.choice(np.arange(1, n), k - 1, replace=False)) if k > 1 else []
    return np.split(np.arange(n), cuts)


def test_merge_is_bitwise_commutative_and_may_alias(capi):
    rng = np.random.default_rng(8)
    for trial in range(50):
        n1, n2 = rng.integers(1, 40, 2)
        off = 10.0 ** rng.uniform(-3, 6)
        a = terms_of(capi, cloud(rng, n1) + off, cloud(rng, n1), rng.uniform(0, 3, n1), n_valid=n1 + 3)
        b = terms_of(capi, cloud(rng, n2) * 0.1, cloud(rng, n2) - off, rng.uniform(0, 3, n2))
        ab, ba = a + b, b + a
        assert bytes(ab.raw) == bytes(ba.raw), trial
        assert ab.n_valid == n1 + n2 + 3 and ab.n_used == n1 + n2
        out = capi.AlignMomentsStruct()
        ctypes.memmove(ctypes.addressof(out), ctypes.addressof(a.raw), ctypes.sizeof(out))
        capi.check(capi.lib().mopt_align_terms_merge(ctypes.byref(out), ctypes.byref(b.raw), ctypes.byref(out)))
        assert bytes(out) == bytes(ab.raw)
        capi.check(capi.lib().mopt_align_terms_merge(ctypes.byref(a.raw), ctypes.byref(out), ctypes.byref(out)))
        assert bytes(out) == bytes((a + ab).raw)


def test_merge_with_zero_weight_is_the_identity(capi):
    rng = np.random.default_rng(9)
    a = terms_of(capi, cloud(rng, 30), cloud(rng, 30), rng.uniform(0, 2, 30))
    empty = capi.AlignTerms()
    empty.raw.n_valid, empty.raw.n_used = 5, 2   # elements that entered with weight 0 (or no element at all)
    for m in (a + empty, empty + a):
        assert as_vec(m).tobytes() == as_vec(a).tobytes()
        assert m.n_valid == a.n_valid + 5 and m.n_used == a.n_used + 2
    z = empty + empty
    assert z.n_valid == 10 and not np.any(as_vec(z))


# The merged means are fp64 values: 1e6 from the origin each carries up to half an ulp (6e-11) of rounding relative to
# the unit spread, which enters the next merge's correction term f d_src d_tgt^T at first order.  Measured over these
# folds: at most 5e-12 of the largest moment (8e-12 over 63 merges of ten other clouds), against 1e-15 at the
# origin and more than 1e-6 for raw sums.  mopt_capi.h states the same for mopt_align_terms_merge.
@pytest.mark.parametrize("offset,rel", [(0.0, 1e-12), (1e6, 2e-11)])
def test_folding_chunks_matches_one_shot(capi, offset, rel):
    rng = np.random.default_rng(10)
    n = 4000
    p = rng.normal(0, 1, (n, 3)) + offset
    R = Rotation.random(random_state=10).as_matrix()
    q = p @ R.T + rng.normal(0, 0.01, (n, 3)) + 2.0
    w = rng.uniform(0.1, 1.0, n)
    one = terms_of(capi, p, q, w)
    for k in (1, 2, 3, 7, 16, 33, 64):
        parts = [terms_of(capi, p[i], q[i], w[i]) for i in chunks(rng, n, k)]
        acc = parts[0]
        for t in parts[1:]:
            acc = acc + t
        assert_moments_close(acc, one, rel)
    # raw sums over the same cloud (sum w p q^T - W mean_p mean_q^T) would miss the cross term by far more
    W = np.sum(w)
    raw = (w[:, None] * p).T @ q - W * np.outer(w @ p / W, w @ q / W)
    err = np.max(np.abs(raw - one.cross)) / max(one.var_src, one.var_tgt)
    if offset:
        assert err > 1e-6, err
    a = capi.align_from_terms(acc)
    Ro, to = kabsch(p, q, w)
    assert np.max(np.abs(Rotation.from_rotvec(a.x[3:]).as_matrix() - Ro)) <= 1e-10
    assert np.max(np.abs(a.x[:3] - to)) <= 1e-8 * max(1.0, offset)
