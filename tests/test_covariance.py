"""Parameter covariance, CPU side: the mopt_cov_terms / mopt_cov_report ABI mirrors, the test oracle's score Gram
loop (tests/oracle_covariance.cpp) against numpy, and mopt_covariance_from_terms (host only) against numpy and
scipy.optimize.curve_fit."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_py as orc
from tests import oracle_covariance as ocov
from tests.common import curve_cost

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def capi():
    from moptimizer_0_b200 import build
    build.build()
    from moptimizer_0_b200 import capi as c
    return c


def test_cov_structs_match_ctypes_mirrors(tmp_path, capi):
    fields = [("mopt_cov_terms", f) for f in ("n_valid", "m", "H", "G", "b", "wsse", "sum_sq")] + \
             [("mopt_cov_report", f) for f in ("dof", "sigma2", "eig_min", "eig_max")]
    c = tmp_path / "s.c"
    c.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mopt_capi.h"\nint main(void) { printf("%zu %zu'
                 + " %zu" * len(fields) + '\\n", sizeof(mopt_cov_terms), sizeof(mopt_cov_report), '
                 + ", ".join(f"offsetof({s}, {f})" for s, f in fields) + "); return 0; }\n")
    exe = str(tmp_path / "s")
    subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(c),
                    "-o", exe], check=True)
    vals = [int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    assert vals[0] == ctypes.sizeof(capi.CovTermsStruct) and vals[1] == ctypes.sizeof(capi.CovReport)
    mirrors = {"mopt_cov_terms": capi.CovTermsStruct, "mopt_cov_report": capi.CovReport}
    assert vals[2:] == [getattr(mirrors[s], f).offset for s, f in fields]


def hat(v):
    return np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])


def np_weight(loss, k, e2):
    if loss == orc.LOSS_NONE:
        return np.ones_like(e2)
    if loss == orc.LOSS_GM:
        return (k * k) / ((e2 + k) * (e2 + k))
    return np.where(e2 <= k * k, 1.0, k / np.sqrt(e2))


def np_terms(J, r, w, C):
    """G, wsse of per-element Jacobians J[n, O, P], residuals r[n, O], weights w[n] and noise matrix C."""
    Cr = r @ C.T
    g = w[:, None] * np.einsum("nop,no->np", J, Cr)
    return g.T @ g, float(np.sum(w * np.sum(r * Cr, axis=1)))


@pytest.mark.parametrize("loss,k,with_cov", [(orc.LOSS_NONE, 0.0, False), (orc.LOSS_HUBER, 0.05, False),
                                             (orc.LOSS_HUBER, 0.05, True)])
def test_oracle_score_gram_point2point_matches_numpy(loss, k, with_cov):
    rng = np.random.default_rng(2)
    n = 997
    src = rng.uniform(0, 10, (n, 3))
    x = np.array([0.5, -0.3, 0.2, 0.1, -0.05, 0.08])
    T = orc.so3_convert6dof(x)
    tgt = src @ T[:3, :3].T + T[:3, 3] + rng.normal(0, 0.05, (n, 3))
    C = np.array([[2.0, 0.3, 0.1], [0.3, 1.5, -0.2], [0.1, -0.2, 0.7]]) if with_cov else np.eye(3)
    cost = orc.Cost(orc.P2P, 6, 3, n, a=src, b=tgt, jac_mode=orc.JAC_ANALYTICAL, variant=orc.P2P_REFTEST, loss=loss,
                    loss_param=k, cov=C if with_cov else None)
    G, wsse, nv = ocov.score_gram(cost, x)
    r = src @ T[:3, :3].T + T[:3, 3] - tgt
    J = np.concatenate([np.broadcast_to(np.eye(3), (n, 3, 3)), -np.stack([hat(p) for p in src])], axis=2)
    Gn, qn = np_terms(J, r, np_weight(loss, k, np.sum(r * r, axis=1)), C)
    assert nv == n
    assert np.max(np.abs(G - Gn)) <= 1e-12 * np.max(np.abs(Gn))
    assert wsse == pytest.approx(qn, rel=1e-12)
    # the b of the oracle's own linearization is the sum of the same scores
    _, bo, _ = orc.linearize(cost, x)
    w = np_weight(loss, k, np.sum(r * r, axis=1))
    gs = (w[:, None] * np.einsum("nop,no->np", J, r @ C.T)).sum(axis=0)
    assert np.max(np.abs(bo - gs)) <= 1e-12 * np.max(np.abs(gs))


@pytest.mark.parametrize("jac", [orc.JAC_ANALYTICAL, orc.JAC_FORWARD, orc.JAC_CENTRAL])
def test_oracle_score_gram_exp_curve_matches_numpy(jac):
    cost = curve_cost(jac_mode=jac, loss=orc.LOSS_HUBER, loss_param=0.2)
    x = [0.3, 0.1]
    G, wsse, nv = ocov.score_gram(cost, x)
    e = np.exp(x[0] * cost.a + x[1])
    r = (cost.b - e)[:, None]
    J = np.stack([-cost.a * e, -e], axis=1)[:, None, :]
    Gn, qn = np_terms(J, r, np_weight(orc.LOSS_HUBER, 0.2, r[:, 0] ** 2), np.eye(1))
    assert nv == cost.n
    # finite differences carry ~sqrt(eps) relative error per Jacobian entry (central: ~eps^(2/3))
    tol = 1e-13 if jac == orc.JAC_ANALYTICAL else 1e-6
    assert np.max(np.abs(G - Gn)) <= tol * np.max(np.abs(Gn))
    assert wsse == pytest.approx(qn, rel=1e-13)


# ---- mopt_covariance_from_terms -----------------------------------------------------------------------------------
def spd(P, seed, cond=1e3):
    rng = np.random.default_rng(seed)
    Q, _ = np.linalg.qr(rng.normal(size=(P, P)))
    ev = np.geomspace(1.0, cond, P)
    d = rng.uniform(0.1, 10.0, P)  # badly scaled parameters
    return (d[:, None] * (Q * ev) @ Q.T) * d[None, :]


def terms_of(capi, H, G=None, wsse=3.0, m=1000):
    P = H.shape[0]
    return capi.CovTerms.from_arrays(H, np.eye(P) if G is None else G, np.zeros(P), wsse, wsse, m, m)


def pinv_trunc_scaled(H, rcond):
    dg = np.diag(H)
    D = np.where(dg > 0, 1.0 / np.sqrt(np.where(dg > 0, dg, 1.0)), 0.0)
    S = D[:, None] * H * D[None, :]
    lam, V = np.linalg.eigh(S)
    keep = lam > rcond * lam.max()
    Sp = (V[:, keep] / lam[keep]) @ V[:, keep].T
    return D[:, None] * Sp * D[None, :], int(keep.sum())


@pytest.mark.parametrize("P", [1, 2, 6, 15, 16])
def test_full_rank_unscaled_is_the_inverse(capi, P):
    H = spd(P, P)
    res = capi.covariance_from_terms(terms_of(capi, H), capi.COV_UNSCALED)
    Hi = np.linalg.inv(H)
    assert np.max(np.abs(res.cov - Hi)) <= 1e-12 * np.max(np.abs(Hi))
    assert res.rank == P and res.dof == 1000 - P
    lam = np.linalg.eigvalsh(H / np.sqrt(np.outer(np.diag(H), np.diag(H))))
    assert res.eig_max == pytest.approx(lam.max(), rel=1e-12) and res.eig_min == pytest.approx(lam.min(), rel=1e-10)


@pytest.mark.parametrize("P,null", [(6, 1), (15, 3)])
def test_rank_deficient_terms(capi, P, null):
    rng = np.random.default_rng(7)
    A = rng.normal(size=(P, P - null)) * rng.uniform(0.1, 10.0, P)[:, None]
    H = A @ A.T
    H[2, :] = H[:, 2] = 0.0  # an unobservable parameter: zero diagonal entry
    res = capi.covariance_from_terms(terms_of(capi, H, m=500), capi.COV_UNSCALED, rcond=1e-9)
    ref, rank = pinv_trunc_scaled(H, 1e-9)
    assert res.rank == rank and res.dof == 500 - rank
    assert np.max(np.abs(res.cov - ref)) <= 1e-9 * np.max(np.abs(ref))
    assert np.all(res.cov[2] == 0.0) and np.isfinite(res.cov).all()


def test_scaled_and_sandwich(capi):
    P = 6
    H = spd(P, 3)
    rng = np.random.default_rng(4)
    B = rng.normal(size=(P, P))
    G = B @ B.T
    t = terms_of(capi, H, G, wsse=123.0, m=400)
    Hi = np.linalg.inv(H)
    sc = capi.covariance_from_terms(t, capi.COV_SCALED)
    assert sc.sigma2 == pytest.approx(123.0 / (400 - P), rel=1e-15)
    assert np.max(np.abs(sc.cov - sc.sigma2 * Hi)) <= 1e-12 * np.max(np.abs(sc.sigma2 * Hi))
    sw = capi.covariance_from_terms(t, capi.COV_SANDWICH)
    ref = Hi @ G @ Hi
    assert np.max(np.abs(sw.cov - ref)) <= 1e-11 * np.max(np.abs(ref)) and np.array_equal(sw.cov, sw.cov.T)
    assert np.allclose(sw.std, np.sqrt(np.diag(ref)), rtol=1e-11)
    assert sw.sigma2 == sc.sigma2


def test_terms_add(capi):
    H1, H2 = spd(3, 1), spd(3, 2)
    t = terms_of(capi, H1, wsse=1.0, m=10) + terms_of(capi, H2, wsse=2.0, m=20)
    assert np.array_equal(t.H, H1 + H2) and t.wsse == 3.0 and t.m == 30 and t.n_valid == 30
    with pytest.raises(ValueError):
        terms_of(capi, H1) + terms_of(capi, spd(2, 1))


def test_invalid_arguments_write_nothing(capi):
    good = terms_of(capi, spd(4, 5))

    def call(t, est=1, rcond=0.0):
        cov = np.full(16 * 16, 7.0)
        rep = capi.CovReport()
        rep.rank, rep.sigma2 = -5, 9.0
        rc = capi.lib().mopt_covariance_from_terms(ctypes.byref(t.raw), est, rcond, capi._dp(cov), ctypes.byref(rep))
        return rc, cov, rep

    rc, cov, rep = call(good)
    assert rc == capi.OK and rep.rank == 4
    bad = []
    for P in (0, 17, -1):
        t = terms_of(capi, spd(4, 5))
        t.raw.num_parameters = P
        bad.append((t, 1, 0.0))
    bad += [(good, 3, 0.0), (good, -1, 0.0), (good, 1, -1e-3), (good, 1, float("nan"))]
    for field, val in (("H", float("nan")), ("G", float("inf")), ("b", float("nan"))):
        t = terms_of(capi, spd(4, 5))
        getattr(t.raw, field)[1] = val
        bad.append((t, 1, 0.0))
    t = terms_of(capi, spd(4, 5))
    t.raw.wsse = float("inf")
    bad.append((t, 1, 0.0))
    t = terms_of(capi, spd(4, 5), m=4)  # m == rank: no degrees of freedom
    bad.append((t, 1, 0.0))
    for t, est, rcond in bad:
        rc, cov, rep = call(t, est, rcond)
        assert rc == 1, (t.P, est, rcond)  # MOPT_ERR_INVALID_ARGUMENT
        assert np.all(cov == 7.0) and rep.rank == -5 and rep.sigma2 == 9.0


def test_scaled_matches_scipy_curve_fit_pcov(capi):
    """Independent check: the exp curve on the 67-sample set, terms built in numpy at scipy's optimum."""
    from scipy.optimize import curve_fit
    cost = curve_cost()
    t, y = cost.a, cost.b

    def f(tt, a, b):
        return np.exp(a * tt + b)

    def jac(tt, a, b):
        e = np.exp(a * tt + b)
        return np.stack([tt * e, e], axis=1)

    popt, pcov = curve_fit(f, t, y, p0=[0.3, 0.1], jac=jac, xtol=1e-15, ftol=1e-15, gtol=1e-15)
    e = np.exp(popt[0] * t + popt[1])
    r = y - e
    J = np.stack([-t * e, -e], axis=1)  # of r = y - f
    g = J * r[:, None]
    terms = capi.CovTerms.from_arrays(J.T @ J, g.T @ g, g.sum(axis=0), float(r @ r), float(r @ r), len(t), len(t))
    res = capi.covariance_from_terms(terms, capi.COV_SCALED)
    assert res.rank == 2 and res.dof == len(t) - 2
    assert np.max(np.abs(res.cov - pcov)) <= 1e-8 * np.max(np.abs(pcov))
