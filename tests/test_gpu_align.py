"""Closed-form rigid alignment on the device (mopt_align_terms / Context.align_terms / Context.align): the terms
against fp64 numpy moments of the store's own values weighted by mopt_evaluate's own weights, the counts against
mopt_evaluate exactly, recovery of synthetic ground truth, a cloud far from the origin, determinism and the merge, the
RANSAC refit and classic (Besl-McKay) ICP end to end, argument validation and one 100 M case."""
import ctypes as C

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

from tests.test_align import kabsch, terms_of
from tests.test_gpu_evaluate import DTYPES, X_P2P, host_data

pytestmark = pytest.mark.gpu

LOSSES = [(0, 0.0), (1, 0.05), (2, 0.05)]  # NONE, Geman-McClure, Huber


@pytest.fixture(scope="module")
def env():
    from moptimizer_0_b200 import capi
    c = capi.Context(0)
    yield capi, c
    c.close()


def p2p_store(capi, ctx, n, sdt, seed=0):
    a, b = host_data(capi, capi.MODEL_POINT2POINT, n, seed)
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, sdt)
    st.upload(0, a)
    st.upload(1, b)
    return st, st.download(0), st.download(1)  # the store's own values


def oracle_terms(capi, ctx, st, prob, x, thr, p, q, first, count):
    """Moments of the used elements from the downloaded p, q and mopt_evaluate's weights in the compute dtype.  The
    used set is numpy's e2 of mopt_evaluate's residuals against thr^2; the few keys within 1e-6 of thr^2, where numpy's
    sum and the device's fma may round to different sides, take mopt_evaluate's decision for that one element."""
    ev = ctx.evaluate(st, prob, x, first=first, count=count, inlier_threshold=thr, out_dtype=prob.compute_dtype)
    r = ev.residuals.cpu().numpy().astype(np.float64)
    w = ev.weights.cpu().numpy().astype(np.float64)
    valid = ~np.isnan(r[:, 0])
    e2 = np.sum(r * r, axis=1)
    used = valid & (e2 <= thr * thr)
    if np.isfinite(thr):
        for i in np.nonzero(valid & (np.abs(e2 - thr * thr) <= 1e-6 * thr * thr))[0]:
            one = ctx.evaluate(st, prob, x, first=first + int(i), count=1, inlier_threshold=thr, residuals=False,
                               weights=False)
            used[i] = one.stats["n_inliers"] == 1
    assert used.sum() == ev.stats["n_inliers"]
    pp, qq = p[first:first + count], q[first:first + count]
    return terms_of(capi, pp[used], qq[used], w[used], n_valid=int(valid.sum())), ev.stats


def assert_terms_close(t, o, rel=1e-12):
    assert t.n_valid == o.n_valid and t.n_used == o.n_used
    if o.n_used == 0:
        assert t.w == 0.0
        return
    assert t.w == pytest.approx(o.w, rel=rel)
    for f in ("mean_src", "mean_tgt"):
        assert np.max(np.abs(getattr(t, f) - getattr(o, f))) <= rel * max(1.0, np.max(np.abs(getattr(o, f)))), f
    scale = max(o.var_src, o.var_tgt, 1e-300)
    for f in ("cross", "var_src", "var_tgt"):
        assert np.max(np.abs(np.asarray(getattr(t, f)) - np.asarray(getattr(o, f)))) <= rel * scale, f


# ---- terms against the oracle -----------------------------------------------------------------------------------
@pytest.mark.parametrize("loss,k", LOSSES)
@pytest.mark.parametrize("sdt,cdt", DTYPES)
def test_terms_match_oracle(env, sdt, cdt, loss, k):
    capi, ctx = env
    x = X_P2P + 0.01
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, cdt, loss=loss, loss_param=k)
    for n in (1, 31, 33, 1_000_003):  # one CTA up to the persistent grid
        st, p, q = p2p_store(capi, ctx, n, sdt, seed=n)
        ranges = [(0, n)]
        if n > 8:
            ranges += [(1, n - 1), (3, n - 5), (n - 3, 2), (5, 1), (7, 0)]  # ragged heads and tails, count < VEC, empty
        for first, count in ranges:
            for thr in (np.inf, 0.11):
                t = ctx.align_terms(st, prob, x, thr, first, count)
                if count == 0:
                    assert bytes(t.raw) == bytes(capi.AlignMomentsStruct())
                    continue
                o, stats = oracle_terms(capi, ctx, st, prob, x, thr, p, q, first, count)
                assert t.n_valid == stats["n_valid"] and t.n_used == stats["n_inliers"]
                assert_terms_close(t, o)
        st.close()


def test_launch_settings_agree_to_rounding(env):
    capi, ctx = env
    n = 1_000_003
    st, p, q = p2p_store(capi, ctx, n, 0, seed=2)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32, loss=2, loss_param=0.05)
    ref = ctx.align_terms(st, prob, X_P2P, 0.11)
    try:
        for cps in (1, 2):
            ctx.set_launch(cps, 0)
            t = ctx.align_terms(st, prob, X_P2P, 0.11)
            assert_terms_close(t, ref, 1e-13)
    finally:
        ctx.set_launch(0, 0)
    st.close()


# ---- exact counts -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
def test_counts_equal_evaluate_on_a_masked_store(env, sdt, cdt):
    from tests.test_icp import X_TRUE, clouds
    capi, ctx = env
    src, tgt = clouds()
    n = src.shape[0]
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, sdt)
    st.upload(0, src)
    ix = capi.NNIndex(ctx, tgt, 0.05, dtype=capi.F64)
    capi.store_set_target(st, ix)
    matched = capi.store_reassociate(st, X_TRUE)
    assert 0 < matched < n
    p, q = st.download(0), st.download(1)
    for loss, k in LOSSES:
        prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, cdt, loss=loss, loss_param=k)
        for x in (X_TRUE, X_TRUE + 0.003):
            for thr in (np.inf, 0.02, 0.003, 0.0):
                t = ctx.align_terms(st, prob, x, thr)
                s = ctx.evaluate(st, prob, x, inlier_threshold=thr, residuals=False, weights=False).stats
                assert (t.n_valid, t.n_used) == (s["n_valid"], s["n_inliers"]) and t.n_valid == matched
            o, _ = oracle_terms(capi, ctx, st, prob, x, np.inf, p, q, 0, n)
            assert_terms_close(ctx.align_terms(st, prob, x), o)
    capi.store_set_target(st, None)
    ix.close()
    st.close()


# ---- recovery ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
def test_noise_free_recovery(env, sdt, cdt):
    """mopt_store_generate forms the targets in fp32 (its rotation rounded to fp32 too), so an fp32 store recovers the
    ground truth to 1e-5; the fp64 store holds noise-free fp64 pairs from the host and recovers it to 1e-10."""
    capi, ctx = env
    n = 1_000_003
    gt = np.array([0.5, -0.3, 0.2, 1.2, -1.0, 1.2])  # |omega| = 1.97 rad
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, sdt)
    if sdt == capi.F32:
        st.generate(seed=21, gt=gt)
        tol = 1e-5
    else:
        p = np.random.default_rng(21).uniform(0, 10, (n, 3))
        st.upload(0, p)
        st.upload(1, p @ Rotation.from_rotvec(gt[3:]).as_matrix().T + gt[:3])
        tol = 1e-10
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, cdt)
    a = ctx.align(st, prob, np.zeros(6))
    assert np.max(np.abs(a.x - gt)) <= tol, a.x - gt
    assert not a.degenerate
    st.close()


def test_cost_matches_compute_cost(env):
    capi, ctx = env
    n = 1_000_003
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F64)
    st.generate(seed=22, gt=X_P2P, noise_sigma=0.01)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64)
    a = ctx.align(st, prob, np.zeros(6))
    c = ctx.compute_cost(st, prob, a.x)
    assert a.cost == pytest.approx(c, rel=1e-9)
    assert a.rms == pytest.approx(np.sqrt(c / n), rel=1e-9)
    st.close()


def test_cloud_far_from_the_origin(env):
    capi, ctx = env
    n = 1_000_003
    rng = np.random.default_rng(23)
    p = rng.normal(0, 1, (n, 3)) + np.array([1e6, -1e6, 5e5])
    R = Rotation.from_rotvec([0.2, -0.1, 0.3]).as_matrix()
    q = p @ R.T + np.array([3.0, -2.0, 1.0]) + rng.normal(0, 0.01, (n, 3))
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F64)
    st.upload(0, p)
    st.upload(1, q)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64)
    a = ctx.align(st, prob, np.zeros(6))
    Ro, to = kabsch(p, q)
    Ra = Rotation.from_rotvec(a.x[3:]).as_matrix()
    assert Rotation.from_matrix(Ra.T @ Ro).magnitude() <= 1e-10
    assert np.max(np.abs(a.x[:3] - to)) <= 1e-8
    st.close()


# ---- determinism and the merge ----------------------------------------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
def test_determinism_and_merge(env, sdt, cdt):
    capi, ctx = env
    n = 1_000_003
    st, _, _ = p2p_store(capi, ctx, n, sdt, seed=24)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, cdt, loss=2, loss_param=0.05)
    t1 = ctx.align_terms(st, prob, X_P2P, 0.11)
    t2 = ctx.align_terms(st, prob, X_P2P, 0.11)
    assert bytes(t1.raw) == bytes(t2.raw)
    # the Jacobian mode, variant, manifold and covariance do not enter
    other = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_CENTRAL, cdt, loss=2, loss_param=0.05,
                              variant=capi.P2P_LEFT, manifold=capi.MANIFOLD_SO3_LEFT, covariance=np.diag([2.0, 1, 1]))
    assert bytes(ctx.align_terms(st, other, X_P2P, 0.11).raw) == bytes(t1.raw)
    for k in (1, 4, 333_331, n - 3):
        a, b = ctx.align_terms(st, prob, X_P2P, 0.11, 0, k), ctx.align_terms(st, prob, X_P2P, 0.11, k, n - k)
        assert_terms_close(a + b, t1, 1e-13)
        assert bytes((a + b).raw) == bytes((b + a).raw)
    st.close()


# ---- end to end -------------------------------------------------------------------------------------------------
def test_ransac_refit(env):
    """tests/test_gpu_hypotheses.py::test_ransac_end_to_end, with the closed-form refit on the best hypothesis's inlier
    set next to that test's Huber LM."""
    from tests.test_gpu_hypotheses import kabsch as kabsch_x
    capi, ctx = env
    n = 1_000_003
    x_gt = np.array([0.5, -0.3, 0.2, 1.2, -1.0, 1.2])
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    st.generate(seed=14, gt=x_gt, noise_sigma=0.01, outlier_fraction=0.6, outlier_range=10.0)
    src, tgt = st.download(0), st.download(1)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32)
    rng = np.random.default_rng(15)
    xs = np.array([kabsch_x(src[i], tgt[i]) for i in (rng.choice(n, 3, replace=False) for _ in range(512))])
    thr = 0.05
    best = int(np.argmax(ctx.score_hypotheses(st, prob, xs, thr).n_inliers))
    refit = ctx.align(st, prob, xs[best], thr)
    huber = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64, loss=capi.LOSS_HUBER,
                              loss_param=thr)
    lm = ctx.lm_minimize([st], [huber], xs[best], max_iterations=50)
    e_refit, e_lm = np.max(np.abs(refit.x - x_gt)), np.max(np.abs(lm.x - x_gt))
    print(f"RANSAC refit: closed form {e_refit:.2e}, Huber LM {e_lm:.2e} from the ground truth")
    assert e_refit <= 1e-3 and e_refit <= e_lm, (e_refit, e_lm)
    st.close()


def test_classic_icp_converges_to_the_ground_truth(env):
    """Besl-McKay point-to-point ICP: re-associate at x, solve in closed form, repeat until the step is below 1e-10; on
    the clouds, start and MAX_DIST of tests/test_icp.py, against the LM-driven ICP of the same scene.  Measured on a
    B200: 8 iterations (the last one a zero step), 1.1e-4 from X_TRUE and 1e-15 from the LM-driven ICP's solution."""
    from tests.test_icp import MAX_DIST, X_TRUE, clouds
    capi, ctx = env
    src, tgt = clouds()
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, src.shape[0], capi.F64)
    st.upload(0, src)
    ix = capi.NNIndex(ctx, tgt, MAX_DIST, dtype=capi.F64)
    capi.store_set_target(st, ix)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64)
    x = np.zeros(6)
    for it in range(1, 201):
        capi.store_reassociate(st, x)
        x_new = ctx.align(st, prob, x).x
        step = np.max(np.abs(x_new - x))
        x = x_new
        if step < 1e-10:
            break
    print(f"classic ICP: {it} iterations, last step {step:.1e}, |x - x_true| {np.max(np.abs(x - X_TRUE)):.2e}")
    assert step < 1e-10
    assert np.allclose(x, X_TRUE, atol=2e-3), x
    lm = ctx.lm_minimize([st], [prob], [0.0] * 6, max_iterations=30)
    assert np.allclose(lm.x, X_TRUE, atol=2e-3)
    print(f"classic ICP vs LM-driven ICP: {np.max(np.abs(x - lm.x)):.1e}")
    assert np.max(np.abs(x - lm.x)) <= 1e-9, (x, lm.x)
    capi.store_set_target(st, None)
    ix.close()
    st.close()


# ---- invalid arguments ------------------------------------------------------------------------------------------
def test_invalid_arguments_write_nothing(env):
    from tests.test_user_model import P2P_SRC
    capi, ctx = env
    n = 1000
    st, _, _ = p2p_store(capi, ctx, n, 0)
    other_ctx = capi.Context(0)
    other, _, _ = p2p_store(capi, other_ctx, n, 0)
    dist = capi.Store(ctx, capi.MODEL_POINT_DIST, n, capi.F32)
    curve = capi.Store(ctx, capi.MODEL_EXP_CURVE, n, capi.F32)
    up = capi.UserModel(P2P_SRC, 6, 3, 3, 3, set_size=12, rot_offset=3)
    user = capi.Store(ctx, up.model, n, capi.F32)
    prob = capi.make_problem(capi.MODEL_POINT2POINT)
    x = np.zeros(6)
    out = capi.AlignMomentsStruct()
    out.n_valid, out.w = -5, -7.25
    sentinel = bytes(out)

    def call(store=st, problem=prob, xv=x, first=0, count=n, thr=0.1, o=out):
        return capi.lib().mopt_align_terms(ctx.handle, store.handle, C.byref(problem),
                                           capi._dp(xv) if xv is not None else None, first, count, thr,
                                           C.byref(o) if o is not None else None)

    try:
        bad = [
            dict(store=dist, problem=capi.make_problem(capi.MODEL_POINT_DIST)),   # not point2point: builtin
            dict(store=curve, problem=capi.make_problem(capi.MODEL_EXP_CURVE)),
            dict(store=user, problem=capi.make_problem(up.model)),                # ... and user
            dict(store=other),                                                     # a store of another context
            dict(problem=capi.make_problem(capi.MODEL_EXP_CURVE)),                 # a problem the store does not accept
            dict(first=-1, count=10), dict(first=0, count=n + 1), dict(first=n - 5, count=6), dict(count=-1),
            dict(thr=-1e-300), dict(thr=-np.inf), dict(thr=np.nan),
            dict(xv=None), dict(o=None),
        ]
        for kw in bad:
            assert call(**kw) == 1, kw  # MOPT_ERR_INVALID_ARGUMENT
            assert bytes(out) == sentinel, kw
        assert call() == 0 and out.n_valid == n
    finally:
        for s in (dist, curve, user, other, st):
            s.close()
        up.release()
        other_ctx.close()


# ---- full size --------------------------------------------------------------------------------------------------
def test_point2point_100m_fp32(env):
    capi, ctx = env
    n = 100_000_000
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    st.generate(seed=1, gt=X_P2P, noise_sigma=0.01, outlier_fraction=0.05, outlier_range=1.0)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32)
    thr = 0.05
    a = ctx.align(st, prob, X_P2P + 0.002, thr)
    s = ctx.evaluate(st, prob, X_P2P + 0.002, inlier_threshold=thr, residuals=False, weights=False).stats
    t = ctx.align_terms(st, prob, X_P2P + 0.002, thr)
    assert (t.n_valid, t.n_used) == (n, s["n_inliers"])
    assert np.max(np.abs(a.x - X_P2P)) <= 1e-4, a.x - X_P2P
    st.close()
