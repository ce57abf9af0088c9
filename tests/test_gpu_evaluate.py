"""Per-residual evaluation on the device (mopt_evaluate / Context.evaluate): residuals and loss weights of every
builtin model against the oracle's computeCost loop with each element kept, fit statistics against numpy and
mopt_compute_cost, ranges, NaN-masked ICP stores, a run-time compiled user model and argument validation."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle_py as orc
from tests import oracle_evaluate as oev
from tests.common import camera_consts, fachada

pytestmark = pytest.mark.gpu

EPS32 = float(np.finfo(np.float32).eps)
SIZES = (1, 31, 33, 1_000_003)
DTYPES = [(0, 0), (0, 1), (1, 1)]  # (store, compute): every pair the pass kernels accept
LOSSES = [(0, 0.0), (1, None), (2, None)]
X_P2P = np.array([0.5, -0.3, 0.2, 0.1, -0.05, 0.08])
X_DIST = np.array([-0.01, 0.02, -0.06, 0.018, -0.0013, 0.027, 586.0, 722.0, 638.0, 323.0, -0.12, 0.05, 0.001, -0.0007,
                   0.01])


@pytest.fixture(scope="module")
def env():
    from moptimizer_0_b200 import capi
    c = capi.Context(0)
    yield capi, c
    c.close()


# model -> (oracle kind, x, loss scale: a typical |r|, consts)
def model_table(capi):
    cam = camera_consts()
    return {
        capi.MODEL_POINT2POINT: (orc.P2P, X_P2P + 0.01, 0.05, None),
        capi.MODEL_EXP_CURVE: (orc.EXP_CURVE, np.array([0.3, 0.1]), 0.2, None),
        capi.MODEL_MICHAELIS_MENTEN: (orc.MICHAELIS_MENTEN, np.array([0.5, 0.6]), 0.05, None),
        capi.MODEL_PINHOLE: (orc.PINHOLE, np.array([-0.01, 0.02, -0.06, 0.018, -0.0013, 0.027]), 1.0, cam),
        capi.MODEL_POWELL: (orc.POWELL, np.array([3.0, -1.0, 0.0, 1.0]), 10.0, None),
        capi.MODEL_POINT_DIST: (orc.POINT_DIST, np.zeros(0), 0.05, None),
        capi.MODEL_PINHOLE_DISTORT: (orc.PINHOLE_DISTORT, X_DIST, 1.0, cam[12:]),
    }


def host_data(capi, model, n, seed=0):
    """Group A / B host arrays of `n` elements (None for the data-free Powell model)."""
    rng = np.random.default_rng(seed)
    if model in (capi.MODEL_POINT2POINT, capi.MODEL_POINT_DIST):
        src = rng.uniform(0, 10, (n, 3))
        T = orc.so3_convert6dof(X_P2P)
        tgt = src @ T[:3, :3].T + T[:3, 3] + rng.normal(0, 0.05, (n, 3))
        return src, tgt
    if model == capi.MODEL_EXP_CURVE:
        t = rng.uniform(0, 5, n)
        return t, np.exp(0.3 * t + 0.1) + rng.normal(0, 0.2, n)
    if model == capi.MODEL_MICHAELIS_MENTEN:
        t = rng.uniform(0.1, 4, n)
        return t, 0.5 * t / (0.6 + t) + rng.normal(0, 0.05, n)
    if model == capi.MODEL_PINHOLE:
        cam = camera_consts()
        K, Cm = cam[:12].reshape(3, 4), cam[12:].reshape(4, 4)
        pts = np.column_stack([rng.uniform(2, 5, n), rng.uniform(-1, 1, n), rng.uniform(-0.5, 1, n)])
        U = np.column_stack([pts, np.ones(n)]) @ (K @ orc.so3_convert6dof(model_table(capi)[model][1]) @ Cm).T
        return pts, U[:, :2] / U[:, 2:3] + rng.normal(0, 0.5, (n, 2))
    return None, None


def make_store(capi, ctx, model, n, sdt, seed=0):
    st = capi.Store(ctx, model, n, sdt)
    if model == capi.MODEL_PINHOLE_DISTORT:
        st.generate(seed=seed + 3, gt=X_DIST, lo=(2.0, -1.0, -0.5), hi=(5.0, 1.0, 1.0), noise_sigma=0.3,
                    consts=camera_consts()[12:])
    elif model != capi.MODEL_POWELL:
        a, b = host_data(capi, model, n, seed)
        st.upload(0, a)
        st.upload(1, b)
    if model == capi.MODEL_POWELL:
        return st, None, None
    return st, st.download(0), st.download(1)  # what the oracle is fed: the store's own values


def np_weight(loss, k, e2):
    if loss == 0:
        return np.ones_like(e2)
    if loss == 1:
        return (k * k) / ((e2 + k) * (e2 + k))
    with np.errstate(divide="ignore"):
        return np.where(e2 <= k * k, 1.0, k / np.sqrt(e2))


def element_scale(r_ref, a, b):
    """Per element: the largest magnitude among its data and its residual (the terms the residual is formed from)."""
    s = np.max(np.abs(r_ref), axis=1)
    for d in (a, b):
        if d is not None:
            s = np.maximum(s, np.max(np.abs(d.reshape(len(s), -1)), axis=1))
    return np.maximum(s, 1.0)


def check_against_oracle(r, w, ro, wo, scale, loss, k, f32):
    """fp64 compute: residuals within 1e-12 of the element's scale, weights within 1e-12.
    fp32 compute: the residual is a few rounded products and sums of terms no larger than the element's scale, plus
    float(x) / float(setup(x)) instead of x: 64 eps_f32 of that scale bounds it with a wide margin.  The weight is the
    loss of a float r^T r: it must lie in the loss's image of r^T r moved by that residual bound (losses are monotone
    in r^T r), widened by 8 eps_f32 for the float evaluation of the loss itself."""
    err = np.max(np.abs(r - ro), axis=1)
    if not f32:
        assert np.all(err <= 1e-12 * scale), np.max(err / scale)
        assert np.max(np.abs(w - wo)) <= 1e-12
        return
    tol = 64 * EPS32 * scale
    assert np.all(err <= tol), np.max(err / scale)
    norm = np.sqrt(np.sum(ro * ro, axis=1))
    e2_lo = np.maximum(norm - np.sqrt(ro.shape[1]) * tol, 0.0) ** 2
    e2_hi = (norm + np.sqrt(ro.shape[1]) * tol) ** 2
    w_a, w_b = np_weight(loss, k, e2_lo), np_weight(loss, k, e2_hi)
    lo, hi = np.minimum(w_a, w_b), np.maximum(w_a, w_b)
    assert np.all((w >= lo * (1 - 8 * EPS32)) & (w <= hi * (1 + 8 * EPS32))), np.max(np.abs(w - wo))


# ---- 1. per-element parity with the oracle -----------------------------------------------------------------------
@pytest.mark.parametrize("loss,kp", LOSSES)
@pytest.mark.parametrize("sdt,cdt", DTYPES)
@pytest.mark.parametrize("model", range(7))
def test_parity_with_oracle(env, model, sdt, cdt, loss, kp):
    capi, ctx = env
    kind, x, scale_k, consts = model_table(capi)[model]
    k = scale_k if kp is None else kp
    P, O, _, _ = capi.MODEL_SHAPE[model]
    for n in SIZES:
        st, a, b = make_store(capi, ctx, model, n, sdt, seed=n)
        prob = capi.make_problem(model, capi.JAC_FORWARD, cdt, loss=loss, loss_param=k, consts=consts)
        res = ctx.evaluate(st, prob, x, out_dtype=capi.F64)
        r, w = res.residuals.cpu().numpy(), res.weights.cpu().numpy()
        oc = orc.Cost(kind, P, O, n, a=a, b=b, consts=consts, loss=loss, loss_param=k)
        ro, wo, valid = oev.evaluate(oc, x)
        assert valid.all() and r.shape == (n, O) and w.shape == (n,)
        check_against_oracle(r, w, ro, wo, element_scale(ro, a, b), loss, k, cdt == capi.F32)
        # 2. consistency: sum r^T r is mopt_compute_cost's value, every element is valid, outputs do not move the stats
        s = res.stats
        assert s["n_valid"] == n and s["n_inliers"] == n
        e2 = np.sum(r * r, axis=1)
        tol = 1e-12 if cdt == capi.F64 else 1e-6
        assert abs(s["sum_sq"] - np.sum(e2)) <= tol * np.sum(e2)
        # the data-free Powell pass adds its n identical residuals serially in the compute dtype: compared where
        # that sum is exact enough to be a reference
        if model != capi.MODEL_POWELL or n <= 33:
            cost = ctx.compute_cost(st, prob, x)
            assert abs(s["sum_sq"] - cost) <= tol * cost
        assert s["max_sq"] == pytest.approx(float(e2.max()), rel=1e-12 if cdt == capi.F64 else 1e-6)
        only = ctx.evaluate(st, prob, x, residuals=False, weights=False, out_dtype=capi.F64)
        assert only.residuals is None and only.weights is None and only.stats == s
        # fp32 outputs are the same values rounded once
        r32 = ctx.evaluate(st, prob, x, out_dtype=capi.F32)
        assert r32.stats == s
        assert np.array_equal(r32.residuals.cpu().numpy(), r.astype(np.float32))
        assert np.array_equal(r32.weights.cpu().numpy(), w.astype(np.float32))
        st.close()


def test_parity_fachada(env):
    capi, ctx = env
    src, tgt, _, _ = fachada()
    n = src.shape[0]
    x = np.array([0.01, -0.02, 0.03, 0.004, -0.003, 0.002])
    for sdt, cdt in DTYPES:
        st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, sdt)
        st.upload(0, src)
        st.upload(1, tgt)
        a, b = st.download(0), st.download(1)
        for loss, k in LOSSES:
            k = 0.05 if k is None else k
            prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, cdt, loss=loss, loss_param=k)
            res = ctx.evaluate(st, prob, x, out_dtype=capi.F64)
            ro, wo, _ = oev.evaluate(orc.Cost(orc.P2P, 6, 3, n, a=a, b=b, loss=loss, loss_param=k), x)
            check_against_oracle(res.residuals.cpu().numpy(), res.weights.cpu().numpy(), ro, wo,
                                 element_scale(ro, a, b), loss, k, cdt == capi.F32)
            cost = ctx.compute_cost(st, prob, x)
            assert abs(res.stats["sum_sq"] - cost) <= (1e-12 if cdt == capi.F64 else 1e-6) * cost
        st.close()


# ---- 2. determinism, 3. ranges ---------------------------------------------------------------------------------
@pytest.mark.parametrize("model", [0, 1, 3, 6])
@pytest.mark.parametrize("sdt,cdt", DTYPES)
def test_repeatable_and_ranges_compose(env, model, sdt, cdt):
    capi, ctx = env
    _, x, k, consts = model_table(capi)[model]
    n = 1_000_003
    st, _, _ = make_store(capi, ctx, model, n, sdt, seed=7)
    prob = capi.make_problem(model, capi.JAC_FORWARD, cdt, loss=capi.LOSS_HUBER, loss_param=k, consts=consts)
    thr = k
    full = ctx.evaluate(st, prob, x, inlier_threshold=thr)
    again = ctx.evaluate(st, prob, x, inlier_threshold=thr)
    assert full.stats == again.stats
    assert np.array_equal(full.residuals.cpu().numpy(), again.residuals.cpu().numpy())
    assert np.array_equal(full.weights.cpu().numpy(), again.weights.cpu().numpy())
    assert 0 < full.stats["n_inliers"] < n
    cuts = [0, 333_331, 333_332 + 5, n]  # ragged: every chunk starts and ends off a 16-byte boundary
    parts = [ctx.evaluate(st, prob, x, first=lo, count=hi - lo, inlier_threshold=thr) for lo, hi in zip(cuts, cuts[1:])]
    r = np.concatenate([p.residuals.cpu().numpy() for p in parts])
    w = np.concatenate([p.weights.cpu().numpy() for p in parts])
    assert np.array_equal(r, full.residuals.cpu().numpy()) and np.array_equal(w, full.weights.cpu().numpy())
    for key in ("n_valid", "n_inliers"):
        assert sum(p.stats[key] for p in parts) == full.stats[key]
    for key in ("sum_sq", "inlier_sum_sq"):
        assert sum(p.stats[key] for p in parts) == pytest.approx(full.stats[key], rel=1e-12)
    assert max(p.stats["max_sq"] for p in parts) == full.stats["max_sq"]
    st.close()


# ---- 4. NaN-masked ICP store, 5. fit statistics after a device LM ------------------------------------------------
def threshold_clear_of(e2, q):
    """A threshold near the q-quantile of sqrt(e2) with no residual norm within 1e-6 relative of it."""
    norms = np.sort(np.sqrt(e2))
    i = int(q * (len(norms) - 1))
    while i + 1 < len(norms) and norms[i + 1] <= norms[i] * (1 + 4e-6):
        i += 1
    return float(np.sqrt(norms[i] * norms[min(i + 1, len(norms) - 1)]))


def check_fit(res, thr):
    r = res.residuals.cpu().numpy()
    valid = ~np.isnan(r[:, 0])
    e2 = np.sum(r[valid] ** 2, axis=1)
    assert np.min(np.abs(np.sqrt(e2) / thr - 1)) > 1e-6
    inl = e2 <= thr * thr
    assert res.stats["n_valid"] == int(valid.sum()) and res.stats["n_inliers"] == int(inl.sum())
    assert res.fitness == int(inl.sum()) / len(r)
    assert res.inlier_rmse == pytest.approx(np.sqrt(np.sum(e2[inl]) / inl.sum()), rel=1e-12)
    assert res.rms == pytest.approx(np.sqrt(np.sum(e2) / valid.sum()), rel=1e-12)


@pytest.mark.parametrize("dtype", [0, 1])
def test_masked_icp_store(env, dtype):
    from tests.test_icp import MAX_DIST, X_TRUE, clouds
    capi, ctx = env
    src, tgt = clouds()
    n = src.shape[0]
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, dtype)
    st.upload(0, src)
    ix = capi.NNIndex(ctx, tgt, MAX_DIST, dtype=capi.F64)
    capi.store_set_target(st, ix)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, dtype, loss=capi.LOSS_HUBER, loss_param=0.05)
    matched = capi.store_reassociate(st, X_TRUE)
    tq = st.download(1)
    res = ctx.evaluate(st, prob, X_TRUE, out_dtype=capi.F64)
    r, w = res.residuals.cpu().numpy(), res.weights.cpu().numpy()
    miss = np.isnan(tq[:, 0])
    assert 0 < miss.sum() < n
    assert np.isnan(r[miss]).all() and (w[miss] == 0).all()
    assert not np.isnan(r[~miss]).any() and (w[~miss] > 0).all()
    assert res.stats["n_valid"] == matched == n - int(miss.sum())
    cost = ctx.compute_cost(st, prob, X_TRUE)  # no re-association here either: same correspondences
    assert abs(res.stats["sum_sq"] - cost) <= (1e-12 if dtype == capi.F64 else 1e-6) * cost
    # evaluation never re-associates: at another x the store still holds the correspondences made at X_TRUE
    ctx.evaluate(st, prob, np.zeros(6), residuals=False, weights=False)
    assert np.array_equal(np.isnan(st.download(1)[:, 0]), miss)
    ro, wo, valid = oev.evaluate(orc.Cost(orc.P2P, 6, 3, n, a=st.download(0), b=tq, loss=orc.LOSS_HUBER,
                                          loss_param=0.05), X_TRUE)
    if dtype == capi.F64:
        assert np.max(np.abs(r[~miss] - ro[~miss])) <= 1e-12 * np.max(np.abs(tq[~miss]))
        assert np.max(np.abs(w[~miss] - wo[~miss])) <= 1e-12
    capi.store_set_target(st, None)
    ix.close()
    st.close()


def test_fit_statistics_after_device_lm(env):
    from tests.test_icp import MAX_DIST, clouds
    capi, ctx = env
    # noisy fachada registration with 5 % outliers, Huber, fp64
    src, tgt, _, _ = fachada()
    rng = np.random.default_rng(11)
    n = src.shape[0]
    noisy = tgt + rng.normal(0, 0.005, tgt.shape)
    out = rng.random(n) < 0.05
    noisy[out] += rng.uniform(-0.5, 0.5, (int(out.sum()), 3))
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F64)
    st.upload(0, src)
    st.upload(1, noisy)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64, loss=capi.LOSS_HUBER, loss_param=0.02)
    lm = ctx.lm_minimize([st], [prob], np.zeros(6), max_iterations=30)
    probe = ctx.evaluate(st, prob, lm.x, weights=False, out_dtype=capi.F64)
    e2 = np.sum(probe.residuals.cpu().numpy() ** 2, axis=1)
    thr = threshold_clear_of(e2, 0.9)
    res = ctx.evaluate(st, prob, lm.x, inlier_threshold=thr, out_dtype=capi.F64)
    check_fit(res, thr)
    assert 0.85 < res.fitness < 0.95 and res.inlier_rmse < thr
    st.close()
    # ICP clouds: LM with re-association, then evaluation at the solution's correspondences
    src, tgt = clouds()
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, src.shape[0], capi.F64)
    st.upload(0, src)
    ix = capi.NNIndex(ctx, tgt, MAX_DIST, dtype=capi.F64)
    capi.store_set_target(st, ix)
    lm = ctx.lm_minimize([st], [prob], np.zeros(6), max_iterations=30)
    capi.store_reassociate(st, lm.x)
    probe = ctx.evaluate(st, prob, lm.x, weights=False, out_dtype=capi.F64)
    r = probe.residuals.cpu().numpy()
    thr = threshold_clear_of(np.sum(r[~np.isnan(r[:, 0])] ** 2, axis=1), 0.5)
    res = ctx.evaluate(st, prob, lm.x, inlier_threshold=thr, out_dtype=capi.F64)
    check_fit(res, thr)
    assert res.fitness < 1.0 and res.stats["n_valid"] < src.shape[0]
    capi.store_set_target(st, None)
    ix.close()
    st.close()


# ---- 6. user model ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
def test_user_model_matches_oracle_and_builtin(env, sdt, cdt):
    from tests.test_user_model import EXP_CURVE_SRC
    capi, ctx = env
    um = capi.UserModel(EXP_CURVE_SRC, 2, 1, 1, 1, has_jacobian=True)
    x = np.array([0.3, 0.1])
    try:
        for n in SIZES:
            a, b = host_data(capi, capi.MODEL_EXP_CURVE, n, seed=n)
            su = capi.Store(ctx, um.model, n, sdt)
            sb = capi.Store(ctx, capi.MODEL_EXP_CURVE, n, sdt)
            for s in (su, sb):
                s.upload(0, a)
                s.upload(1, b)
            da, db = su.download(0), su.download(1)
            for loss, k in LOSSES:
                k = 0.2 if k is None else k
                pu = capi.make_problem(um.model, capi.JAC_FORWARD, cdt, loss=loss, loss_param=k)
                res = ctx.evaluate(su, pu, x, inlier_threshold=0.3, out_dtype=capi.F64)
                ro, wo, _ = oev.evaluate(orc.Cost(orc.EXP_CURVE, 2, 1, n, a=da, b=db, loss=loss, loss_param=k), x)
                r, w = res.residuals.cpu().numpy(), res.weights.cpu().numpy()
                check_against_oracle(r, w, ro, wo, element_scale(ro, da, db), loss, k, cdt == capi.F32)
                pb = capi.make_problem(capi.MODEL_EXP_CURVE, capi.JAC_FORWARD, cdt, loss=loss, loss_param=k)
                rb = ctx.evaluate(sb, pb, x, inlier_threshold=0.3, out_dtype=capi.F64)
                assert rb.stats["n_inliers"] == res.stats["n_inliers"]
                assert rb.stats["sum_sq"] == pytest.approx(res.stats["sum_sq"], rel=1e-12 if cdt else 1e-6)
                f32 = ctx.evaluate(su, pu, x, inlier_threshold=0.3, out_dtype=capi.F32)
                assert f32.stats == res.stats and np.array_equal(f32.residuals.cpu().numpy(), r.astype(np.float32))
            su.close()
            sb.close()
    finally:
        um.release()


# ---- 7. invalid arguments -----------------------------------------------------------------------------------------
def test_invalid_arguments_write_nothing(env):
    import torch
    capi, ctx = env
    n = 1000
    st, _, _ = make_store(capi, ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    prob = capi.make_problem(capi.MODEL_POINT2POINT)
    x = np.zeros(6)
    xs = np.ascontiguousarray(x)
    r = torch.full((n, 3), 7.25, dtype=torch.float32, device="cuda:0")
    w = torch.full((n,), 7.25, dtype=torch.float32, device="cuda:0")
    stats = capi.EvalStats()
    stats.n_valid, stats.sum_sq = -5, -7.25

    def call(first, count, out_dtype, rp, wp, sp, threshold=float("inf")):
        return capi.lib().mopt_evaluate(ctx.handle, st.handle, C.byref(prob), capi._dp(xs), first, count, threshold,
                                        out_dtype, rp, wp, sp)

    rp, wp, sp = r.data_ptr(), w.data_ptr(), C.byref(stats)
    host = np.zeros(3 * n, dtype=np.float32)
    bad = [
        (-1, 10, capi.F32, rp, wp, sp),     # range outside the store
        (0, n + 1, capi.F32, rp, wp, sp),
        (n - 5, 6, capi.F32, rp, wp, sp),
        (0, -1, capi.F32, None, None, sp),  # negative count
        (0, n, 2, rp, wp, sp),              # out_dtype
        (0, 0, capi.F32, rp, None, sp),     # outputs with an empty range
        (0, 0, capi.F32, None, wp, sp),
        (0, n, capi.F32, None, None, None),  # nothing to do
        (0, n, capi.F32, host.ctypes.data, None, sp),  # host memory is not a device output
    ]
    for args in bad:
        assert call(*args) == 1, args  # MOPT_ERR_INVALID_ARGUMENT
    torch.cuda.synchronize()
    assert bool((r == 7.25).all()) and bool((w == 7.25).all())
    assert stats.n_valid == -5 and stats.sum_sq == -7.25
    # a wrong problem for the store is rejected by the same validation as the passes
    other = capi.make_problem(capi.MODEL_EXP_CURVE)
    assert capi.lib().mopt_evaluate(ctx.handle, st.handle, C.byref(other), capi._dp(xs), 0, n, float("inf"), capi.F32,
                                    rp, wp, C.byref(stats)) == 1
    assert bool((r == 7.25).all()) and stats.n_valid == -5
    # the Python wrapper checks supplied tensors
    with pytest.raises(ValueError):
        ctx.evaluate(st, prob, x, out=(torch.empty((n, 3), dtype=torch.float64, device="cuda:0"), None))
    with pytest.raises(ValueError):
        ctx.evaluate(st, prob, x, out=(None, torch.empty((n + 1,), dtype=torch.float32, device="cuda:0")))
    # an empty stats-only range is fine; caller-supplied tensors are written in place
    assert call(5, 0, capi.F32, None, None, sp) == 0 and stats.n_valid == 0 and stats.sum_sq == 0.0
    res = ctx.evaluate(st, prob, x, out=(r, w))
    assert res.residuals is r and res.stats["n_valid"] == n
    st.close()


# ---- 8. one 100 M point2point fp32 case -------------------------------------------------------------------------
def test_point2point_100m_fp32(env):
    capi, ctx = env
    n = 100_000_000
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    st.generate(seed=1, gt=X_P2P, noise_sigma=0.01, outlier_fraction=0.05, outlier_range=1.0)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32, loss=capi.LOSS_HUBER, loss_param=0.05)
    x = X_P2P
    res = ctx.evaluate(st, prob, x, inlier_threshold=0.05)
    cost = ctx.compute_cost(st, prob, x)
    assert res.stats["n_valid"] == n and abs(res.stats["sum_sq"] - cost) <= 1e-6 * cost
    assert 0.9 < res.fitness < 0.99
    w = res.weights
    assert int((w < 1).sum()) == pytest.approx(n - res.stats["n_inliers"], rel=0.05)
    st.close()
