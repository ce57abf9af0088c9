"""Exact residual quantiles on the device (mopt_residual_quantiles / Context.quantiles).  The reference is numpy:
e = r^T r recomputed from Context.evaluate's residuals in the compute dtype (e = r0 r0, then e = e + ro ro, every
step rounded), ranked with np.sort / np.partition and interpolated by np.quantile.  Every comparison is exact."""
import ctypes as C

import numpy as np
import pytest

from tests.test_gpu_evaluate import DTYPES, SIZES, X_P2P, make_store, model_table

pytestmark = pytest.mark.gpu

QS = np.array([0.0, 0.1, 0.5, 0.9, 0.99, 1.0])
CHI2_MEDIAN = {1: 0.454936423119572, 2: 1.386294361119891, 3: 2.3659738843753377, 4: 3.3566939800333224}


@pytest.fixture(scope="module")
def env():
    from moptimizer_0_b200 import capi
    c = capi.Context(0)
    yield capi, c
    c.close()


def keys_of(r, cdt):
    """e = r^T r as the library forms it: compute dtype, component order, no fused multiply-add."""
    r = r.astype(np.float32 if cdt == 0 else np.float64)
    with np.errstate(over="ignore", invalid="ignore"):  # +inf and NaN keys are part of the cases
        e = r[:, 0] * r[:, 0]
        for o in range(1, r.shape[1]):
            e = e + r[:, o] * r[:, o]
    return e.astype(np.float64)


def device_keys(capi, ctx, st, prob, x, first=0, count=None):
    res = ctx.evaluate(st, prob, x, first=first, count=count, weights=False, out_dtype=prob.compute_dtype)
    return keys_of(res.residuals.cpu().numpy(), prob.compute_dtype)


def expect(e, qs, ordered=None):
    """lo, hi, value of np.quantile's method="linear" for the ranked sample e (value = lo where t = 0)."""
    n = len(e)
    h = (n - 1) * qs
    j = np.floor(h).astype(np.int64)
    j1 = np.minimum(j + 1, n - 1)
    if ordered is None:
        ordered = np.partition(e, np.unique(np.concatenate([j, j1])))
    lo, hi = ordered[j], ordered[j1]
    with np.errstate(invalid="ignore"):
        val = np.quantile(e, qs) if n < 50_000_000 else None
    if val is None:  # _lerp on the selected pair (np.quantile's own steps), for samples too large to copy again
        t = h - j
        d = hi - lo
        val = np.where(t >= 0.5, hi - d * (1 - t), lo + d * t)
    val = np.where(h - j == 0, lo, val)
    return lo, hi, val


def check(res, e, qs, O):
    lo, hi, val = expect(e, qs)
    assert res.n_ranked == len(e)
    assert np.array_equal(res.lo, lo) and np.array_equal(res.hi, hi)
    assert np.array_equal(res.values, val, equal_nan=True)
    med = expect(e, np.array([0.5]))[2][0]
    assert res.median == med or (np.isnan(res.median) and np.isnan(med))
    assert res.robust_sigma == np.sqrt(med / CHI2_MEDIAN[O]) or np.isnan(med)
    assert np.array_equal(res.norm_values, np.sqrt(val), equal_nan=True)


def raw_bytes(res):
    return bytes(res.raw)


# ---- every builtin model x (store, compute) pair, at ragged sizes ------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
@pytest.mark.parametrize("model", range(7))
def test_every_model_matches_numpy(env, model, sdt, cdt):
    capi, ctx = env
    _, x, k, consts = model_table(capi)[model]
    O = capi.MODEL_SHAPE[model][1]
    for n in SIZES:
        st, _, _ = make_store(capi, ctx, model, n, sdt, seed=n)
        prob = capi.make_problem(model, capi.JAC_FORWARD, cdt, loss=capi.LOSS_HUBER, loss_param=k, consts=consts)
        e = device_keys(capi, ctx, st, prob, x)
        res = ctx.quantiles(st, prob, x, QS)
        assert res.n_nan == 0
        check(res, e, QS, O)
        st.close()


@pytest.mark.parametrize("sdt,cdt", DTYPES)
@pytest.mark.parametrize("model", [0, 1, 6])
def test_ragged_sub_ranges(env, model, sdt, cdt):
    capi, ctx = env
    _, x, _, consts = model_table(capi)[model]
    n = 1_000_003
    st, _, _ = make_store(capi, ctx, model, n, sdt, seed=3)
    prob = capi.make_problem(model, capi.JAC_FORWARD, cdt, consts=consts)
    e = device_keys(capi, ctx, st, prob, x)
    for first, count in ((5, 333_331), (333_337, 1), (17, n - 20), (n - 3, 3), (1, 2), (123_457, 33)):
        res = ctx.quantiles(st, prob, x, QS, first=first, count=count)
        check(res, e[first:first + count], QS, capi.MODEL_SHAPE[model][1])
    st.close()


# ---- ties, +inf and NaN keys ------------------------------------------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
def test_ties(env, sdt, cdt):
    capi, ctx = env
    n = 1_000_000
    rng = np.random.default_rng(5)
    st = capi.Store(ctx, capi.MODEL_POINT_DIST, n, sdt)
    prob = capi.make_problem(capi.MODEL_POINT_DIST, compute_dtype=cdt)
    # every key equal
    st.upload(0, np.tile([1.0, 2.0, 3.0], (n, 1)))
    st.upload(1, np.tile([1.5, 1.25, 3.125], (n, 1)))
    e = device_keys(capi, ctx, st, prob, [])
    assert np.all(e == e[0]) and e[0] > 0
    res = ctx.quantiles(st, prob, [], QS)
    check(res, e, QS, 3)
    assert np.all(res.values == e[0])
    # 90 % exact zeros (p = q)
    p = rng.uniform(-1, 1, (n, 3))
    q = p.copy()
    far = rng.random(n) < 0.1
    q[far] += rng.uniform(-0.1, 0.1, (int(far.sum()), 3))
    st.upload(0, p)
    st.upload(1, q)
    e = device_keys(capi, ctx, st, prob, [])
    assert 0.85 < np.mean(e == 0) < 0.95
    res = ctx.quantiles(st, prob, [], QS)
    check(res, e, QS, 3)
    assert res.median == 0.0 and res.robust_sigma == 0.0 and res.values[-1] > 0
    st.close()


def test_inf_and_nan_keys(env):
    capi, ctx = env
    n = 100_003
    rng = np.random.default_rng(9)
    t = rng.uniform(0, 5, n)
    y = np.exp(0.3 * t + 0.1) + rng.normal(0, 0.2, n)
    big = rng.random(n) < 0.02
    y[big] = 3.0e38  # r ~ -3e38: r * r overflows to +inf in fp32
    nan = rng.random(n) < 0.01
    t[nan] = np.nan
    st = capi.Store(ctx, capi.MODEL_EXP_CURVE, n, capi.F32)
    st.upload(0, t)
    st.upload(1, y)
    prob = capi.make_problem(capi.MODEL_EXP_CURVE, compute_dtype=capi.F32)
    x = np.array([0.3, 0.1])
    e = device_keys(capi, ctx, st, prob, x)
    ranked = e[~np.isnan(e)]
    assert np.isinf(ranked).sum() == (big & ~nan).sum() > 0
    res = ctx.quantiles(st, prob, x, QS)
    assert res.n_nan == int(np.isnan(e).sum()) == int(nan.sum()) > 0
    assert res.n_ranked == n - res.n_nan
    check(res, ranked, QS, 1)
    assert res.lo[-1] == res.hi[-1] == res.values[-1] == np.inf  # q = 1: the largest key, +inf
    # q = 0.99 falls among the +inf keys at t > 0: numpy's lerp gives inf - inf = NaN, and so does the library
    assert res.lo[-2] == res.hi[-2] == np.inf and np.isnan(res.values[-2])
    st.close()


# ---- masked ICP stores, empty and all-masked ranges -------------------------------------------------------------
@pytest.mark.parametrize("dtype", [0, 1])
def test_masked_icp_store(env, dtype):
    from tests.test_icp import X_TRUE, clouds
    capi, ctx = env
    src, tgt = clouds()
    n = src.shape[0]
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, dtype)
    st.upload(0, src)
    ix = capi.NNIndex(ctx, tgt, 0.05, dtype=capi.F64)
    capi.store_set_target(st, ix)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, dtype)
    matched = capi.store_reassociate(st, X_TRUE)
    miss = np.isnan(st.download(1)[:, 0])
    assert 0 < miss.sum() < n and matched == n - miss.sum()
    e = device_keys(capi, ctx, st, prob, X_TRUE)
    res = ctx.quantiles(st, prob, X_TRUE, QS)
    assert res.n_nan == 0
    check(res, e[~miss], QS, 3)
    # never re-associates: at another x the store keeps the correspondences made at X_TRUE
    ctx.quantiles(st, prob, np.zeros(6), QS)
    assert np.array_equal(np.isnan(st.download(1)[:, 0]), miss)
    # all masked: nothing within 1e-9
    ix2 = capi.NNIndex(ctx, tgt, 1e-9, dtype=capi.F64)
    capi.store_set_target(st, ix2)
    assert capi.store_reassociate(st, X_TRUE) == 0
    for r in (ctx.quantiles(st, prob, X_TRUE, QS), ctx.quantiles(st, prob, X_TRUE, QS, first=7, count=0)):
        assert r.n_ranked == 0 and r.n_nan == 0
        assert np.isnan(r.lo).all() and np.isnan(r.hi).all() and np.isnan(r.values).all()
        assert np.isnan(r.median) and np.isnan(r.robust_sigma)
    capi.store_set_target(st, None)
    ix.close()
    ix2.close()
    st.close()


# ---- determinism, robust scale -----------------------------------------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
def test_bit_identical_across_calls_and_launch_shapes(env, sdt, cdt):
    capi, ctx = env
    _, x, _, consts = model_table(capi)[6]
    st, _, _ = make_store(capi, ctx, 6, 1_000_003, sdt, seed=2)
    prob = capi.make_problem(6, capi.JAC_FORWARD, cdt, consts=consts)
    a = raw_bytes(ctx.quantiles(st, prob, x, QS))
    assert raw_bytes(ctx.quantiles(st, prob, x, QS)) == a
    try:
        for shape in ((1, 0), (3, 0), (8, 0)):
            ctx.set_launch(*shape)
            assert raw_bytes(ctx.quantiles(st, prob, x, QS)) == a, shape
    finally:
        ctx.set_launch(0, 0)
    st.close()


def test_robust_sigma_ignores_outliers(env):
    capi, ctx = env
    n = 2_000_000
    sigma = 0.01
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F64)
    st.generate(seed=4, gt=X_P2P, noise_sigma=sigma, outlier_fraction=0.05, outlier_range=1.0)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64)
    res = ctx.quantiles(st, prob, X_P2P, [0.5])
    assert res.robust_sigma == np.sqrt(res.median / CHI2_MEDIAN[3])
    assert abs(res.robust_sigma - sigma) < 0.1 * sigma, res.robust_sigma
    rms = np.sqrt(ctx.compute_cost(st, prob, X_P2P) / (3 * n))
    assert rms > 3 * res.robust_sigma
    st.close()


# ---- user model, invalid arguments, one 100 M case --------------------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
def test_user_model_matches_builtin(env, sdt, cdt):
    from tests.test_gpu_evaluate import host_data
    from tests.test_user_model import EXP_CURVE_SRC
    capi, ctx = env
    um = capi.UserModel(EXP_CURVE_SRC, 2, 1, 1, 1, has_jacobian=True)
    x = np.array([0.3, 0.1])
    try:
        for n in (33, 1_000_003):
            a, b = host_data(capi, capi.MODEL_EXP_CURVE, n, seed=n)
            su = capi.Store(ctx, um.model, n, sdt)
            sb = capi.Store(ctx, capi.MODEL_EXP_CURVE, n, sdt)
            for s in (su, sb):
                s.upload(0, a)
                s.upload(1, b)
            ru = ctx.quantiles(su, capi.make_problem(um.model, capi.JAC_FORWARD, cdt), x, QS)
            rb = ctx.quantiles(sb, capi.make_problem(capi.MODEL_EXP_CURVE, capi.JAC_FORWARD, cdt), x, QS)
            assert raw_bytes(ru) == raw_bytes(rb)
            check(ru, device_keys(capi, ctx, su, capi.make_problem(um.model, capi.JAC_FORWARD, cdt), x), QS, 1)
            su.close()
            sb.close()
    finally:
        um.release()


def test_invalid_arguments_write_nothing(env):
    capi, ctx = env
    n = 1000
    st, _, _ = make_store(capi, ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    other_ctx = capi.Context(0)
    other, _, _ = make_store(capi, other_ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    prob = capi.make_problem(capi.MODEL_POINT2POINT)
    xs = np.zeros(6)
    out = capi.QuantilesStruct()
    out.n_ranked, out.median = -5, -7.25
    sentinel = bytes(out)

    def call(store=st, problem=prob, x=xs, first=0, count=n, q=(0.5,), n_q=None, o=C.byref(out)):
        qa = np.ascontiguousarray(np.asarray(q, dtype=np.float64)) if q is not None else None
        nq = (len(qa) if qa is not None else 0) if n_q is None else n_q
        return capi.lib().mopt_residual_quantiles(ctx.handle, store.handle, C.byref(problem),
                                                  capi._dp(x) if x is not None else None, first, count, nq,
                                                  capi._dp(qa) if qa is not None else None, o)

    bad = [
        dict(store=other),                                    # a store of another context
        dict(problem=capi.make_problem(capi.MODEL_EXP_CURVE)),  # a problem the store does not accept
        dict(first=-1, count=10), dict(first=0, count=n + 1), dict(first=n - 5, count=6), dict(count=-1),
        dict(q=np.full(9, 0.5)),                              # n_q > MOPT_MAX_QUANTILES
        dict(n_q=-1),
        dict(q=(0.5, np.nan)), dict(q=(-1e-300,)), dict(q=(1.0 + 2e-16,)), dict(q=(np.inf,)),
        dict(q=None, n_q=2),                                  # null q with n_q > 0
        dict(o=None),                                         # null out
        dict(x=None),                                         # null x for a model with parameters
    ]
    for kw in bad:
        assert call(**kw) == 1, kw  # MOPT_ERR_INVALID_ARGUMENT
        assert bytes(out) == sentinel, kw
    # n_q = 0 with a null q is fine: the median alone
    assert call(q=None) == 0 and out.n_ranked == n and not np.isnan(out.median)
    with pytest.raises(ValueError):
        ctx.quantiles(st, prob, xs, np.linspace(0, 1, 9))
    other.close()
    other_ctx.close()
    st.close()


def test_point2point_100m_fp32(env):
    capi, ctx = env
    n = 100_000_000
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    st.generate(seed=1, gt=X_P2P, noise_sigma=0.01, outlier_fraction=0.05, outlier_range=1.0)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32)
    x = X_P2P + 1e-3
    q = np.array([0.5, 0.9, 0.99])
    res = ctx.quantiles(st, prob, x, q)
    e = device_keys(capi, ctx, st, prob, x)
    lo, hi, val = expect(e, q)
    assert res.n_ranked == n and res.n_nan == 0
    assert np.array_equal(res.lo, lo) and np.array_equal(res.hi, hi) and np.array_equal(res.values, val)
    assert res.median == val[0]
    st.close()
