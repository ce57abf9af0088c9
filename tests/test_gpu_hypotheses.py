"""Hypothesis scoring on the device (mopt_score_hypotheses / Context.score_hypotheses) against mopt_evaluate called
once per hypothesis: counts and max_sq exactly, the sums to 1e-12 relative (the same fp64 values added in another
order), for every builtin model with parameters and dtype pair.  Then batch independence, edges, user models,
argument validation, RANSAC end to end and one 100 M case."""
import ctypes as C

import numpy as np
import pytest

from tests.test_gpu_evaluate import DTYPES, SIZES, X_P2P, make_store, model_table

pytestmark = pytest.mark.gpu

MODELS = [0, 1, 2, 3, 4, 6]  # every builtin model with parameters (point_dist has none)


@pytest.fixture(scope="module")
def env():
    from moptimizer_0_b200 import capi
    c = capi.Context(0)
    yield capi, c
    c.close()


def eval_stats(ctx, st, prob, x, thr, first=0, count=None):
    return ctx.evaluate(st, prob, x, first=first, count=count, inlier_threshold=thr, residuals=False,
                        weights=False).stats


def hypotheses(x, K, seed, rel=0.01, absolute=1e-3):
    rng = np.random.default_rng(seed)
    return x + rng.normal(0, 1, (K, len(x))) * (rel * np.abs(x) + absolute)


def check_against_evaluate(ctx, st, prob, xs, thr, first=0, count=None):
    sc = ctx.score_hypotheses(st, prob, xs, thr, first=first, count=count)
    for k, x in enumerate(xs):
        ref = eval_stats(ctx, st, prob, x, thr, first, count)
        assert sc.n_valid[k] == ref["n_valid"], k
        assert sc.n_inliers[k] == ref["n_inliers"], k
        assert sc.max_sq[k] == ref["max_sq"] or (np.isnan(sc.max_sq[k]) and np.isnan(ref["max_sq"])), k
        for f in ("sum_sq", "inlier_sum_sq"):
            a, b = getattr(sc, f)[k], ref[f]
            assert a == b or abs(a - b) <= 1e-12 * abs(b) or (np.isnan(a) and np.isnan(b)), (k, f, a, b)
    return sc


def split_threshold(ctx, st, prob, x):
    """The RMS residual norm at x: a threshold that puts part of the data on either side."""
    s = eval_stats(ctx, st, prob, x, np.inf)
    return float(np.sqrt(s["sum_sq"] / max(s["n_valid"], 1)))


# ---- agreement with mopt_evaluate ----------------------------------------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
@pytest.mark.parametrize("model", MODELS)
def test_every_model_agrees_with_evaluate(env, model, sdt, cdt):
    capi, ctx = env
    _, x, _, consts = model_table(capi)[model]
    rel, ab = (0.2, 0.1) if model == capi.MODEL_POWELL else (0.01, 1e-3)
    for n in SIZES:
        st, _, _ = make_store(capi, ctx, model, n, sdt, seed=n)
        prob = capi.make_problem(model, capi.JAC_FORWARD, cdt, consts=consts)
        thr = split_threshold(ctx, st, prob, x)
        Ks = (1, 5, 32, 33) + ((300,) if n == SIZES[-1] and model in (0, 3) else ())
        for K in Ks:
            check_against_evaluate(ctx, st, prob, hypotheses(x, K, seed=K + n, rel=rel, absolute=ab), thr)
        st.close()


# ---- batch independence and determinism -----------------------------------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
def test_batch_independence(env, sdt, cdt):
    capi, ctx = env
    _, x, _, _ = model_table(capi)[0]
    st, _, _ = make_store(capi, ctx, 0, 1_000_003, sdt, seed=5)
    prob = capi.make_problem(0, capi.JAC_ANALYTICAL, cdt)
    xs = hypotheses(x, 70, seed=6)
    thr = split_threshold(ctx, st, prob, x)
    full = ctx.score_hypotheses(st, prob, xs, thr)

    def same_counts(sc, idx):
        for f in ("n_valid", "n_inliers", "max_sq"):
            assert np.array_equal(getattr(sc, f), getattr(full, f)[idx]), f

    for k in (0, 31, 32, 69):  # alone
        same_counts(ctx.score_hypotheses(st, prob, xs[k:k + 1], thr), [k])
    rev = np.arange(69, -1, -1)
    same_counts(ctx.score_hypotheses(st, prob, xs[rev], thr), rev)
    for cuts in ((1, 6, 38), (33,), (5, 10, 15, 20, 50)):
        parts = np.split(np.arange(70), cuts)
        for p in parts:
            same_counts(ctx.score_hypotheses(st, prob, xs[p], thr), p)
    # every output bit-identical between two identical calls
    again = ctx.score_hypotheses(st, prob, xs, thr)
    for f in ("n_valid", "n_inliers", "sum_sq", "inlier_sum_sq", "max_sq"):
        assert getattr(again, f).tobytes() == getattr(full, f).tobytes(), f
    try:
        for shape in ((1, 0), (3, 0), (8, 0)):
            ctx.set_launch(*shape)
            same_counts(ctx.score_hypotheses(st, prob, xs, thr), np.arange(70))
    finally:
        ctx.set_launch(0, 0)
    st.close()


# ---- edges -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
def test_key_equal_to_threshold_is_an_inlier(env, sdt, cdt):
    capi, ctx = env
    n = 1001
    rng = np.random.default_rng(7)
    p = np.round(rng.uniform(0, 8, (n, 3)) * 64) / 64  # exact in fp32
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, sdt)
    st.upload(0, p)
    st.upload(1, p + np.array([0.5, 0.0, 0.0]))  # identity hypothesis: r = (-0.5, 0, 0), e2 = 0.25 exactly
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, cdt)
    xs = np.vstack([np.zeros(6), hypotheses(X_P2P, 4, seed=8)])
    sc = check_against_evaluate(ctx, st, prob, xs, 0.5)
    assert sc.n_inliers[0] == n and sc.max_sq[0] == 0.25 and sc.inlier_sum_sq[0] == 0.25 * n
    below = ctx.score_hypotheses(st, prob, xs[:1], float(np.nextafter(0.5, 0.0)))
    assert below.n_inliers[0] == 0
    st.close()


def test_infinite_threshold_ragged_ranges_and_empty_range(env):
    capi, ctx = env
    n = 1_000_003
    _, x, _, _ = model_table(capi)[0]
    st, _, _ = make_store(capi, ctx, 0, n, capi.F32, seed=9)
    prob = capi.make_problem(0, capi.JAC_ANALYTICAL, capi.F32)
    xs = hypotheses(x, 40, seed=10)
    sc = ctx.score_hypotheses(st, prob, xs, np.inf)
    assert (sc.n_inliers == n).all() and (sc.n_valid == n).all()
    thr = split_threshold(ctx, st, prob, x)
    for first, count in ((5, 333_331), (333_337, 1), (17, n - 20), (n - 3, 3), (1, 2), (123_457, 33)):
        check_against_evaluate(ctx, st, prob, xs[:9], thr, first, count)
    empty = ctx.score_hypotheses(st, prob, xs, thr, first=7, count=0)
    for f in ("n_valid", "n_inliers", "sum_sq", "inlier_sum_sq", "max_sq"):
        assert (getattr(empty, f) == 0).all(), f
    st.close()


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
    assert 0 < matched < n
    xs = np.vstack([X_TRUE, hypotheses(np.asarray(X_TRUE, dtype=np.float64), 20, seed=11)])
    sc = check_against_evaluate(ctx, st, prob, xs, 0.02)
    assert (sc.n_valid == matched).all()
    ix2 = capi.NNIndex(ctx, tgt, 1e-9, dtype=capi.F64)  # all masked
    capi.store_set_target(st, ix2)
    assert capi.store_reassociate(st, X_TRUE) == 0
    sc = check_against_evaluate(ctx, st, prob, xs, 0.02)
    assert (sc.n_valid == 0).all() and (sc.max_sq == 0).all() and (sc.sum_sq == 0).all()
    capi.store_set_target(st, None)
    ix.close()
    ix2.close()
    st.close()


def test_nan_hypothesis_leaves_the_others_alone(env):
    capi, ctx = env
    _, x, _, _ = model_table(capi)[0]
    st, _, _ = make_store(capi, ctx, 0, 1_000_003, capi.F32, seed=12)
    prob = capi.make_problem(0, capi.JAC_ANALYTICAL, capi.F32)
    xs = hypotheses(x, 64, seed=13)
    thr = split_threshold(ctx, st, prob, x)
    clean = ctx.score_hypotheses(st, prob, xs, thr)
    bad = xs.copy()
    bad[17, 4] = np.nan
    sc = check_against_evaluate(ctx, st, prob, bad, thr)
    keep = np.arange(64) != 17
    for f in ("n_valid", "n_inliers", "max_sq"):
        assert np.array_equal(getattr(sc, f)[keep], getattr(clean, f)[keep]), f
    st.close()


# ---- user models -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
def test_user_models(env, sdt, cdt):
    from tests.test_gpu_evaluate import host_data
    from tests.test_user_model import EXP_CURVE_SRC, P2P_SRC
    capi, ctx = env
    ue = capi.UserModel(EXP_CURVE_SRC, 2, 1, 1, 1, has_jacobian=True)
    up = capi.UserModel(P2P_SRC, 6, 3, 3, 3, set_size=12, rot_offset=3)
    try:
        for n in (33, 1_000_003):
            x = np.array([0.3, 0.1])
            xs = hypotheses(x, 37, seed=n)
            a, b = host_data(capi, capi.MODEL_EXP_CURVE, n, seed=n)
            su, sb = capi.Store(ctx, ue.model, n, sdt), capi.Store(ctx, capi.MODEL_EXP_CURVE, n, sdt)
            for s in (su, sb):
                s.upload(0, a)
                s.upload(1, b)
            pu = capi.make_problem(ue.model, capi.JAC_FORWARD, cdt)
            pb = capi.make_problem(capi.MODEL_EXP_CURVE, capi.JAC_FORWARD, cdt)
            thr = split_threshold(ctx, sb, pb, x)
            ru = check_against_evaluate(ctx, su, pu, xs, thr)
            rb = ctx.score_hypotheses(sb, pb, xs, thr)
            for f in ("n_valid", "n_inliers", "sum_sq", "inlier_sum_sq", "max_sq"):
                assert getattr(ru, f).tobytes() == getattr(rb, f).tobytes(), f
            su.close()
            sb.close()
            a, b = host_data(capi, capi.MODEL_POINT2POINT, n, seed=n)
            sp = capi.Store(ctx, up.model, n, sdt)
            sp.upload(0, a)
            sp.upload(1, b)
            pp = capi.make_problem(up.model, capi.JAC_FORWARD, cdt)
            check_against_evaluate(ctx, sp, pp, hypotheses(X_P2P, 37, seed=n + 1), split_threshold(ctx, sp, pp, X_P2P))
            sp.close()
    finally:
        ue.release()
        up.release()


# ---- invalid arguments -------------------------------------------------------------------------------------------
def test_invalid_arguments_write_nothing(env):
    capi, ctx = env
    n = 1000
    st, _, _ = make_store(capi, ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    other_ctx = capi.Context(0)
    other, _, _ = make_store(capi, other_ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    dist = capi.Store(ctx, capi.MODEL_POINT_DIST, n, capi.F32)
    prob = capi.make_problem(capi.MODEL_POINT2POINT)
    xs = np.zeros((4, 6))
    out = (capi.EvalStats * 4)()
    for k in range(4):
        out[k].n_valid, out[k].max_sq = -5, -7.25
    sentinel = bytes(out)

    def call(store=st, problem=prob, n_hyp=4, x=xs, first=0, count=n, thr=0.1, o=out):
        return capi.lib().mopt_score_hypotheses(ctx.handle, store.handle, C.byref(problem), n_hyp,
                                                capi._dp(x) if x is not None else None, first, count, thr,
                                                o if o is not None else None)

    bad = [
        dict(n_hyp=0), dict(n_hyp=-1), dict(n_hyp=capi.MAX_HYPOTHESES + 1),
        dict(x=None), dict(o=None),
        dict(store=dist, problem=capi.make_problem(capi.MODEL_POINT_DIST)),  # a model without parameters
        dict(store=other),                                                   # a store of another context
        dict(problem=capi.make_problem(capi.MODEL_EXP_CURVE)),               # a problem the store does not accept
        dict(first=-1, count=10), dict(first=0, count=n + 1), dict(first=n - 5, count=6), dict(count=-1),
        dict(thr=-1e-300), dict(thr=-np.inf),
    ]
    for kw in bad:
        assert call(**kw) == 1, kw  # MOPT_ERR_INVALID_ARGUMENT
        assert bytes(out) == sentinel, kw
    assert call() == 0 and out[0].n_valid == n
    dist.close()
    other.close()
    other_ctx.close()
    st.close()


# ---- RANSAC end to end, full size ---------------------------------------------------------------------------------
def kabsch(p, q):
    """R, t minimising sum |R p + t - q|^2, as x = [t, rotation vector]."""
    from scipy.spatial.transform import Rotation
    pc, qc = p.mean(0), q.mean(0)
    U, _, Vt = np.linalg.svd((p - pc).T @ (q - qc))
    d = np.sign(np.linalg.det(Vt.T @ U.T))
    R = Vt.T @ np.diag([1.0, 1.0, d]) @ U.T
    return np.concatenate([qc - R @ pc, Rotation.from_matrix(R).as_rotvec()])


def test_ransac_end_to_end(env):
    capi, ctx = env
    n = 1_000_003
    x_gt = np.array([0.5, -0.3, 0.2, 1.2, -1.0, 1.2])  # |omega| = 1.97 rad
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    st.generate(seed=14, gt=x_gt, noise_sigma=0.01, outlier_fraction=0.6, outlier_range=10.0)
    src, tgt = st.download(0), st.download(1)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32)
    rng = np.random.default_rng(15)
    xs = np.array([kabsch(src[i], tgt[i]) for i in (rng.choice(n, 3, replace=False) for _ in range(512))])
    thr = 0.05
    sc = ctx.score_hypotheses(st, prob, xs, thr)
    ref = np.array([eval_stats(ctx, st, prob, x, thr)["n_inliers"] for x in xs])
    assert np.array_equal(sc.n_inliers, ref)
    best = int(np.argmax(sc.n_inliers))
    assert best == int(np.argmax(ref))
    at_gt = eval_stats(ctx, st, prob, x_gt, thr)["n_inliers"]
    assert sc.n_inliers[best] >= 0.95 * at_gt, (sc.n_inliers[best], at_gt)
    huber = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64, loss=capi.LOSS_HUBER,
                              loss_param=thr)
    res = ctx.lm_minimize([st], [huber], xs[best], max_iterations=50)
    assert np.max(np.abs(res.x - x_gt)) < 1e-3, (res.x, res.status)
    st.close()


def test_point2point_100m_fp32(env):
    capi, ctx = env
    n = 100_000_000
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    st.generate(seed=1, gt=X_P2P, noise_sigma=0.01, outlier_fraction=0.05, outlier_range=1.0)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32)
    xs = hypotheses(X_P2P, 64, seed=16, rel=0.002, absolute=1e-3)
    check_against_evaluate(ctx, st, prob, xs, 0.03)
    st.close()
