"""Parameter covariance on the device (mopt_covariance_terms / Context.covariance): the score Gram sums of every
builtin model against the reference loops with the score accumulated (tests/oracle_covariance.cpp), agreement with
mopt_linearize, additivity over split stores and cost terms, masked ICP stores, statistical validity of the SCALED and
SANDWICH estimators over repeated synthetic registrations, rank deficiency, the calibration model, a run-time compiled
user model, argument validation and one 100 M case."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle_py as orc
from tests import oracle_covariance as ocov
from tests.common import camera_consts
from tests.test_gpu_evaluate import DTYPES, X_P2P, make_store, model_table

pytestmark = pytest.mark.gpu

SIZES = (1, 31, 33, 1_000_003)
LOSSES = [(0, 0.0), (1, None), (2, None)]
MODELS = [0, 1, 2, 3, 4, 6]  # every builtin model with parameters
COV3 = np.array([[2.0, 0.3, 0.1], [0.3, 1.5, -0.2], [0.1, -0.2, 0.7]])
COV2 = np.array([[1.5, 0.2], [0.2, 0.8]])


@pytest.fixture(scope="module")
def env():
    from moptimizer_0_b200 import capi
    c = capi.Context(0)
    yield capi, c
    c.close()


def fro_err(A, B):
    return float(np.linalg.norm(A - B) / max(np.linalg.norm(B), 1e-300))


def g_tol(model, jac, f32):
    """Bound on |G - G_oracle|_F / |G_oracle|_F.
    fp64 compute, analytical Jacobian: 1e-10, the two differ by the order of fp64 sums.
    fp64 finite differences: both sides form the literal quotient (r(x + h e_j) - r(x)) / h_j, h_j = sqrt(eps) |x_j|,
    from parameter sets that round differently on the device and in the oracle; the quotient amplifies that rounding
    by 1/h_j.  tests/test_gpu_parity.py holds H of these paths to 1e-6, and so is G here -- except for the camera
    models: a rotation component of 1.3e-3 gives h_j = 2e-11, and the ~1e-13 rounding of a ~1e3-pixel projection then
    moves a Jacobian entry by ~5e-6 of its size; G is quadratic in J and a single element (n = 1) averages nothing
    (1.4e-5 measured on a B200), so 1e-4 for those.
    fp32 compute (against the fp64 oracle): G is quadratic in the score w J^T C r, whose fp32 residual carries
    eps_f32 of the data's magnitude -- up to ~1e-3 of a 0.3-pixel residual of a ~1e3-pixel projection -- so the
    relative error of G is up to twice that for a single element and averages down over many; 2e-2 bounds the
    smallest sizes.  (tests/test_gpu_parity.py holds fp32 finite-difference H to 5e-3 on fachada.)"""
    if f32:
        return 2e-2
    if jac == 0:
        return 1e-10
    return 1e-4 if model in (3, 6) else 1e-6


def jac_modes(capi, model):
    """The Jacobian modes the model supports (the camera models have no analytical one)."""
    analytical = model in (capi.MODEL_POINT2POINT, capi.MODEL_EXP_CURVE, capi.MODEL_MICHAELIS_MENTEN, capi.MODEL_POWELL)
    return ([capi.JAC_ANALYTICAL] if analytical else []) + [capi.JAC_FORWARD, capi.JAC_CENTRAL]


def oracle_cost(capi, model, n, a, b, jac, loss, k, cov=None):
    kind, _, _, consts = model_table(capi)[model]
    P, O, _, _ = capi.MODEL_SHAPE[model]
    return orc.Cost(kind, P, O, n, a=a, b=b, consts=consts, jac_mode=jac, loss=loss, loss_param=k, cov=cov)


# ---- 1. oracle parity of G, wsse and n_valid ----------------------------------------------------------------------
@pytest.mark.parametrize("loss,kp", LOSSES)
@pytest.mark.parametrize("sdt,cdt", DTYPES)
@pytest.mark.parametrize("model", MODELS)
def test_parity_with_oracle(env, model, sdt, cdt, loss, kp):
    capi, ctx = env
    _, x, scale_k, consts = model_table(capi)[model]
    k = scale_k if kp is None else kp
    O = capi.MODEL_SHAPE[model][1]
    for n in SIZES:
        # the data-free Powell pass adds its n identical blocks serially in the compute dtype (as the pass does)
        if model == capi.MODEL_POWELL and n > 33:
            continue
        st, a, b = make_store(capi, ctx, model, n, sdt, seed=n)
        for jac in jac_modes(capi, model):
            prob = capi.make_problem(model, jac, cdt, loss=loss, loss_param=k, consts=consts)
            t = ctx.covariance_terms([st], [prob], x)
            Go, qo, no = ocov.score_gram(oracle_cost(capi, model, n, a, b, jac, loss, k), x)
            assert t.n_valid == no == n and t.m == n * O
            tol = g_tol(model, jac, cdt == capi.F32)
            assert fro_err(t.G, Go) <= tol, (model, jac, n, fro_err(t.G, Go))
            assert abs(t.wsse - qo) <= max(tol, 1e-12) * abs(qo), (model, jac, n, t.wsse, qo)
        st.close()


@pytest.mark.parametrize("sdt,cdt", DTYPES)
@pytest.mark.parametrize("model", [0, 3])
def test_parity_with_covariance_matrix(env, model, sdt, cdt):
    capi, ctx = env
    _, x, scale_k, consts = model_table(capi)[model]
    cov = COV3 if model == capi.MODEL_POINT2POINT else COV2
    for n in (33, 1_000_003):
        st, a, b = make_store(capi, ctx, model, n, sdt, seed=n + 1)
        for jac in jac_modes(capi, model):
            prob = capi.make_problem(model, jac, cdt, loss=capi.LOSS_HUBER, loss_param=scale_k, consts=consts,
                                     covariance=cov)
            t = ctx.covariance_terms([st], [prob], x)
            Go, qo, no = ocov.score_gram(oracle_cost(capi, model, n, a, b, jac, capi.LOSS_HUBER, scale_k, cov), x)
            tol = g_tol(model, jac, cdt == capi.F32)
            assert t.n_valid == no and fro_err(t.G, Go) <= tol and abs(t.wsse - qo) <= max(tol, 1e-12) * abs(qo)
        st.close()


# ---- 2. agreement with the existing pass, determinism -------------------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
@pytest.mark.parametrize("model", MODELS)
def test_h_b_sum_are_mopt_linearize_bits(env, model, sdt, cdt):
    capi, ctx = env
    _, x, scale_k, consts = model_table(capi)[model]
    n = 1000 if model == capi.MODEL_POWELL else 100_003
    st, _, _ = make_store(capi, ctx, model, n, sdt, seed=3)
    for jac in jac_modes(capi, model):
        prob = capi.make_problem(model, jac, cdt, loss=capi.LOSS_HUBER, loss_param=scale_k, consts=consts)
        t1 = ctx.covariance_terms([st], [prob], x)
        H, b, s = ctx.linearize(st, prob, x)
        assert np.array_equal(t1.H, H) and np.array_equal(t1.b, b) and t1.sum_sq == s
        t2 = ctx.covariance_terms([st], [prob], x)
        assert bytes(t1.raw) == bytes(t2.raw)
    st.close()


# ---- 3. additivity (stands in for sharding on one GPU) ------------------------------------------------------------
def test_split_stores_and_cost_terms_add(env):
    capi, ctx = env
    n, cut = 1_000_003, 400_001
    whole, a, b = make_store(capi, ctx, capi.MODEL_POINT2POINT, n, capi.F64, seed=9)
    parts = []
    for lo, hi in ((0, cut), (cut, n)):
        s = capi.Store(ctx, capi.MODEL_POINT2POINT, hi - lo, capi.F64)
        s.upload(0, a[lo:hi])
        s.upload(1, b[lo:hi])
        parts.append(s)
    for jac in (capi.JAC_ANALYTICAL, capi.JAC_CENTRAL):
        prob = capi.make_problem(capi.MODEL_POINT2POINT, jac, capi.F64, loss=capi.LOSS_HUBER, loss_param=0.05)
        tw = ctx.covariance_terms([whole], [prob], X_P2P)
        ts = ctx.covariance_terms([parts[0]], [prob], X_P2P) + ctx.covariance_terms([parts[1]], [prob], X_P2P)
        assert ts.n_valid == tw.n_valid == n and ts.m == tw.m == 3 * n
        for f in ("H", "G", "b"):
            assert fro_err(getattr(ts, f), getattr(tw, f)) <= 1e-12, f
        assert ts.wsse == pytest.approx(tw.wsse, rel=1e-12) and ts.sum_sq == pytest.approx(tw.sum_sq, rel=1e-12)
        # two cost terms in one call: the sum of their separate terms
        p2 = capi.make_problem(capi.MODEL_POINT2POINT, jac, capi.F64, loss=capi.LOSS_GEMAN_MCCLURE, loss_param=0.02)
        both = ctx.covariance_terms([parts[0], parts[1]], [prob, p2], X_P2P)
        sep = ctx.covariance_terms([parts[0]], [prob], X_P2P) + ctx.covariance_terms([parts[1]], [p2], X_P2P)
        assert both.n_valid == sep.n_valid and both.m == sep.m
        for f in ("H", "G", "b"):
            assert fro_err(getattr(both, f), getattr(sep, f)) <= 1e-12, f
        assert both.wsse == pytest.approx(sep.wsse, rel=1e-12)
    for s in parts + [whole]:
        s.close()


# ---- 4. masked ICP store ------------------------------------------------------------------------------------------
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
    sq, tq = st.download(0), st.download(1)
    keep = ~np.isnan(tq[:, 0])
    assert 0 < matched < n
    t = ctx.covariance_terms([st], [prob], X_TRUE)
    assert t.n_valid == matched == int(keep.sum()) and t.m == 3 * matched
    dense = capi.Store(ctx, capi.MODEL_POINT2POINT, matched, dtype)
    dense.upload(0, sq[keep])
    dense.upload(1, tq[keep])
    td = ctx.covariance_terms([dense], [prob], X_TRUE)
    tol = 1e-12 if dtype == capi.F64 else 1e-5  # same elements, other grid: fp32 partial sums fold differently
    assert td.n_valid == t.n_valid
    for f in ("H", "G", "b"):
        assert fro_err(getattr(t, f), getattr(td, f)) <= tol, f
    assert t.wsse == pytest.approx(td.wsse, rel=tol)
    # never re-associates: the store still holds the correspondences made at X_TRUE
    ctx.covariance_terms([st], [prob], np.zeros(6))
    assert np.array_equal(np.isnan(st.download(1)[:, 0]), ~keep)
    capi.store_set_target(st, None)
    ix.close()
    dense.close()
    st.close()


# ---- 5. statistical validity ----------------------------------------------------------------------------------------
K_TRIALS, N_POINTS = 200, 10_000
GT = np.array([0.3, -0.2, 0.1, 0.05, -0.04, 0.03])


def solve_and_predict(capi, ctx, st, estimator, dtype=1):
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, dtype)
    r = ctx.lm_minimize([st], [prob], np.zeros(6), max_iterations=30)
    return r.x, ctx.covariance([st], [prob], r.x, estimator).cov


def ratios(xs, covs):
    emp = np.var(np.array(xs), axis=0, ddof=1)
    pred = np.mean(np.array([np.diag(c) for c in covs]), axis=0)
    return emp / pred


def test_scaled_covariance_matches_repeated_fits(env):
    capi, ctx = env
    xs, covs = [], []
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, N_POINTS, capi.F64)
    for k in range(K_TRIALS):
        st.generate(seed=1000 + k, gt=GT, noise_sigma=0.01)
        x, cv = solve_and_predict(capi, ctx, st, capi.COV_SCALED)
        xs.append(x)
        covs.append(cv)
    st.close()
    q = ratios(xs, covs)
    assert np.all((q >= 0.7) & (q <= 1.4)), q  # +-3 standard errors of a variance ratio at K = 200


def test_sandwich_covariance_under_heteroscedastic_noise(env):
    """Noise std grows with the 6th power of the distance from the centroid: the rotation is fixed by the far,
    noisy points, which SCALED (one pooled noise level) under-weights by ~1.9x on the rotation block."""
    capi, ctx = env
    rng = np.random.default_rng(77)
    T = orc.so3_convert6dof(GT)
    xs, cs, cw = [], [], []
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, N_POINTS, capi.F64)
    for _ in range(K_TRIALS):
        src = rng.uniform(0, 10, (N_POINTS, 3))
        d = np.linalg.norm(src - src.mean(axis=0), axis=1)
        sig = 0.001 + 0.03 * (d / d.max()) ** 6
        tgt = src @ T[:3, :3].T + T[:3, 3] + rng.normal(size=(N_POINTS, 3)) * sig[:, None]
        st.upload(0, src)
        st.upload(1, tgt)
        prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64)
        r = ctx.lm_minimize([st], [prob], np.zeros(6), max_iterations=30)
        terms = ctx.covariance_terms([st], [prob], r.x)
        xs.append(r.x)
        cs.append(capi.covariance_from_terms(terms, capi.COV_SCALED).cov)
        cw.append(capi.covariance_from_terms(terms, capi.COV_SANDWICH).cov)
    st.close()
    qw, qs = ratios(xs, cw), ratios(xs, cs)
    assert np.all((qw >= 0.7) & (qw <= 1.4)), qw
    assert np.all(qs[3:] >= 1.5), qs


# ---- 6. rank deficiency -------------------------------------------------------------------------------------------
def test_collinear_points_are_rank_five(env):
    capi, ctx = env
    rng = np.random.default_rng(5)
    n = 5000
    u = rng.uniform(-5, 5, n)
    src = np.outer(u, [1.0, 2.0, 0.5]) + np.array([1.0, 2.0, 3.0])  # one line: rotation about it is unobservable
    T = orc.so3_convert6dof(GT)
    tgt = src @ T[:3, :3].T + T[:3, 3] + rng.normal(0, 0.01, (n, 3))
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F64)
    st.upload(0, src)
    st.upload(1, tgt)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64)
    t = ctx.covariance_terms([st], [prob], GT)
    res = capi.covariance_from_terms(t, capi.COV_SCALED)
    assert res.rank == 5 and res.dof == 3 * n - 5 and np.isfinite(res.cov).all()
    dg = np.diag(t.H)
    D = 1.0 / np.sqrt(dg)
    lam, V = np.linalg.eigh(D[:, None] * t.H * D[None, :])
    w = V[:, 0] / D  # D^-1 v for the null vector v of S
    assert np.linalg.norm(res.cov @ w) <= 1e-6 * np.linalg.norm(res.cov) * np.linalg.norm(w)
    st.close()


# ---- 7. pinhole + distortion, fp32 vs fp64 compute ----------------------------------------------------------------
def test_pinhole_distort_fp32_std_matches_fp64(env):
    capi, ctx = env
    _, x, _, consts = model_table(capi)[capi.MODEL_PINHOLE_DISTORT]
    st, _, _ = make_store(capi, ctx, capi.MODEL_PINHOLE_DISTORT, 1_000_000, capi.F32, seed=11)
    s = {}
    # fp64 with MOPT_FLAG_STABLE_FD: the same common-denominator quotient fp32 compute takes by default, so the two
    # differ by fp32 rounding only (the literal fp64 quotient carries its own 1/h-amplified noise, see g_tol)
    for cdt, flags in ((capi.F32, 0), (capi.F64, capi.FLAG_STABLE_FD)):
        prob = capi.make_problem(capi.MODEL_PINHOLE_DISTORT, capi.JAC_CENTRAL, cdt, consts=consts, flags=flags)
        s[cdt] = ctx.covariance([st], [prob], x, capi.COV_SCALED, rcond=1e-12).std
    assert np.all(s[capi.F32] > 0) and np.all(s[capi.F64] > 0)
    # tests/test_gpu_parity.py holds the fp32 common-denominator H of the camera to 2e-4 of the fp64 one.  A standard
    # deviation is the square root of a diagonal entry of the inverse, so that difference reaches it amplified by the
    # correlation of the parameters: the rotation and the distortion coefficients move most (2.9e-4 on a B200).
    assert np.max(np.abs(s[capi.F32] / s[capi.F64] - 1)) <= 1e-3, s
    st.close()


# ---- 8. run-time compiled user model --------------------------------------------------------------------------------
@pytest.mark.parametrize("sdt,cdt", DTYPES)
def test_user_model_matches_builtin(env, sdt, cdt):
    from tests.test_user_model import EXP_CURVE_SRC
    capi, ctx = env
    um = capi.UserModel(EXP_CURVE_SRC, 2, 1, 1, 1, has_jacobian=True)
    x = np.array([0.3, 0.1])
    try:
        for n in (33, 1_000_003):
            sb, a, b = make_store(capi, ctx, capi.MODEL_EXP_CURVE, n, sdt, seed=n)
            su = capi.Store(ctx, um.model, n, sdt)
            su.upload(0, a)
            su.upload(1, b)
            # the builtin exp curve takes common-denominator differences with fp32 compute: compare the same form
            for jac in (capi.JAC_ANALYTICAL, capi.JAC_FORWARD, capi.JAC_CENTRAL):
                fl = capi.FLAG_GENERIC_KERNEL if jac != capi.JAC_ANALYTICAL else 0
                pu = capi.make_problem(um.model, jac, cdt, loss=capi.LOSS_HUBER, loss_param=0.2)
                pb = capi.make_problem(capi.MODEL_EXP_CURVE, jac, cdt, loss=capi.LOSS_HUBER, loss_param=0.2, flags=fl)
                tu = ctx.covariance_terms([su], [pu], x)
                tb = ctx.covariance_terms([sb], [pb], x)
                tol = 1e-12 if cdt == capi.F64 else 1e-5
                assert tu.n_valid == tb.n_valid == n
                assert fro_err(tu.G, tb.G) <= tol and fro_err(tu.H, tb.H) <= tol, (jac, fro_err(tu.G, tb.G))
                assert tu.wsse == pytest.approx(tb.wsse, rel=tol)
            su.close()
            sb.close()
    finally:
        um.release()


# ---- 9. argument validation ---------------------------------------------------------------------------------------
def test_invalid_arguments_write_nothing(env):
    capi, ctx = env
    st, _, _ = make_store(capi, ctx, capi.MODEL_POINT2POINT, 100, capi.F64)
    sc, _, _ = make_store(capi, ctx, capi.MODEL_EXP_CURVE, 100, capi.F64)
    sd = capi.Store(ctx, capi.MODEL_POINT_DIST, 100, capi.F64)
    other = capi.Context(0)
    so = capi.Store(other, capi.MODEL_POINT2POINT, 100, capi.F64)
    pp = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64)
    pc = capi.make_problem(capi.MODEL_EXP_CURVE, capi.JAC_ANALYTICAL, capi.F64)
    pd = capi.make_problem(capi.MODEL_POINT_DIST, capi.JAC_FORWARD, capi.F64)
    x = np.ascontiguousarray(X_P2P)
    L = capi.lib()

    def call(stores, problems, xv, n=None):
        n = len(stores) if n is None else n
        hs = (C.c_void_p * max(len(stores), 1))(*[s.handle for s in stores])
        ps = (capi.Problem * max(len(problems), 1))(*problems)
        out = capi.CovTermsStruct()
        out.num_parameters, out.wsse = -7, 5.0
        rc = L.mopt_covariance_terms(ctx.handle, n, hs, ps, capi._dp(xv) if xv is not None else None, C.byref(out))
        return rc, out

    rc, out = call([st], [pp], x)
    assert rc == capi.OK and out.num_parameters == 6
    for stores, problems, xv, n in [([st], [pp], x, 0), ([st] * 9, [pp] * 9, x, 9), ([st], [pp], x, -1),
                                    ([so], [pp], x, None), ([st], [pp], None, None), ([sd], [pd], x, None),
                                    ([st, sc], [pp, pc], x, None)]:
        rc, out = call(stores, problems, xv, n)
        assert rc == 1 and out.num_parameters == -7 and out.wsse == 5.0, (n, rc)
    for s in (st, sc, sd, so):
        s.close()
    other.close()


# ---- 10. one 100 M point2point case ---------------------------------------------------------------------------------
def test_point2point_100m_fp32(env):
    capi, ctx = env
    n = 100_000_000
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    st.generate(seed=1, gt=X_P2P, noise_sigma=0.01, outlier_fraction=0.05, outlier_range=1.0)
    t = {}
    for cdt in (capi.F32, capi.F64):
        prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, cdt, loss=capi.LOSS_HUBER,
                                 loss_param=0.05)
        t[cdt] = ctx.covariance_terms([st], [prob], X_P2P)
    assert t[capi.F32].n_valid == t[capi.F64].n_valid == n
    assert fro_err(t[capi.F32].G, t[capi.F64].G) <= 1e-5, fro_err(t[capi.F32].G, t[capi.F64].G)
    res = capi.covariance_from_terms(t[capi.F32], capi.COV_SANDWICH)
    assert res.rank == 6 and np.all(res.std > 0)
    st.close()
