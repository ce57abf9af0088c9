"""An fp64 store with fp32 compute has no kernel: every entry point rejects the pair (MOPT_ERR_UNSUPPORTED, "store dtype
f64 with compute dtype f32 is not supported") in its argument validation, before anything is launched and with nothing
written -- empty ranges of mopt_evaluate, mopt_residual_quantiles and mopt_score_hypotheses included -- for builtin
and run-time compiled models alike."""
import ctypes as C

import numpy as np
import pytest

from tests.test_gpu_evaluate import make_store
from tests.test_user_model import P2P_SRC

pytestmark = pytest.mark.gpu

UNSUPPORTED = 4  # MOPT_ERR_UNSUPPORTED
MESSAGE = "store dtype f64 with compute dtype f32 is not supported"


@pytest.fixture(scope="module")
def env():
    from moptimizer_0_b200 import capi
    c = capi.Context(0)
    yield capi, c
    c.close()


def test_builtin_model_writes_nothing(env):
    import torch
    capi, ctx = env
    n = 1000
    st, _, _ = make_store(capi, ctx, capi.MODEL_POINT2POINT, n, capi.F64)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32)
    xs = np.zeros(6)
    L = capi.lib()

    def rejected(rc):
        return rc == UNSUPPORTED and MESSAGE in L.mopt_last_error().decode()

    # mopt_evaluate: with outputs, and an empty stats-only range
    r = torch.full((n, 3), 7.25, dtype=torch.float32, device="cuda:0")
    w = torch.full((n,), 7.25, dtype=torch.float32, device="cuda:0")
    stats = capi.EvalStats()
    stats.n_valid, stats.sum_sq = -5, -7.25
    for first, count, rp, wp in ((0, n, r.data_ptr(), w.data_ptr()), (5, 0, None, None)):
        assert rejected(L.mopt_evaluate(ctx.handle, st.handle, C.byref(prob), capi._dp(xs), first, count, float("inf"),
                                        capi.F32, rp, wp, C.byref(stats))), count
    torch.cuda.synchronize()
    assert bool((r == 7.25).all()) and bool((w == 7.25).all()) and stats.n_valid == -5 and stats.sum_sq == -7.25

    # mopt_residual_quantiles
    q = np.array([0.5])
    out = capi.QuantilesStruct()
    out.n_ranked, out.median = -5, -7.25
    sentinel = bytes(out)
    for count in (n, 0):
        assert rejected(L.mopt_residual_quantiles(ctx.handle, st.handle, C.byref(prob), capi._dp(xs), 0, count, 1,
                                                  capi._dp(q), C.byref(out))), count
        assert bytes(out) == sentinel, count

    # mopt_score_hypotheses
    hx = np.zeros((4, 6))
    hs = (capi.EvalStats * 4)()
    for k in range(4):
        hs[k].n_valid, hs[k].max_sq = -5, -7.25
    sentinel = bytes(hs)
    for count in (n, 0):
        assert rejected(L.mopt_score_hypotheses(ctx.handle, st.handle, C.byref(prob), 4, capi._dp(hx), 0, count, 0.1,
                                                hs)), count
        assert bytes(hs) == sentinel, count

    # mopt_covariance_terms
    hsd = (C.c_void_p * 1)(st.handle)
    ps = (capi.Problem * 1)(prob)
    ct = capi.CovTermsStruct()
    ct.num_parameters, ct.wsse = -7, 5.0
    assert rejected(L.mopt_covariance_terms(ctx.handle, 1, hsd, ps, capi._dp(xs), C.byref(ct)))
    assert ct.num_parameters == -7 and ct.wsse == 5.0

    # the passes and the LM, analytical (moment kernel) and finite differences
    for jac in (capi.JAC_ANALYTICAL, capi.JAC_FORWARD):
        p = capi.make_problem(capi.MODEL_POINT2POINT, jac, capi.F32)
        for call in (lambda: ctx.linearize(st, p, xs), lambda: ctx.compute_cost(st, p, xs),
                     lambda: ctx.lm_minimize([st], [p], xs, max_iterations=3)):
            with pytest.raises(capi.MoptError) as e:
                call()
            assert e.value.code == UNSUPPORTED and MESSAGE in str(e.value), jac
    st.close()


def test_user_model(env):
    capi, ctx = env
    um = capi.UserModel(P2P_SRC, 6, 3, 3, 3, set_size=12, rot_offset=3)
    try:
        st = capi.Store(ctx, um.model, 16, capi.F64)
        st.upload(0, np.zeros((16, 3)))
        st.upload(1, np.zeros((16, 3)))
        p32 = capi.make_problem(um.model, capi.JAC_FORWARD, capi.F32)
        x = np.zeros(6)
        calls = [lambda: ctx.linearize(st, p32, x), lambda: ctx.covariance_terms([st], [p32], x),
                 lambda: ctx.evaluate(st, p32, x),
                 lambda: ctx.evaluate(st, p32, x, count=0, residuals=False, weights=False),
                 lambda: ctx.quantiles(st, p32, x, (0.5,)), lambda: ctx.quantiles(st, p32, x, count=0),
                 lambda: ctx.score_hypotheses(st, p32, x[None], 0.1),
                 lambda: ctx.score_hypotheses(st, p32, x[None], 0.1, count=0)]
        for k, call in enumerate(calls):
            with pytest.raises(capi.MoptError) as e:
                call()
            assert e.value.code == UNSUPPORTED and MESSAGE in str(e.value), k
        st.close()
    finally:
        um.release()
