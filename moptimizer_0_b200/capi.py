"""ctypes binding of include/mopt_capi.h (the C-ABI drop-in boundary).

Python here is test / benchmark plumbing only: the product is libmopt_b200.so (hand-written
sm_100a CUDA) and the C++ host mirror of the reference API in include/moptimizer/.
Loading fails loudly when the library is missing — there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libmopt_b200.so")

MAX_PARAMETERS, MAX_OUTPUTS, MAX_COSTS, MAX_TRACE, NCCL_ID_BYTES = 16, 4, 8, 1024, 128
MAX_QUANTILES = 8
MAX_HYPOTHESES = 1024
OK = 0
F32, F64 = 0, 1
(MODEL_POINT2POINT, MODEL_EXP_CURVE, MODEL_MICHAELIS_MENTEN, MODEL_PINHOLE, MODEL_POWELL,
 MODEL_POINT_DIST, MODEL_PINHOLE_DISTORT) = range(7)
JAC_ANALYTICAL, JAC_FORWARD, JAC_CENTRAL = range(3)
P2P_EXACT, P2P_REFTEST, P2P_REFTEST_COLMAJOR, P2P_LEFT = range(4)
MANIFOLD_ADDITIVE, MANIFOLD_SO3_LEFT = 0, 1
FLAG_GENERIC_KERNEL = 1
FLAG_STABLE_FD = 2
FLAG_REFERENCE_FLOAT_GUARD = 4
LM_STAGNATION_STOP = 1
LOSS_NONE, LOSS_GEMAN_MCCLURE, LOSS_HUBER = range(3)
COV_UNSCALED, COV_SCALED, COV_SANDWICH = range(3)
STATUS = ["CONVERGED", "MAXIMUM_ITERATIONS_REACHED", "SMALL_DELTA", "NUMERIC_ERROR", "FATAL_ERROR"]
MODEL_SHAPE = {  # model -> (P, O, ncomp_a, ncomp_b)
    MODEL_POINT2POINT: (6, 3, 3, 3), MODEL_EXP_CURVE: (2, 1, 1, 1), MODEL_MICHAELIS_MENTEN: (2, 1, 1, 1),
    MODEL_PINHOLE: (6, 2, 3, 2), MODEL_POWELL: (4, 4, 0, 0), MODEL_POINT_DIST: (0, 3, 3, 3),
    MODEL_PINHOLE_DISTORT: (15, 2, 3, 2),
}

EXPORTS = [
    "mopt_last_error", "mopt_version", "mopt_device_count", "mopt_ctx_create", "mopt_ctx_create_sharded",
    "mopt_comm_unique_id", "mopt_ctx_destroy", "mopt_ctx_synchronize", "mopt_ctx_stream", "mopt_ctx_set_launch",
    "mopt_store_create", "mopt_store_destroy", "mopt_store_size", "mopt_store_upload", "mopt_store_download",
    "mopt_store_generate", "mopt_linearize", "mopt_compute_cost", "mopt_linearize_async", "mopt_ctx_result",
    "mopt_upload_and_linearize", "mopt_lm_minimize", "mopt_lm_default_options", "mopt_so3_convert6dof",
    "mopt_ldlt_solve", "mopt_host_alloc", "mopt_host_free",
    "mopt_cloud_read_text", "mopt_cloud_write_binary", "mopt_cloud_read_binary", "mopt_cloud_free",
    "mopt_nn_index_create", "mopt_nn_index_destroy", "mopt_store_set_target", "mopt_store_reassociate",
    "mopt_ctx_peer_handle", "mopt_ctx_open_peers", "mopt_ctx_set_exchange_enabled",
    "mopt_user_model_compile", "mopt_user_model_release", "mopt_user_model_log",
    "mopt_measure_peaks", "mopt_measure_h2d", "mopt_evaluate", "mopt_covariance_terms", "mopt_covariance_from_terms",
    "mopt_residual_quantiles", "mopt_score_hypotheses", "mopt_align_terms", "mopt_align_terms_merge",
    "mopt_align_from_terms",
]
MODEL_USER_BASE = 1000
PEER_HANDLE_BYTES = 64


class Problem(C.Structure):
    _fields_ = [("model", C.c_int32), ("variant", C.c_int32), ("num_parameters", C.c_int32),
                ("num_outputs", C.c_int32), ("jacobian", C.c_int32), ("compute_dtype", C.c_int32),
                ("loss", C.c_int32), ("has_covariance", C.c_int32), ("loss_param", C.c_double),
                ("covariance", C.c_double * (MAX_OUTPUTS * MAX_OUTPUTS)), ("consts", C.c_double * 32),
                ("manifold", C.c_int32), ("flags", C.c_int32)]


class LmOptions(C.Structure):
    _fields_ = [("max_iterations", C.c_int32), ("lm_max_iterations", C.c_int32), ("lambda_factor", C.c_double),
                ("scalar_dtype", C.c_int32), ("speculative", C.c_int32), ("flags", C.c_int32),
                ("reserved", C.c_int32)]


class LmTrial(C.Structure):
    _fields_ = [("outer_iteration", C.c_int32), ("k", C.c_int32), ("accepted", C.c_int32), ("reserved", C.c_int32),
                ("y0", C.c_double), ("yi", C.c_double), ("rho", C.c_double), ("lambda_", C.c_double),
                ("nu", C.c_double)]


_TRIAL_DTYPE = np.dtype([("outer_iteration", "<i4"), ("k", "<i4"), ("accepted", "<i4"), ("reserved", "<i4"),
                         ("y0", "<f8"), ("yi", "<f8"), ("rho", "<f8"), ("lambda_", "<f8"), ("nu", "<f8")])


class LmReport(C.Structure):
    _fields_ = [("status", C.c_int32), ("executed_iterations", C.c_int32), ("num_trials", C.c_int32),
                ("num_passes", C.c_int32), ("final_cost", C.c_double), ("trials", LmTrial * MAX_TRACE)]


class Synth(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("first_index", C.c_int64), ("gt", C.c_double * MAX_PARAMETERS),
                ("lo", C.c_double * 3), ("hi", C.c_double * 3), ("n_total", C.c_int64),
                ("noise_sigma", C.c_double), ("outlier_fraction", C.c_double), ("outlier_range", C.c_double),
                ("consts", C.c_double * 32)]


class UserModelDesc(C.Structure):
    _fields_ = [("num_parameters", C.c_int32), ("num_outputs", C.c_int32), ("ncomp_a", C.c_int32),
                ("ncomp_b", C.c_int32), ("has_jacobian", C.c_int32), ("set_size", C.c_int32),
                ("rot_offset", C.c_int32), ("reserved", C.c_int32)]


class Peaks(C.Structure):
    _fields_ = [("fp32_fma_tflops", C.c_double), ("fp32_fma2_tflops", C.c_double),
                ("issue_gwarp_inst_per_s", C.c_double), ("hbm_read_gbs", C.c_double), ("reserved", C.c_double * 4)]


class EvalStats(C.Structure):
    _fields_ = [("n_valid", C.c_int64), ("n_inliers", C.c_int64), ("sum_sq", C.c_double),
                ("inlier_sum_sq", C.c_double), ("max_sq", C.c_double), ("reserved", C.c_double * 3)]


mopt_eval_stats = EvalStats  # the C name


class HypothesisScores:
    """Context.score_hypotheses: mopt_eval_stats of K hypotheses as numpy arrays of shape (K,) -- `n_valid`,
    `n_inliers`, `sum_sq`, `inlier_sum_sq`, `max_sq` -- and `msac`, the truncated-quadratic (MSAC) score."""

    def __init__(self, raw, inlier_threshold: float):
        st = np.ctypeslib.as_array(raw)
        self.n_valid = np.array(st["n_valid"], dtype=np.int64)
        self.n_inliers = np.array(st["n_inliers"], dtype=np.int64)
        self.sum_sq = np.array(st["sum_sq"], dtype=np.float64)
        self.inlier_sum_sq = np.array(st["inlier_sum_sq"], dtype=np.float64)
        self.max_sq = np.array(st["max_sq"], dtype=np.float64)
        self.inlier_threshold = float(inlier_threshold)

    @property
    def msac(self) -> np.ndarray:
        """inlier_sum_sq + (n_valid - n_inliers) thr^2: every outlier costs thr^2 (lower is better)."""
        return self.inlier_sum_sq + (self.n_valid - self.n_inliers) * self.inlier_threshold ** 2


class QuantilesStruct(C.Structure):
    _fields_ = [("n_ranked", C.c_int64), ("n_nan", C.c_int64), ("lo", C.c_double * MAX_QUANTILES),
                ("hi", C.c_double * MAX_QUANTILES), ("value", C.c_double * MAX_QUANTILES), ("median", C.c_double),
                ("robust_sigma", C.c_double), ("reserved", C.c_double * 4)]


mopt_quantiles = QuantilesStruct  # the C name


class Quantiles:
    """Context.quantiles: order statistics of e = r^T r.  `lo`, `hi`, `values` (numpy, one per requested q), the
    `median` of e, `robust_sigma` = sqrt(median / chi2_median(O)), the counts `n_ranked` / `n_nan`, and
    `norm_values` = sqrt(values), the quantiles of the residual norm |r|."""

    def __init__(self, raw: QuantilesStruct, n_q: int):
        self.raw = raw
        self.lo = np.array(raw.lo[:n_q], dtype=np.float64)
        self.hi = np.array(raw.hi[:n_q], dtype=np.float64)
        self.values = np.array(raw.value[:n_q], dtype=np.float64)
        self.median, self.robust_sigma = raw.median, raw.robust_sigma
        self.n_ranked, self.n_nan = raw.n_ranked, raw.n_nan

    @property
    def norm_values(self) -> np.ndarray:
        return np.sqrt(self.values)


class CovTermsStruct(C.Structure):
    _fields_ = [("num_parameters", C.c_int32), ("reserved0", C.c_int32), ("n_valid", C.c_int64), ("m", C.c_int64),
                ("H", C.c_double * (MAX_PARAMETERS * MAX_PARAMETERS)),
                ("G", C.c_double * (MAX_PARAMETERS * MAX_PARAMETERS)), ("b", C.c_double * MAX_PARAMETERS),
                ("wsse", C.c_double), ("sum_sq", C.c_double), ("reserved", C.c_double * 4)]


class CovReport(C.Structure):
    _fields_ = [("rank", C.c_int32), ("reserved0", C.c_int32), ("dof", C.c_int64), ("sigma2", C.c_double),
                ("eig_min", C.c_double), ("eig_max", C.c_double), ("reserved", C.c_double * 3)]


mopt_cov_terms, mopt_cov_report = CovTermsStruct, CovReport  # the C names


class CovTerms:
    """mopt_cov_terms with numpy views: `H`, `G` (P x P), `b` (P) and the scalars.  Terms add (`+`): sum the terms of
    cost groups, or of the ranks of a sharded problem, before covariance_from_terms."""

    def __init__(self, raw: Optional[CovTermsStruct] = None):
        self.raw = raw if raw is not None else CovTermsStruct()

    @property
    def P(self) -> int:
        return self.raw.num_parameters

    def _mat(self, name):
        P = self.P
        return np.ctypeslib.as_array(getattr(self.raw, name))[:P * P].reshape(P, P).T  # column-major

    H = property(lambda self: self._mat("H"))
    G = property(lambda self: self._mat("G"))
    b = property(lambda self: np.ctypeslib.as_array(self.raw.b)[:self.P])
    n_valid = property(lambda self: self.raw.n_valid)
    m = property(lambda self: self.raw.m)
    wsse = property(lambda self: self.raw.wsse)
    sum_sq = property(lambda self: self.raw.sum_sq)

    def __add__(self, other: "CovTerms") -> "CovTerms":
        if self.P != other.P:
            raise ValueError(f"terms of different parameter counts ({self.P} and {other.P})")
        out = CovTermsStruct()
        out.num_parameters = self.P
        out.n_valid, out.m = self.n_valid + other.n_valid, self.m + other.m
        for name in ("H", "G", "b"):
            np.ctypeslib.as_array(getattr(out, name))[:] = (np.ctypeslib.as_array(getattr(self.raw, name)) +
                                                            np.ctypeslib.as_array(getattr(other.raw, name)))
        out.wsse, out.sum_sq = self.wsse + other.wsse, self.sum_sq + other.sum_sq
        return CovTerms(out)

    @staticmethod
    def from_arrays(H, G, b, wsse: float, sum_sq: float, n_valid: int, m: int) -> "CovTerms":
        """Terms assembled on the host (e.g. after summing ranks with torch.distributed.all_reduce)."""
        H, G, b = (np.asarray(v, dtype=np.float64) for v in (H, G, b))
        P = b.shape[0]
        t = CovTermsStruct()
        t.num_parameters, t.n_valid, t.m, t.wsse, t.sum_sq = P, int(n_valid), int(m), float(wsse), float(sum_sq)
        np.ctypeslib.as_array(t.H)[:P * P] = H.T.reshape(-1)
        np.ctypeslib.as_array(t.G)[:P * P] = G.T.reshape(-1)
        np.ctypeslib.as_array(t.b)[:P] = b
        return CovTerms(t)


class Covariance:
    """Context.covariance / covariance_from_terms: `cov` (P x P), `std` (sqrt of its diagonal), and the report."""

    def __init__(self, cov: np.ndarray, rep: CovReport):
        self.cov = cov
        self.rank, self.dof, self.sigma2 = rep.rank, rep.dof, rep.sigma2
        self.eig_min, self.eig_max = rep.eig_min, rep.eig_max

    @property
    def std(self) -> np.ndarray:
        return np.sqrt(np.diag(self.cov))


def covariance_from_terms(terms: CovTerms, estimator: int = COV_SCALED, rcond: float = 0.0) -> Covariance:
    """mopt_covariance_from_terms (host only): the covariance of x from (summed) terms."""
    P = terms.P
    cov = np.zeros(P * P if P > 0 else 1, dtype=np.float64)
    rep = CovReport()
    check(lib().mopt_covariance_from_terms(C.byref(terms.raw), int(estimator), float(rcond), _dp(cov), C.byref(rep)))
    return Covariance(cov[:P * P].reshape(P, P).T.copy(), rep)


class AlignMomentsStruct(C.Structure):
    _fields_ = [("n_valid", C.c_int64), ("n_used", C.c_int64), ("w", C.c_double), ("mean_src", C.c_double * 3),
                ("mean_tgt", C.c_double * 3), ("cross", C.c_double * 9), ("var_src", C.c_double),
                ("var_tgt", C.c_double), ("reserved", C.c_double * 4)]


class AlignReport(C.Structure):
    _fields_ = [("cost", C.c_double), ("rms", C.c_double), ("eig", C.c_double * 4), ("degenerate", C.c_int32),
                ("reserved0", C.c_int32), ("reserved", C.c_double * 3)]


mopt_align_moments, mopt_align_report = AlignMomentsStruct, AlignReport  # the C names


class AlignTerms:
    """mopt_align_moments with numpy views: `mean_src`, `mean_tgt` (3), `cross` (3 x 3, source rows, target columns)
    and the scalars.  Terms of disjoint ranges or of the ranks of a sharded problem combine with `+`
    (mopt_align_terms_merge), in a fixed order for identical bits."""

    def __init__(self, raw: Optional[AlignMomentsStruct] = None):
        self.raw = raw if raw is not None else AlignMomentsStruct()

    n_valid = property(lambda self: self.raw.n_valid)
    n_used = property(lambda self: self.raw.n_used)
    w = property(lambda self: self.raw.w)
    mean_src = property(lambda self: np.ctypeslib.as_array(self.raw.mean_src))
    mean_tgt = property(lambda self: np.ctypeslib.as_array(self.raw.mean_tgt))
    cross = property(lambda self: np.ctypeslib.as_array(self.raw.cross).reshape(3, 3))
    var_src = property(lambda self: self.raw.var_src)
    var_tgt = property(lambda self: self.raw.var_tgt)

    def __add__(self, other: "AlignTerms") -> "AlignTerms":
        out = AlignMomentsStruct()
        check(lib().mopt_align_terms_merge(C.byref(self.raw), C.byref(other.raw), C.byref(out)))
        return AlignTerms(out)


class Alignment:
    """align_from_terms / Context.align: `x` = [t, omega] (the point2point parameter vector), `cost` = sum w |R p + t - q|^2
    at x, `rms`, `eig` (Horn's N, descending) and `degenerate`."""

    def __init__(self, x: np.ndarray, rep: AlignReport):
        self.x = x
        self.cost, self.rms = rep.cost, rep.rms
        self.eig = np.array(rep.eig[:], dtype=np.float64)
        self.degenerate = bool(rep.degenerate)


def align_from_terms(terms: AlignTerms) -> Alignment:
    """mopt_align_from_terms (host only): Horn's closed-form rigid transform from (merged) terms."""
    x = np.zeros(6, dtype=np.float64)
    rep = AlignReport()
    check(lib().mopt_align_from_terms(C.byref(terms.raw), _dp(x), C.byref(rep)))
    return Alignment(x, rep)


class MoptError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"mopt error {code}: {msg}")
        self.code = code


_lib = None


def lib():
    """Load libmopt_b200.so.  Raises if it has not been built: there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing — run `python -m moptimizer_0_b200.build` "
                              "(the CUDA library is the only implementation of this path)")
        L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        L.mopt_last_error.restype = C.c_char_p
        L.mopt_version.restype = C.c_char_p
        vp, dp, i64 = C.c_void_p, C.POINTER(C.c_double), C.c_int64
        L.mopt_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
        L.mopt_ctx_create_sharded.argtypes = [C.c_int, C.c_int, C.c_int, vp, C.POINTER(vp)]
        L.mopt_comm_unique_id.argtypes = [vp]
        L.mopt_ctx_destroy.argtypes = [vp]
        L.mopt_ctx_synchronize.argtypes = [vp]
        L.mopt_ctx_stream.argtypes = [vp, C.POINTER(C.c_uint64)]
        L.mopt_ctx_set_launch.argtypes = [vp, C.c_int, C.c_int]
        L.mopt_store_create.argtypes = [vp, C.c_int, C.c_int, i64, C.POINTER(vp)]
        L.mopt_store_destroy.argtypes = [vp]
        L.mopt_store_size.argtypes = [vp, C.POINTER(i64)]
        L.mopt_store_upload.argtypes = [vp, C.c_int, vp, C.c_int, i64, i64, i64]
        L.mopt_store_download.argtypes = [vp, C.c_int, vp, C.c_int, i64, i64]
        L.mopt_store_generate.argtypes = [vp, C.POINTER(Synth)]
        L.mopt_linearize.argtypes = [vp, vp, C.POINTER(Problem), dp, dp, dp, dp]
        L.mopt_compute_cost.argtypes = [vp, vp, C.POINTER(Problem), dp, dp]
        L.mopt_linearize_async.argtypes = [vp, vp, C.POINTER(Problem), dp]
        L.mopt_ctx_result.argtypes = [vp, C.c_int, dp, dp, dp]
        L.mopt_measure_peaks.argtypes = [vp, C.POINTER(Peaks)]
        L.mopt_evaluate.argtypes = [vp, vp, C.POINTER(Problem), dp, i64, i64, C.c_double, C.c_int, vp, vp,
                                    C.POINTER(EvalStats)]
        L.mopt_score_hypotheses.argtypes = [vp, vp, C.POINTER(Problem), C.c_int, dp, i64, i64, C.c_double,
                                            C.POINTER(EvalStats)]
        L.mopt_residual_quantiles.argtypes = [vp, vp, C.POINTER(Problem), dp, i64, i64, C.c_int, dp,
                                              C.POINTER(QuantilesStruct)]
        L.mopt_covariance_terms.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(Problem), dp,
                                            C.POINTER(CovTermsStruct)]
        L.mopt_covariance_from_terms.argtypes = [C.POINTER(CovTermsStruct), C.c_int, C.c_double, dp,
                                                 C.POINTER(CovReport)]
        L.mopt_align_terms.argtypes = [vp, vp, C.POINTER(Problem), dp, i64, i64, C.c_double,
                                       C.POINTER(AlignMomentsStruct)]
        L.mopt_align_terms_merge.argtypes = [C.POINTER(AlignMomentsStruct), C.POINTER(AlignMomentsStruct),
                                             C.POINTER(AlignMomentsStruct)]
        L.mopt_align_from_terms.argtypes = [C.POINTER(AlignMomentsStruct), dp, C.POINTER(AlignReport)]
        L.mopt_measure_h2d.argtypes = [vp, C.c_uint64, C.c_double, dp]
        L.mopt_upload_and_linearize.argtypes = [vp, vp, C.POINTER(Problem), vp, vp, C.c_int, i64, dp, dp, dp, dp]
        L.mopt_lm_minimize.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(Problem), C.POINTER(LmOptions), dp,
                                       C.POINTER(LmReport)]
        L.mopt_lm_default_options.argtypes = [C.POINTER(LmOptions)]
        L.mopt_lm_default_options.restype = None
        L.mopt_so3_convert6dof.argtypes = [dp, dp]
        L.mopt_ldlt_solve.argtypes = [C.c_int, dp, dp, dp]
        L.mopt_host_alloc.argtypes = [C.POINTER(vp), C.c_uint64]
        L.mopt_host_free.argtypes = [vp]
        L.mopt_cloud_read_text.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp),
                                           C.POINTER(i64)]
        L.mopt_cloud_write_binary.argtypes = [C.c_char_p, vp, C.c_int, C.c_int, i64]
        L.mopt_cloud_read_binary.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                             C.POINTER(vp), C.POINTER(i64)]
        L.mopt_cloud_free.argtypes = [vp, C.c_int]
        L.mopt_nn_index_create.argtypes = [vp, vp, C.c_int, C.c_int, i64, C.c_double, C.POINTER(vp)]
        L.mopt_nn_index_destroy.argtypes = [vp]
        L.mopt_store_set_target.argtypes = [vp, vp]
        L.mopt_store_reassociate.argtypes = [vp, dp, C.POINTER(i64)]
        L.mopt_ctx_peer_handle.argtypes = [vp, vp]
        L.mopt_ctx_open_peers.argtypes = [vp, vp]
        L.mopt_ctx_set_exchange_enabled.argtypes = [vp, C.c_int]
        L.mopt_user_model_compile.argtypes = [C.c_char_p, C.POINTER(UserModelDesc), C.POINTER(C.c_int)]
        L.mopt_user_model_release.argtypes = [C.c_int]
        L.mopt_user_model_log.argtypes = [C.c_int]
        L.mopt_user_model_log.restype = C.c_char_p
        _lib = L
    return _lib


def check(code: int):
    if code != OK:
        raise MoptError(code, lib().mopt_last_error().decode())


def _dp(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def make_problem(model: int, jacobian: int = JAC_ANALYTICAL, compute_dtype: int = F64, loss: int = LOSS_NONE,
                 loss_param: float = 0.0, variant: int = P2P_EXACT, covariance: Optional[np.ndarray] = None,
                 consts: Optional[Sequence[float]] = None, manifold: int = 0, flags: int = 0) -> Problem:
    P, O, _, _ = MODEL_SHAPE[model]
    p = Problem()
    p.manifold = manifold
    p.flags = flags
    p.model, p.variant, p.num_parameters, p.num_outputs = model, variant, P, O
    p.jacobian, p.compute_dtype, p.loss, p.loss_param = jacobian, compute_dtype, loss, float(loss_param)
    p.has_covariance = 0
    if covariance is not None:
        cv = np.asarray(covariance, dtype=np.float64).reshape(O, O)
        flat = cv.T.reshape(-1)  # column-major
        for i, v in enumerate(flat):
            p.covariance[i] = v
        p.has_covariance = 1
    if consts is not None:
        for i, v in enumerate(np.asarray(consts, dtype=np.float64).reshape(-1)):
            p.consts[i] = v
    return p


class UserModel:
    """A run-time compiled device model (mopt_user_model_compile): CUDA C++ source defining mopt_f
    (+ mopt_f_df, mopt_setup).  `.model` is the id to pass to Store(...) and make_problem(...)."""

    def __init__(self, source: str, num_parameters: int, num_outputs: int, ncomp_a: int, ncomp_b: int,
                 has_jacobian: bool = False, set_size: int = 0, rot_offset: int = -1):
        d = UserModelDesc(num_parameters, num_outputs, ncomp_a, ncomp_b, 1 if has_jacobian else 0, set_size,
                          rot_offset, 0)
        mid = C.c_int(0)
        check(lib().mopt_user_model_compile(source.encode(), C.byref(d), C.byref(mid)))
        self.model = mid.value
        MODEL_SHAPE[self.model] = (num_parameters, num_outputs, ncomp_a, ncomp_b)

    @property
    def log(self) -> str:
        return lib().mopt_user_model_log(self.model).decode()

    def release(self):
        if self.model:
            MODEL_SHAPE.pop(self.model, None)
            check(lib().mopt_user_model_release(self.model))
            self.model = 0


class Context:
    """One GPU (mopt_ctx).  `sharded=(rank, world, unique_id_bytes)` joins a NCCL communicator."""

    def __init__(self, device: int = 0, sharded=None):
        self.device = device
        self._h = C.c_void_p()
        if sharded is None:
            check(lib().mopt_ctx_create(device, C.byref(self._h)))
        else:
            rank, world, uid = sharded  # uid None: no NCCL communicator, open_peers() must follow
            buf = C.create_string_buffer(bytes(uid), NCCL_ID_BYTES) if uid is not None else None
            check(lib().mopt_ctx_create_sharded(device, rank, world, C.cast(buf, C.c_void_p) if buf else None,
                                                C.byref(self._h)))

    @staticmethod
    def unique_id() -> bytes:
        buf = C.create_string_buffer(NCCL_ID_BYTES)
        check(lib().mopt_comm_unique_id(C.cast(buf, C.c_void_p)))
        return buf.raw

    @property
    def handle(self):
        return self._h

    def peer_handle(self) -> bytes:
        """CUDA IPC handle of this rank's exchange buffer (NVLink peer exchange, see mopt_ctx_open_peers)."""
        buf = C.create_string_buffer(PEER_HANDLE_BYTES)
        check(lib().mopt_ctx_peer_handle(self._h, C.cast(buf, C.c_void_p)))
        return buf.raw

    def open_peers(self, handles_in_rank_order: Sequence[bytes]):
        blob = b"".join(bytes(h) for h in handles_in_rank_order)
        buf = C.create_string_buffer(blob, len(blob))
        check(lib().mopt_ctx_open_peers(self._h, C.cast(buf, C.c_void_p)))

    def set_exchange_enabled(self, enabled: bool):
        check(lib().mopt_ctx_set_exchange_enabled(self._h, 1 if enabled else 0))

    def synchronize(self):
        check(lib().mopt_ctx_synchronize(self._h))

    def stream(self) -> int:
        s = C.c_uint64(0)
        check(lib().mopt_ctx_stream(self._h, C.byref(s)))
        return s.value

    def measure_peaks(self) -> dict:
        """Measured ceilings of this GPU (fp32 FMA / packed FMA TFLOP/s, warp-instruction issue rate, HBM read)."""
        p = Peaks()
        check(lib().mopt_measure_peaks(self._h, C.byref(p)))
        return {"fp32_fma_tflops": p.fp32_fma_tflops, "fp32_fma2_tflops": p.fp32_fma2_tflops,
                "issue_gwarp_inst_per_s": p.issue_gwarp_inst_per_s, "hbm_read_gbs": p.hbm_read_gbs}

    def measure_h2d(self, nbytes: int = 1 << 30, seconds: float = 1.0) -> float:
        """Pinned host -> device GB/s of this process over at least `seconds` (ranks overlap when called together)."""
        g = C.c_double(0)
        check(lib().mopt_measure_h2d(self._h, int(nbytes), float(seconds), C.byref(g)))
        return g.value

    def set_launch(self, ctas_per_sm: int = 0, threads: int = 0):
        check(lib().mopt_ctx_set_launch(self._h, ctas_per_sm, threads))

    def close(self):
        if self._h:
            lib().mopt_ctx_destroy(self._h)
            self._h = C.c_void_p()

    # ---- the hot path ---------------------------------------------------------------------
    def linearize(self, store: "Store", problem: Problem, x):
        P = problem.num_parameters
        xs = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
        H = np.zeros((P, P), dtype=np.float64)
        b = np.zeros(P, dtype=np.float64)
        s = C.c_double(0)
        check(lib().mopt_linearize(self._h, store.handle, C.byref(problem), _dp(xs), _dp(H), _dp(b), C.byref(s)))
        return H, b, s.value

    def compute_cost(self, store: "Store", problem: Problem, x) -> float:
        xs = np.ascontiguousarray(np.asarray(x if len(x) else [0.0], dtype=np.float64))
        s = C.c_double(0)
        check(lib().mopt_compute_cost(self._h, store.handle, C.byref(problem), _dp(xs), C.byref(s)))
        return s.value

    def evaluate(self, store: "Store", problem: Problem, x, first: int = 0, count: Optional[int] = None,
                 inlier_threshold: float = float("inf"), residuals: bool = True, weights: bool = True,
                 out_dtype: int = F32, out=None) -> "EvalResult":
        """Per-residual evaluation (mopt_evaluate) of the elements [first, first + count) at x: residuals (count, O)
        and loss weights (count,) as CUDA tensors on this context's device, plus fit statistics.  `out` =
        (residuals, weights) supplies the output tensors (either may be None); they must be contiguous, on the
        context's device, of `out_dtype` and of those shapes.  Never re-associates: call store_reassociate first
        for fresh correspondences.  Elements without a correspondence get NaN residuals and weight 0."""
        import torch
        count = store.n - first if count is None else int(count)
        O = problem.num_outputs
        tdt = torch.float32 if out_dtype == F32 else torch.float64
        dev = torch.device("cuda", self.device)
        r_t = w_t = None
        if out is not None:
            r_t, w_t = out
            for t, shape, name in ((r_t, (count, O), "residuals"), (w_t, (count,), "weights")):
                if t is None:
                    continue
                if t.device != dev or t.dtype != tdt or tuple(t.shape) != shape or not t.is_contiguous():
                    raise ValueError(f"out {name}: need a contiguous {tdt} tensor of shape {shape} on {dev}, got "
                                     f"{t.dtype} {tuple(t.shape)} on {t.device}")
        else:
            if residuals:
                r_t = torch.empty((count, O), dtype=tdt, device=dev)
            if weights:
                w_t = torch.empty((count,), dtype=tdt, device=dev)
        xs = np.ascontiguousarray(np.asarray(x if len(x) else [0.0], dtype=np.float64))
        st = EvalStats()
        check(lib().mopt_evaluate(self._h, store.handle, C.byref(problem), _dp(xs), int(first), count,
                                  float(inlier_threshold), out_dtype, r_t.data_ptr() if r_t is not None else None,
                                  w_t.data_ptr() if w_t is not None else None, C.byref(st)))
        return EvalResult(st, count, r_t, w_t)

    def score_hypotheses(self, store: "Store", problem: Problem, xs, inlier_threshold: float, first: int = 0,
                         count: Optional[int] = None) -> HypothesisScores:
        """mopt_score_hypotheses: mopt_evaluate's statistics of the elements [first, first + count) at each row of xs
        (shape (K, P)), the store read once per 32 rows.  More than MAX_HYPOTHESES rows take several calls, which
        changes no count.  This context's store only; never re-associates."""
        P = problem.num_parameters
        xs = np.asarray(xs, dtype=np.float64)
        if xs.ndim != 2 or xs.shape[0] < 1 or xs.shape[1] != P:
            raise ValueError(f"xs must have shape (K, {P}) with K >= 1, got {xs.shape}")
        xs = np.ascontiguousarray(xs)
        count = store.n - first if count is None else int(count)
        out = (EvalStats * xs.shape[0])()
        for k0 in range(0, xs.shape[0], MAX_HYPOTHESES):
            k = min(MAX_HYPOTHESES, xs.shape[0] - k0)
            check(lib().mopt_score_hypotheses(self._h, store.handle, C.byref(problem), k, _dp(xs[k0:]), int(first),
                                              count, float(inlier_threshold),
                                              C.cast(C.addressof(out) + k0 * C.sizeof(EvalStats), C.POINTER(EvalStats))))
        return HypothesisScores(out, inlier_threshold)

    def quantiles(self, store: "Store", problem: Problem, x, q=(), first: int = 0,
                  count: Optional[int] = None) -> Quantiles:
        """mopt_residual_quantiles: exact quantiles (numpy's method="linear") of e = r^T r over the elements
        [first, first + count) at x, for the levels q (at most MAX_QUANTILES), plus the median and the robust scale.
        This context's store only; never re-associates."""
        count = store.n - first if count is None else int(count)
        qs = np.ascontiguousarray(np.asarray(q, dtype=np.float64).reshape(-1))
        if qs.size > MAX_QUANTILES:
            raise ValueError(f"at most {MAX_QUANTILES} quantile levels, got {qs.size}")
        xs = np.ascontiguousarray(np.asarray(x if len(x) else [0.0], dtype=np.float64))
        out = QuantilesStruct()
        check(lib().mopt_residual_quantiles(self._h, store.handle, C.byref(problem), _dp(xs), int(first), count,
                                            int(qs.size), _dp(qs) if qs.size else None, C.byref(out)))
        return Quantiles(out, int(qs.size))

    def covariance_terms(self, stores: Sequence["Store"], problems: Sequence[Problem], x) -> CovTerms:
        """mopt_covariance_terms: additive covariance terms (H, G, b, wsse, sum_sq, n_valid, m) of the cost terms at x,
        this context's stores only.  Never re-associates."""
        n = len(stores)
        hs = (C.c_void_p * n)(*[s.handle for s in stores])
        ps = (Problem * n)(*problems)
        xs = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
        out = CovTermsStruct()
        check(lib().mopt_covariance_terms(self._h, n, hs, ps, _dp(xs), C.byref(out)))
        return CovTerms(out)

    def covariance(self, stores: Sequence["Store"], problems: Sequence[Problem], x, estimator: int = COV_SCALED,
                   rcond: float = 0.0) -> Covariance:
        """Covariance of x (`.cov`, `.std`, `.rank`, `.dof`, `.sigma2`) from this context's stores: the terms on the
        device, then mopt_covariance_from_terms."""
        return covariance_from_terms(self.covariance_terms(stores, problems, x), estimator, rcond)

    def align_terms(self, store: "Store", problem: Problem, x, inlier_threshold: float = np.inf, first: int = 0,
                    count: Optional[int] = None) -> AlignTerms:
        """mopt_align_terms: weighted moments of the source and target points of the elements [first, first + count)
        of a point2point store that mopt_evaluate counts as inliers at x, each weighted by its loss weight at x.  This
        context's store only; never re-associates."""
        count = store.n - first if count is None else int(count)
        xs = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
        out = AlignMomentsStruct()
        check(lib().mopt_align_terms(self._h, store.handle, C.byref(problem), _dp(xs), int(first), count,
                                     float(inlier_threshold), C.byref(out)))
        return AlignTerms(out)

    def align(self, store: "Store", problem: Problem, x, inlier_threshold: float = np.inf, first: int = 0,
              count: Optional[int] = None) -> Alignment:
        """The closed-form rigid transform (`.x`, `.cost`, `.rms`) of the pairs align_terms selects: the terms on the
        device, then mopt_align_from_terms."""
        return align_from_terms(self.align_terms(store, problem, x, inlier_threshold, first, count))

    def linearize_async(self, store: "Store", problem: Problem, xs: np.ndarray):
        check(lib().mopt_linearize_async(self._h, store.handle, C.byref(problem), _dp(xs)))

    def result(self, P: int):
        H = np.zeros((P, P), dtype=np.float64)
        b = np.zeros(P, dtype=np.float64)
        s = C.c_double(0)
        check(lib().mopt_ctx_result(self._h, P, _dp(H), _dp(b), C.byref(s)))
        return H, b, s.value

    def upload_and_linearize(self, store: "Store", problem: Problem, host_a: np.ndarray, host_b: np.ndarray, x):
        assert host_a.dtype == host_b.dtype and host_a.dtype in (np.float32, np.float64)
        P = problem.num_parameters
        xs = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
        H = np.zeros((P, P), dtype=np.float64)
        b = np.zeros(P, dtype=np.float64)
        s = C.c_double(0)
        dt = F32 if host_a.dtype == np.float32 else F64
        check(lib().mopt_upload_and_linearize(self._h, store.handle, C.byref(problem), host_a.ctypes.data,
                                              host_b.ctypes.data, dt, store.n, _dp(xs), _dp(H), _dp(b), C.byref(s)))
        return H, b, s.value

    def lm_minimize(self, stores: Sequence["Store"], problems: Sequence[Problem], x0, max_iterations: int = 15,
                    lm_iterations: int = 3, scalar_dtype: int = F64, speculative: bool = True,
                    stagnation_stop: bool = True) -> "LmResult":
        n = len(stores)
        hs = (C.c_void_p * n)(*[s.handle for s in stores])
        ps = (Problem * n)(*problems)
        opt = self.__dict__.get("_lm_options")
        if opt is None:  # every field the library's defaults set is either overwritten below or left as it is
            opt = self._lm_options = LmOptions()
            lib().mopt_lm_default_options(C.byref(opt))
        opt.max_iterations, opt.lm_max_iterations = max_iterations, lm_iterations
        opt.scalar_dtype, opt.speculative = scalar_dtype, 1 if speculative else 0
        opt.flags = LM_STAGNATION_STOP if stagnation_stop else 0
        x = np.array(x0, dtype=np.float64)
        # the report is 57 KB (1024-entry trace): one per context, copied out of by LmResult (a small solve is ~100 us)
        rep = self.__dict__.get("_lm_report")
        if rep is None:
            rep = self._lm_report = LmReport()
        check(lib().mopt_lm_minimize(self._h, n, hs, ps, C.byref(opt), _dp(x), C.byref(rep)))
        return LmResult(x, rep)


class EvalResult:
    """Context.evaluate: `residuals` (count, O) / `weights` (count,) CUDA tensors (None when not requested),
    `stats` (mopt_eval_stats as a dict) and the registration / calibration figures derived from it."""

    def __init__(self, st: EvalStats, count: int, residuals, weights):
        self.stats = {"n_valid": st.n_valid, "n_inliers": st.n_inliers, "sum_sq": st.sum_sq,
                      "inlier_sum_sq": st.inlier_sum_sq, "max_sq": st.max_sq}
        self.count = count
        self.residuals = residuals
        self.weights = weights

    @property
    def fitness(self) -> float:
        """Fraction of the evaluated elements that are inliers (n_inliers / count)."""
        return self.stats["n_inliers"] / self.count if self.count else 0.0

    @property
    def inlier_rmse(self) -> float:
        """sqrt(inlier_sum_sq / n_inliers): RMS residual norm over the inliers."""
        n = self.stats["n_inliers"]
        return float(np.sqrt(self.stats["inlier_sum_sq"] / n)) if n else 0.0

    @property
    def rms(self) -> float:
        """sqrt(sum_sq / n_valid): RMS residual norm over every valid element."""
        n = self.stats["n_valid"]
        return float(np.sqrt(self.stats["sum_sq"] / n)) if n else 0.0


class LmResult:
    def __init__(self, x: np.ndarray, rep: LmReport):
        self.x = x
        self.status = STATUS[rep.status]
        self.executed_iterations = rep.executed_iterations
        self.num_passes = rep.num_passes
        self.final_cost = rep.final_cost
        # the report object is reused by the context: copy the used part of the trace out as raw bytes now (1 us), parse
        # it when somebody asks (a small solve is ~90 us; building the arrays eagerly cost 8 us of it)
        self._raw = C.string_at(C.addressof(rep) + LmReport.trials.offset, rep.num_trials * _TRIAL_DTYPE.itemsize)
        self._trials_arr = None
        self._trace = None

    @property
    def _trials(self) -> np.ndarray:
        if self._trials_arr is None:
            self._trials_arr = np.frombuffer(self._raw, dtype=_TRIAL_DTYPE)
        return self._trials_arr

    @property
    def trace(self) -> np.ndarray:
        """[num_trials, 8]: outer_iteration, k, y0, yi, rho, lambda, nu, accepted."""
        if self._trace is None:
            t = self._trials
            self._trace = np.stack([t[f].astype(np.float64) for f in
                                    ("outer_iteration", "k", "y0", "yi", "rho", "lambda_", "nu", "accepted")],
                                   axis=1).reshape(len(t), 8)
        return self._trace

    @property
    def sequence(self) -> str:
        return "".join("A" if a else "R" for a in self._trials["accepted"])


class Store:
    """Device-buffer residual store (mopt_store): planar fp32/fp64 streams in HBM."""

    def __init__(self, ctx: Context, model: int, n: int, dtype: int = F32):
        self.ctx, self.model, self.n, self.dtype = ctx, model, int(n), dtype
        self._h = C.c_void_p()
        check(lib().mopt_store_create(ctx.handle, model, dtype, int(n), C.byref(self._h)))

    @property
    def handle(self):
        return self._h

    def upload(self, group: int, host: np.ndarray, first: int = 0, stride: int = 0):
        host = np.ascontiguousarray(host)
        if host.dtype not in (np.float32, np.float64):
            host = host.astype(np.float64)
        ncomp = MODEL_SHAPE[self.model][2 + group]
        count = host.size // (stride if stride else ncomp)
        dt = F32 if host.dtype == np.float32 else F64
        check(lib().mopt_store_upload(self._h, group, host.ctypes.data, dt, stride, first, count))

    def download(self, group: int, dtype=np.float64, first: int = 0, count: Optional[int] = None) -> np.ndarray:
        ncomp = MODEL_SHAPE[self.model][2 + group]
        count = self.n - first if count is None else count
        out = np.zeros((count, ncomp), dtype=dtype)
        dt = F32 if out.dtype == np.float32 else F64
        check(lib().mopt_store_download(self._h, group, out.ctypes.data, dt, first, count))
        return out

    def generate(self, seed: int, gt: Sequence[float], lo=(0, 0, 0), hi=(10, 10, 10), first_index: int = 0,
                 n_total: int = 0, noise_sigma: float = 0.0, outlier_fraction: float = 0.0,
                 outlier_range: float = 0.0, consts=None):
        d = Synth()
        d.seed, d.first_index, d.n_total = seed, first_index, n_total
        for i, v in enumerate(gt):
            d.gt[i] = float(v)
        for k in range(3):
            d.lo[k], d.hi[k] = float(lo[k]), float(hi[k])
        d.noise_sigma, d.outlier_fraction, d.outlier_range = noise_sigma, outlier_fraction, outlier_range
        if consts is not None:
            for i, v in enumerate(np.asarray(consts, dtype=np.float64).reshape(-1)):
                d.consts[i] = float(v)
        check(lib().mopt_store_generate(self._h, C.byref(d)))

    def close(self):
        if self._h:
            lib().mopt_store_destroy(self._h)
            self._h = C.c_void_p()


class NNIndex:
    """Fixed target cloud in a device uniform grid (mopt_nn_index): the data behind model->update(x)."""

    def __init__(self, ctx: Context, target_xyz: np.ndarray, max_distance: float, dtype: int = F64):
        t = np.ascontiguousarray(target_xyz)
        if t.dtype not in (np.float32, np.float64):
            t = t.astype(np.float64)
        self._h = C.c_void_p()
        self._keep = ctx
        check(lib().mopt_nn_index_create(ctx.handle, t.ctypes.data, F32 if t.dtype == np.float32 else F64, dtype,
                                         t.shape[0], float(max_distance), C.byref(self._h)))

    @property
    def handle(self):
        return self._h

    def close(self):
        if self._h:
            lib().mopt_nn_index_destroy(self._h)
            self._h = C.c_void_p()


def store_set_target(store: "Store", index: Optional[NNIndex]):
    check(lib().mopt_store_set_target(store.handle, index.handle if index is not None else None))


def store_reassociate(store: "Store", x) -> int:
    xs = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
    m = C.c_int64(0)
    check(lib().mopt_store_reassociate(store.handle, _dp(xs), C.byref(m)))
    return m.value


def cloud_read_text(path: str, columns: int = 6, keep: int = 3, dtype=np.float64, pinned: bool = False) -> np.ndarray:
    """tst/point2point.cpp:125-138 loader: text records -> (n, keep) array (copied out of the library buffer)."""
    ptr, n = C.c_void_p(), C.c_int64(0)
    dt = F32 if np.dtype(dtype) == np.float32 else F64
    check(lib().mopt_cloud_read_text(path.encode(), columns, keep, dt, 1 if pinned else 0, C.byref(ptr), C.byref(n)))
    try:
        ctype = C.c_float if dt == F32 else C.c_double
        arr = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ctype)), shape=(max(n.value, 0) * keep,)).copy()
    finally:
        lib().mopt_cloud_free(ptr, 1 if pinned else 0)
    return arr.reshape(n.value, keep)


def cloud_write_binary(path: str, data: np.ndarray):
    data = np.ascontiguousarray(data)
    assert data.dtype in (np.float32, np.float64) and data.ndim == 2
    dt = F32 if data.dtype == np.float32 else F64
    check(lib().mopt_cloud_write_binary(path.encode(), data.ctypes.data, dt, data.shape[1], data.shape[0]))


def cloud_read_binary(path: str) -> np.ndarray:
    ptr, n, dt, keep = C.c_void_p(), C.c_int64(0), C.c_int(0), C.c_int(0)
    check(lib().mopt_cloud_read_binary(path.encode(), 0, C.byref(dt), C.byref(keep), C.byref(ptr), C.byref(n)))
    try:
        ctype = C.c_float if dt.value == F32 else C.c_double
        arr = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ctype)), shape=(max(n.value, 0) * keep.value,)).copy()
    finally:
        lib().mopt_cloud_free(ptr, 0)
    return arr.reshape(n.value, keep.value)


def ldlt_solve_device(A: np.ndarray, rhs: np.ndarray) -> np.ndarray:
    n = A.shape[0]
    Af = np.ascontiguousarray(np.asarray(A, dtype=np.float64).T.reshape(-1))
    r = np.ascontiguousarray(np.asarray(rhs, dtype=np.float64))
    out = np.zeros(n, dtype=np.float64)
    check(lib().mopt_ldlt_solve(n, _dp(Af), _dp(r), _dp(out)))
    return out


def so3_convert6dof(x) -> np.ndarray:
    xs = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
    T = np.zeros(16, dtype=np.float64)
    check(lib().mopt_so3_convert6dof(_dp(xs), _dp(T)))
    return T.reshape(4, 4)
