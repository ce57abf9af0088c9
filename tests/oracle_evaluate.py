"""TEST INFRASTRUCTURE ONLY: ctypes view of the per-element reference loop (tests/oracle_evaluate.cpp), the oracle
that mopt_evaluate is checked against, plus the fit statistics of its arrays in numpy.

The library is compiled with g++ on first use (oracle/Makefile's flags) into a cache directory under the system's
temporary directory, keyed by the hash of its sources, so the repository tree is never written.  Cost descriptions
are oracle.oracle_py.Cost objects: the C struct is the oracle's own orc_cost.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from typing import Optional, Sequence

import numpy as np

from oracle import oracle_py as orc

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_SOURCES = [os.path.join(_HERE, "oracle_evaluate.cpp"), os.path.join(_ORACLE, "oracle_capi.cpp"),
            os.path.join(_ORACLE, "moptimizer_oracle.hpp")]
_FLAGS = ["-O3", "-march=x86-64-v3", "-ffp-contract=off", "-std=c++17", "-fPIC", "-Wall", "-Wextra", "-pthread"]

_lib = None


def build() -> str:
    h = hashlib.sha256(" ".join(_FLAGS).encode())
    for p in _SOURCES:
        with open(p, "rb") as f:
            h.update(f.read())
    d = os.path.join(tempfile.gettempdir(), f"mopt_oracle_eval_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    path = os.path.join(d, f"liboracle_evaluate_{h.hexdigest()[:16]}.so")
    if not os.path.exists(path):
        tmp = f"{path}.{os.getpid()}.tmp"
        subprocess.run([os.environ.get("CXX", "g++"), *_FLAGS, "-shared", "-I", _ORACLE, "-o", tmp, _SOURCES[0]],
                       check=True)
        os.replace(tmp, path)  # atomic: concurrent builders leave one complete library
    return path


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build(), mode=os.RTLD_LOCAL)
        dp = C.POINTER(C.c_double)
        L.orc_evaluate.argtypes = [C.POINTER(orc._OrcCost), C.c_int, dp, C.c_int, C.c_int, dp, dp, C.POINTER(C.c_int)]
        _lib = L
    return _lib


def evaluate(cost: orc.Cost, x: Sequence[float], scalar: int = orc.F64, first: int = 0, count: Optional[int] = None):
    """-> (r[count, O], w[count], valid[count] bool): the reference's computeCost loop with each element kept.
    Elements whose model f returned false have NaN residuals and weight 0."""
    count = cost.n - first if count is None else count
    xs = np.ascontiguousarray(np.asarray(x if len(x) else [0.0], dtype=np.float64))
    r = np.zeros((count, cost.O), dtype=np.float64)
    w = np.zeros(count, dtype=np.float64)
    valid = np.zeros(count, dtype=np.int32)
    cs = cost.c_struct()
    dp = C.POINTER(C.c_double)
    rc = lib().orc_evaluate(C.byref(cs), scalar, xs.ctypes.data_as(dp), int(first), int(count), r.ctypes.data_as(dp),
                            w.ctypes.data_as(dp), valid.ctypes.data_as(C.POINTER(C.c_int)))
    if rc:
        raise RuntimeError("oracle: unsupported cost description or range")
    return r, w, valid.astype(bool)


def eval_stats(r: np.ndarray, valid: np.ndarray, inlier_threshold: float = float("inf")) -> dict:
    """Fit statistics of per-element residuals, in numpy (fp64): what mopt_evaluate reports."""
    e2 = np.sum(np.asarray(r, dtype=np.float64)[valid] ** 2, axis=1)
    inl = e2 <= float(inlier_threshold) ** 2
    return {"n_valid": int(valid.sum()), "n_inliers": int(inl.sum()), "sum_sq": float(e2.sum()),
            "inlier_sum_sq": float(e2[inl].sum()), "max_sq": float(e2.max()) if e2.size else 0.0}
