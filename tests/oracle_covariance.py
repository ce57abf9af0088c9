"""TEST INFRASTRUCTURE ONLY: ctypes view of the reference's linearization loops with the score Gram accumulation
(tests/oracle_covariance.cpp), the oracle that mopt_covariance_terms' G, wsse and n_valid are checked against.

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
from typing import Sequence

import numpy as np

from oracle import oracle_py as orc

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_SOURCES = [os.path.join(_HERE, "oracle_covariance.cpp"), os.path.join(_ORACLE, "oracle_capi.cpp"),
            os.path.join(_ORACLE, "moptimizer_oracle.hpp")]
_FLAGS = ["-O3", "-march=x86-64-v3", "-ffp-contract=off", "-std=c++17", "-fPIC", "-Wall", "-Wextra", "-pthread"]

_lib = None


def build() -> str:
    h = hashlib.sha256(" ".join(_FLAGS).encode())
    for p in _SOURCES:
        with open(p, "rb") as f:
            h.update(f.read())
    d = os.path.join(tempfile.gettempdir(), f"mopt_oracle_cov_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    path = os.path.join(d, f"liboracle_covariance_{h.hexdigest()[:16]}.so")
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
        L.orc_score_gram.argtypes = [C.POINTER(orc._OrcCost), C.c_int, dp, dp, dp, C.POINTER(C.c_int64)]
        _lib = L
    return _lib


def score_gram(cost: orc.Cost, x: Sequence[float], scalar: int = orc.F64):
    """-> (G[P, P], wsse, n_valid): sum g g^T with g = w J^T C r, sum w r^T C r and the count of elements whose model
    f returned true, over the reference's computeHessian / computeHessianNumerical loop at x."""
    P = cost.P
    xs = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
    G = np.zeros(P * P, dtype=np.float64)
    q = C.c_double(0)
    n = C.c_int64(0)
    cs = cost.c_struct()
    dp = C.POINTER(C.c_double)
    if lib().orc_score_gram(C.byref(cs), scalar, xs.ctypes.data_as(dp), G.ctypes.data_as(dp), C.byref(q), C.byref(n)):
        raise RuntimeError("oracle: unsupported cost description")
    return G.reshape(P, P).T.copy(), q.value, n.value
