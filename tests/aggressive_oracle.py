"""ctypes front-end of the aggressive-coarsening restatement (tests/aggressive_oracle.c), TEST INFRASTRUCTURE ONLY.

The C source is compiled on first use against the parity oracle (oracle/oracle.h,
oracle/_build/liboracle.so) into a per-user temporary directory, so the repository tree is never
written.  `Hierarchy` is an oracle.Hierarchy whose levels come from the aggressive setup: every
accessor of the oracle (A, P, S, cf, l1, precond, vcycle) and its Krylov methods work on it
unchanged; `S2(l)` returns the second-stage strength of an aggressive level and `passes(l)` the
multipass pass numbers.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import scipy.sparse as sp

from oracle import oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_LIB = None


class AggParams(C.Structure):
    _fields_ = [("num_levels", C.c_int), ("num_paths", C.c_int), ("max_nnz_row", C.c_int),
                ("trunc_factor", C.c_double)]


def _build() -> str:
    ora = O.build()
    src = os.path.join(_HERE, "aggressive_oracle.c")
    h = hashlib.sha256()
    for f in (src, os.path.join(_ORACLE, "oracle.h"), ora):
        with open(f, "rb") as fh:
            h.update(fh.read())
    d = os.path.join(tempfile.gettempdir(), f"hdk_aggressive_oracle_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    out = os.path.join(d, f"libaggressive_oracle_{h.hexdigest()[:16]}.so")
    if not os.path.exists(out):
        tmp = f"{out}.{os.getpid()}.tmp"
        subprocess.run(["gcc", "-O2", "-std=c99", "-fPIC", "-fopenmp", "-ffp-contract=off", "-Wall", "-Wextra",
                        "-Wno-unused-parameter", "-shared", f"-I{_ORACLE}", "-o", tmp, src,
                        f"-L{os.path.dirname(ora)}", "-loracle", f"-Wl,-rpath,{os.path.dirname(ora)}", "-lm"],
                       check=True)
        os.replace(tmp, out)
    return out


def lib():
    global _LIB
    if _LIB is None:
        O.lib()                                   # liboracle first: the restatement links against it
        L = C.CDLL(_build())
        L.oagg_setup.restype = C.c_void_p
        L.oagg_setup.argtypes = [O.PO, C.POINTER(O.Params), C.POINTER(AggParams)]
        L.oagg_hierarchy.restype = C.POINTER(O.OAMG)
        L.oagg_hierarchy.argtypes = [C.c_void_p]
        L.oagg_s2_of.restype = O.PO
        L.oagg_s2_of.argtypes = [C.c_void_p, C.c_int]
        L.oagg_pass_of.restype = O.PI
        L.oagg_pass_of.argtypes = [C.c_void_p, C.c_int]
        L.oagg_destroy.argtypes = [C.c_void_p]
        L.oagg_s2.restype = O.PO
        L.oagg_s2.argtypes = [O.PO, O.PI, C.c_int]
        _LIB = L
    return _LIB


class Hierarchy(O.Hierarchy):
    """AMG hierarchy with aggressive coarsening (two-stage PMIS, multipass interpolation) on the
    first `num_levels` levels."""

    def __init__(self, A: sp.csr_matrix, params: O.Params | None = None, num_levels: int = 1,
                 num_paths: int = 1, max_nnz_row: int = 0, trunc_factor: float = 0.0):
        self.params = params if params is not None else O.default_params(True)
        self.agg = AggParams(int(num_levels), int(num_paths), int(max_nnz_row), float(trunc_factor))
        self._A = O.to_ocsr(A)
        self._agg = lib().oagg_setup(self._A, C.byref(self.params), C.byref(self.agg))
        self._h = lib().oagg_hierarchy(self._agg)
        self.n = A.shape[0]

    def __del__(self):
        try:
            if self._agg:
                lib().oagg_destroy(self._agg)      # frees the oracle hierarchy too
                self._agg = None
                self._h = None
            if self._A:
                O.lib().ocsr_free(self._A)
                self._A = None
        except Exception:
            pass

    def S2(self, l):
        """Second-stage strength of level l (first-stage C points, row order), or None."""
        p = lib().oagg_s2_of(self._agg, l)
        return O.from_ocsr(p, pattern_only=True) if p else None

    def passes(self, l):
        """Multipass pass numbers of level l (1 = C, 0 = unreached), or None."""
        p = lib().oagg_pass_of(self._agg, l)
        if not p:
            return None
        return np.ctypeslib.as_array(p, shape=(self._h.contents.A[l].contents.nrows,)).copy()


def s2(S: sp.csr_matrix, cf1: np.ndarray, num_paths: int) -> sp.csr_matrix:
    """Second-stage strength of the restatement for a strength pattern S and first-stage C/F cf1."""
    S = sp.csr_matrix(S)
    S.data = np.ones(S.nnz)
    pS = O.to_ocsr(S)
    c = np.ascontiguousarray(cf1, dtype=np.int32)
    p = lib().oagg_s2(pS, O._pi(c), int(num_paths))
    out = O.from_ocsr(p, pattern_only=True)
    O.lib().ocsr_free(p)
    O.lib().ocsr_free(pS)
    return out
