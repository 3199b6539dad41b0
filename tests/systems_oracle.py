"""ctypes front-end of the systems AMG restatement (tests/systems_oracle.c), TEST INFRASTRUCTURE ONLY.

The C source is compiled on first use against the parity oracle (oracle/oracle.h,
oracle/_build/liboracle.so) into a per-user temporary directory, so the repository tree is never
written.  `Hierarchy` is an oracle.Hierarchy whose levels come from the systems setup: every
accessor of the oracle (A, P, S, cf, l1, precond, vcycle) and its Krylov methods work on it
unchanged, and `dof(l)` returns the function labels of level l.
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


def _build() -> str:
    ora = O.build()
    src = os.path.join(_HERE, "systems_oracle.c")
    h = hashlib.sha256()
    for f in (src, os.path.join(_ORACLE, "oracle.h"), ora):
        with open(f, "rb") as fh:
            h.update(fh.read())
    d = os.path.join(tempfile.gettempdir(), f"hdk_systems_oracle_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    out = os.path.join(d, f"libsystems_oracle_{h.hexdigest()[:16]}.so")
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
        L.osys_setup.restype = C.c_void_p
        L.osys_setup.argtypes = [O.PO, C.POINTER(O.Params), C.c_int, O.PI]
        L.osys_hierarchy.restype = C.POINTER(O.OAMG)
        L.osys_hierarchy.argtypes = [C.c_void_p]
        L.osys_dof.restype = O.PI
        L.osys_dof.argtypes = [C.c_void_p, C.c_int]
        L.osys_destroy.argtypes = [C.c_void_p]
        L.osys_strength.restype = O.PO
        L.osys_strength.argtypes = [O.PO, C.c_double, C.c_double, C.c_int, O.PI]
        _LIB = L
    return _LIB


class Hierarchy(O.Hierarchy):
    """Systems AMG hierarchy (num_functions > 1, unknown approach); dof_func labels the rows
    (None: interleaved, row % num_functions)."""

    def __init__(self, A: sp.csr_matrix, params: O.Params | None = None, num_functions: int = 1,
                 dof_func: np.ndarray | None = None):
        self.params = params if params is not None else O.default_params(True)
        self._A = O.to_ocsr(A)
        dof = None if dof_func is None else np.ascontiguousarray(dof_func, dtype=np.int32)
        self._sys = lib().osys_setup(self._A, C.byref(self.params), int(num_functions),
                                     None if dof is None else O._pi(dof))
        self._h = lib().osys_hierarchy(self._sys)
        self.n = A.shape[0]

    def __del__(self):
        try:
            if self._sys:
                lib().osys_destroy(self._sys)      # frees the oracle hierarchy too
                self._sys = None
                self._h = None
            if self._A:
                O.lib().ocsr_free(self._A)
                self._A = None
        except Exception:
            pass

    def dof(self, l):
        """Function labels of the rows of level l."""
        p = lib().osys_dof(self._sys, l)
        return np.ctypeslib.as_array(p, shape=(self._h.contents.A[l].contents.nrows,)).copy()


def strength(A, num_functions, dof, theta=0.25, max_row_sum=0.9):
    """Strength pattern of the systems setup for the row labels `dof` (A with its diagonal first)."""
    pA = O.to_ocsr(A)
    d = np.ascontiguousarray(dof, dtype=np.int32)
    pS = lib().osys_strength(pA, theta, max_row_sum, int(num_functions), O._pi(d))
    S = O.from_ocsr(pS, pattern_only=True)
    O.lib().ocsr_free(pS)
    O.lib().ocsr_free(pA)
    return S
