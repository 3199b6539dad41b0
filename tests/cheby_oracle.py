"""ctypes front-end of the Chebyshev-smoothing restatement (tests/cheby_oracle.c), TEST INFRASTRUCTURE ONLY.

The C source is compiled on first use against the parity oracle (oracle/oracle.h, oracle/krylov.c,
oracle/_build/liboracle.so) into a per-user temporary directory, so the repository tree is never
written.  `Hierarchy` wraps any oracle hierarchy (the oracle's, or one of the systems / aggressive
restatements) and adds the per-level Chebyshev data of the levels that smooth with relax 16:
`cheby(l)`, `precond`, `vcycle`, `sweep`.  `pcg` / `gmres` are the oracle's Krylov methods (same
signature as oracle.pcg / oracle.gmres) running with this preconditioner.
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
PD = C.POINTER(C.c_double)


class ChebyParams(C.Structure):
    _fields_ = [("order", C.c_int), ("fraction", C.c_double), ("eig_est", C.c_int), ("scale", C.c_int)]


class _OCheby(C.Structure):
    _fields_ = [("h", C.c_void_p), ("cp", ChebyParams), ("has", C.c_int * 32), ("ds", PD * 32),
                ("eig", (C.c_double * 2) * 32), ("c", (C.c_double * 4) * 32)]


def _build() -> str:
    ora = O.build()
    src = os.path.join(_HERE, "cheby_oracle.c")
    h = hashlib.sha256()
    for f in (src, os.path.join(_ORACLE, "oracle.h"), os.path.join(_ORACLE, "krylov.c"), ora):
        with open(f, "rb") as fh:
            h.update(fh.read())
    d = os.path.join(tempfile.gettempdir(), f"hdk_cheby_oracle_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    out = os.path.join(d, f"libcheby_oracle_{h.hexdigest()[:16]}.so")
    if not os.path.exists(out):
        tmp = f"{out}.{os.getpid()}.tmp"
        subprocess.run(["gcc", "-O2", "-std=c99", "-fPIC", "-ffp-contract=off", "-Wall", "-Wextra",
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
        L.ocheby_attach.restype = C.POINTER(_OCheby)
        L.ocheby_attach.argtypes = [C.POINTER(O.OAMG), C.POINTER(ChebyParams), PD, C.POINTER(C.c_int)]
        L.ocheby_destroy.argtypes = [C.POINTER(_OCheby)]
        for f in ("ocheby_vcycle", "ocheby_precond"):
            getattr(L, f).argtypes = [C.POINTER(_OCheby), PD, PD]
        L.ocheby_sweep_level.argtypes = [C.POINTER(_OCheby), C.c_int, PD, PD]
        L.ocheby_gershgorin.argtypes = [O.PO, C.c_int, PD, PD]
        L.ocheby_cg_eig.argtypes = [O.PO, C.c_int, C.c_int, PD]
        L.ocheby_coefs.argtypes = [C.c_double, C.c_double, C.c_double, C.c_int, PD]
        for f in ("ocheby_pcg", "ocheby_gmres"):
            getattr(L, f).argtypes = [O.PO, C.c_void_p, PD, PD, C.POINTER(O.Krylov)]
        _LIB = L
    return _LIB


def _pd(x):
    return x.ctypes.data_as(PD)


class Hierarchy:
    """Chebyshev data on top of an oracle hierarchy `base` (its params choose which levels use relax 16).
    eigs: optional per-level (max_eig, min_eig) that replace the estimate (e.g. the device's), None
    entries keep it."""

    def __init__(self, base: O.Hierarchy, order: int = 2, fraction: float = 0.3, eig_est: int = 10,
                 scale: int = 1, eigs=None):
        self.base = base
        self.n = base.n
        self.cp = ChebyParams(int(order), float(fraction), int(eig_est), int(scale))
        ev = None
        if eigs is not None:
            ev = np.full(2 * 32, np.nan)
            for l, e in enumerate(eigs):
                if e is not None:
                    ev[2 * l], ev[2 * l + 1] = e
        st = C.c_int(0)
        self._ch = lib().ocheby_attach(base._h, C.byref(self.cp), _pd(ev) if ev is not None else None, C.byref(st))
        self.status = st.value
        if self.status != 0:
            raise ValueError(f"Chebyshev setup rejected on level {-self.status - 1}")

    def __del__(self):
        try:
            if self._ch:
                lib().ocheby_destroy(self._ch)
                self._ch = None
        except Exception:
            pass

    @property
    def nlev(self):
        return self.base.nlev

    @property
    def _h(self):          # what the Krylov methods hand to the preconditioner
        return C.cast(self._ch, C.c_void_p)

    def A(self, l):
        return self.base.A(l)

    def cheby(self, l):
        """dict(eig=(max, min), coefs, ds) of level l, or None when no type-16 sweep runs there."""
        c = self._ch.contents
        if not c.has[l]:
            return None
        n = self.base.A(l).shape[0]
        return dict(eig=(c.eig[l][0], c.eig[l][1]), coefs=np.array(c.c[l][:self.cp.order]),
                    ds=np.ctypeslib.as_array(c.ds[l], shape=(n,)).copy())

    def precond(self, r):
        r = np.ascontiguousarray(r, dtype=np.float64)
        z = np.zeros_like(r)
        lib().ocheby_precond(self._ch, _pd(r), _pd(z))
        return z

    def vcycle(self, f, u0):
        f = np.ascontiguousarray(f, dtype=np.float64)
        u = np.array(u0, dtype=np.float64, copy=True)
        lib().ocheby_vcycle(self._ch, _pd(f), _pd(u))
        return u

    def sweep(self, l, f, u0):
        """One Chebyshev sweep on level l from u0."""
        f = np.ascontiguousarray(f, dtype=np.float64)
        u = np.array(u0, dtype=np.float64, copy=True)
        lib().ocheby_sweep_level(self._ch, l, _pd(f), _pd(u))
        return u


def gershgorin(A: sp.csr_matrix, scale: int = 1):
    """(ds, (max_eig, min_eig)) of the Gershgorin rule; raises on a zero diagonal with scale = 1."""
    pA = O.to_ocsr(A)
    ds = np.zeros(A.shape[0])
    eig = np.zeros(2)
    rc = lib().ocheby_gershgorin(pA, int(scale), _pd(ds), _pd(eig))
    O.lib().ocsr_free(pA)
    if rc != 0:
        raise ValueError("zero diagonal")
    return ds, (eig[0], eig[1])


def cg_eig(A: sp.csr_matrix, steps: int, scale: int = 1):
    """(max_eig, min_eig) of the CG-Lanczos estimate and the number of completed steps."""
    pA = O.to_ocsr(A)
    eig = np.zeros(2)
    m = lib().ocheby_cg_eig(pA, int(scale), int(steps), _pd(eig))
    O.lib().ocsr_free(pA)
    return (eig[0], eig[1]), m


def coefs(max_eig: float, min_eig: float, fraction: float, order: int):
    c = np.zeros(4)
    if lib().ocheby_coefs(float(max_eig), float(min_eig), float(fraction), int(order), _pd(c)) != 0:
        raise ValueError("degenerate interval")
    return c[:order].copy()


def interval(max_eig: float, min_eig: float, fraction: float):
    """(lower, upper) of the rule, in the library's expression order."""
    if min_eig >= 0.0:
        upper = 1.1 * max_eig
        return (upper - min_eig) * fraction + min_eig, upper
    if max_eig <= 0.0:
        upper = 1.1 * min_eig
        return max_eig - (max_eig - upper) * fraction, upper
    upper = 1.1 * max_eig
    return (upper - 0.0) * fraction + 0.0, upper


class _Handle:
    def __init__(self, M):
        self._h = M._h if M is not None else None


def pcg(A, b, x0=None, M: Hierarchy | None = None, max_iter=100, rel_tol=1e-6, abs_tol=0.0):
    return O._krylov(lib().ocheby_pcg, A, b, x0, _Handle(M), max_iter, rel_tol, abs_tol, 0, 0)


def gmres(A, b, x0=None, M: Hierarchy | None = None, max_iter=300, rel_tol=1e-6, abs_tol=0.0,
          krylov_dim=30, skip_real_res_check=0):
    return O._krylov(lib().ocheby_gmres, A, b, x0, _Handle(M), max_iter, rel_tol, abs_tol, krylov_dim,
                     skip_real_res_check)
