"""ctypes binding of the hdk_* C-ABI (include/hdk.h) exported by libHYPREDRV.so.

This is the thin device layer underneath the HYPREDRV_* API.  It fails loudly when the CUDA
library is missing or no GPU is visible -- there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HDK_LIB") or os.path.join(_HERE, "lib", "libHYPREDRV.so")   # HDK_LIB: an experimental variant build
_lib = None


class HdkError(RuntimeError):
    pass


class AmgParams(C.Structure):
    _fields_ = [("coarsen_type", C.c_int), ("strong_th", C.c_double), ("max_row_sum", C.c_double),
                ("max_coarse_size", C.c_int), ("min_coarse_size", C.c_int), ("max_levels", C.c_int),
                ("interp_type", C.c_int), ("max_nnz_row", C.c_int), ("trunc_factor", C.c_double),
                ("relax_down", C.c_int), ("relax_up", C.c_int), ("relax_coarse", C.c_int),
                ("sweeps_down", C.c_int), ("sweeps_up", C.c_int), ("sweeps_coarse", C.c_int),
                ("relax_weight", C.c_double), ("outer_weight", C.c_double), ("rand_seed", C.c_int),
                ("keep_transpose", C.c_int), ("print_level", C.c_int),
                ("num_functions", C.c_int), ("dof_func", C.POINTER(C.c_int32)),
                ("agg_num_levels", C.c_int), ("agg_num_paths", C.c_int), ("agg_interp_type", C.c_int),
                ("agg_max_nnz_row", C.c_int), ("agg_trunc_factor", C.c_double),
                ("cheby_order", C.c_int), ("cheby_fraction", C.c_double), ("cheby_eig_est", C.c_int),
                ("cheby_variant", C.c_int), ("cheby_scale", C.c_int)]


class Krylov(C.Structure):
    _fields_ = [("max_iter", C.c_int), ("rel_tol", C.c_double), ("abs_tol", C.c_double),
                ("krylov_dim", C.c_int), ("min_iter", C.c_int), ("skip_real_res_check", C.c_int),
                ("iters", C.c_int), ("converged", C.c_int), ("rel_res_norm", C.c_double),
                ("solve_ms", C.c_double)]


def lib():
    """Load libHYPREDRV.so (built in-tree by __graft_entry__.build() / csrc/Makefile)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HdkError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(nvcc, sm_100a). hypredrive_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        L.hdk_last_error.restype = C.c_char_p
        L.hdk_stream.restype = C.c_void_p
        L.hdk_launch_count_reset.restype = C.c_int64
        L.hdk_amg_operator_complexity.restype = C.c_double
        L.hdk_amg_operator_complexity.argtypes = [C.c_void_p]
        L.hdk_amg_vcycle_bytes.restype = C.c_double
        L.hdk_amg_vcycle_bytes.argtypes = [C.c_void_p]
        L.hdk_amg_num_levels.argtypes = [C.c_void_p]
        L.hdk_vec_fill.argtypes = [C.c_void_p, C.c_double, C.c_int64]
        L.hdk_vec_axpy.argtypes = [C.c_double, C.c_void_p, C.c_void_p, C.c_int64]
        L.hdk_vec_scale.argtypes = [C.c_double, C.c_void_p, C.c_int64]
        L.hdk_vec_alloc.argtypes = [C.c_int64, C.POINTER(C.c_void_p)]
        L.hdk_vec_free.argtypes = [C.c_void_p]
        L.hdk_vec_h2d.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.hdk_vec_d2h.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.hdk_vec_copy.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.hdk_vec_dot.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_double)]
        L.hdk_vec_norm.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.POINTER(C.c_double)]
        L.hdk_vec_random.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int]
        L.hdk_csr_from_host.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.POINTER(C.c_void_p)]
        L.hdk_csr_stencil.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int64,
                                      C.c_int64, C.POINTER(C.c_void_p), C.c_void_p]
        L.hdk_csr_destroy.argtypes = [C.c_void_p]
        L.hdk_csr_info.argtypes = [C.c_void_p] + [C.POINTER(C.c_int64)] * 4
        L.hdk_csr_get_diag.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.hdk_csr_matvec.argtypes = [C.c_void_p, C.c_double, C.c_void_p, C.c_double, C.c_void_p]
        L.hdk_csr_residual.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.hdk_csr_spmv_kind.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_double), C.POINTER(C.c_int)]
        L.hdk_amg_default_params.argtypes = [C.POINTER(AmgParams)]
        L.hdk_amg_setup.argtypes = [C.c_void_p, C.POINTER(AmgParams), C.POINTER(C.c_void_p)]
        L.hdk_amg_destroy.argtypes = [C.c_void_p]
        L.hdk_amg_apply.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.hdk_amg_vcycle.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.hdk_amg_level_info.argtypes = [C.c_void_p, C.c_int] + [C.POINTER(C.c_int64)] * 3
        L.hdk_amg_get_matrix.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.hdk_amg_get_cf.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.hdk_amg_get_measure.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.hdk_amg_get_dof_func.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.hdk_amg_get_l1.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.hdk_amg_get_cheby.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.hdk_pcg.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Krylov)]
        L.hdk_gmres.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Krylov)]
        L.hdk_fgmres.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Krylov)]
        L.hdk_bicgstab.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Krylov)]
        L.hdk_time_kernel.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double),
                                      C.POINTER(C.c_double)]
        L.hdk_comm_unique_id.argtypes = [C.c_void_p]
        L.hdk_comm_init.argtypes = [C.c_int, C.c_int, C.c_void_p]
        L.hdk_init.argtypes = [C.c_int]
        _lib = L
    return _lib


def check(rc: int):
    if rc != 0:
        raise HdkError(f"hdk error {rc}: {lib().hdk_last_error().decode(errors='replace')}")


def init(device: int = -1):
    check(lib().hdk_init(device))


def device_count() -> int:
    return lib().hdk_device_count()


class DVec:
    """fp64 vector resident in HBM."""

    def __init__(self, n: int, data: np.ndarray | None = None):
        self.n = int(n)
        self.p = C.c_void_p()
        check(lib().hdk_vec_alloc(self.n, C.byref(self.p)))
        if data is not None:
            self.set(data)

    def set(self, data):
        a = np.ascontiguousarray(data, dtype=np.float64)
        assert a.size == self.n
        check(lib().hdk_vec_h2d(self.p, a.ctypes.data, self.n))

    def get(self) -> np.ndarray:
        out = np.empty(self.n, dtype=np.float64)
        if self.n:
            check(lib().hdk_vec_d2h(out.ctypes.data, self.p, self.n))
        return out

    def fill(self, v: float):
        check(lib().hdk_vec_fill(self.p, float(v), self.n))

    def free(self):
        if self.p:
            lib().hdk_vec_free(self.p)
            self.p = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class DCsr:
    """Rank-local ParCSR matrix on the device."""

    def __init__(self, handle):
        self.h = handle

    @classmethod
    def from_csr(cls, indptr, cols, data, row_start=0, row_end=None, global_rows=None):
        ip = np.ascontiguousarray(indptr, dtype=np.int64)
        cj = np.ascontiguousarray(cols, dtype=np.int64)
        va = np.ascontiguousarray(data, dtype=np.float64)
        n = ip.size - 1
        if row_end is None:
            row_end = row_start + n - 1
        if global_rows is None:
            global_rows = row_end + 1
        h = C.c_void_p()
        check(lib().hdk_csr_from_host(row_start, row_end, global_rows, ip.ctypes.data, cj.ctypes.data,
                                      va.ctypes.data, C.byref(h)))
        return cls(h)

    @classmethod
    def from_scipy(cls, A):
        A = A.tocsr()
        return cls.from_csr(A.indptr, A.indices, A.data)

    @classmethod
    def stencil(cls, kind: int, nx: int, ny: int, nz: int, c=(1.0, 1.0, 1.0), row_start=0, row_end=None):
        n = nx * ny * nz
        if row_end is None:
            row_end = n - 1
        h = C.c_void_p()
        b = DVec(row_end - row_start + 1)
        cc = (C.c_double * 3)(*map(float, c))
        check(lib().hdk_csr_stencil(kind, nx, ny, nz, cc, row_start, row_end, C.byref(h), b.p))
        return cls(h), b

    def info(self):
        v = [C.c_int64() for _ in range(4)]
        check(lib().hdk_csr_info(self.h, *[C.byref(x) for x in v]))
        return dict(local_rows=v[0].value, global_rows=v[1].value, local_nnz=v[2].value, global_nnz=v[3].value)

    def diag_arrays(self):
        i = self.info()
        n, nnz = i["local_rows"], i["local_nnz"]
        rp = np.empty(n + 1, dtype=np.int32)
        cj = np.empty(max(nnz, 1), dtype=np.int32)
        va = np.empty(max(nnz, 1), dtype=np.float64)
        check(lib().hdk_csr_get_diag(self.h, rp.ctypes.data, cj.ctypes.data, va.ctypes.data))
        nn = int(rp[n])
        return rp, cj[:nn], va[:nn]

    def matvec(self, x: DVec, y: DVec, alpha=1.0, beta=0.0):
        check(lib().hdk_csr_matvec(self.h, float(alpha), x.p, float(beta), y.p))

    def residual(self, x: DVec, b: DVec, r: DVec):
        check(lib().hdk_csr_residual(self.h, x.p, b.p, r.p))

    def spmv_kind(self):
        k, a, m = C.c_int(), C.c_double(), C.c_int()
        check(lib().hdk_csr_spmv_kind(self.h, C.byref(k), C.byref(a), C.byref(m)))
        return dict(kind=k.value, avg_row=a.value, max_row=m.value)

    def free(self):
        if self.h:
            lib().hdk_csr_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def amg_params(**kw) -> AmgParams:
    p = AmgParams()
    lib().hdk_amg_default_params(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise KeyError(k)
        setattr(p, k, v)
    return p


class DAmg:
    """Device BoomerAMG hierarchy."""

    def __init__(self, A: DCsr, params: AmgParams | None = None, dof_func=None):
        """dof_func: this rank's row labels for systems AMG (params.num_functions > 1); None: interleaved."""
        self.params = params if params is not None else amg_params()
        self.h = C.c_void_p()
        self.A = A
        if dof_func is not None:
            dof = np.ascontiguousarray(dof_func, dtype=np.int32)
            self.params.dof_func = dof.ctypes.data_as(C.POINTER(C.c_int32))
        check(lib().hdk_amg_setup(A.h, C.byref(self.params), C.byref(self.h)))
        self.params.dof_func = None   # read during the setup only

    @property
    def nlev(self):
        return lib().hdk_amg_num_levels(self.h)

    def level_info(self, l):
        v = [C.c_int64() for _ in range(3)]
        check(lib().hdk_amg_level_info(self.h, l, *[C.byref(x) for x in v]))
        return dict(rows=v[0].value, nnz_A=v[1].value, nnz_P=v[2].value)

    def sizes(self):
        return [(self.level_info(l)["rows"], self.level_info(l)["nnz_A"]) for l in range(self.nlev)]

    def matrix(self, l, which):
        """which: 'A', 'P', 'R', 'S', 'S2' -> (rowptr, col, val) in storage order.  'S2' is the
        second-stage strength of an aggressive level over its first-stage C points (amg_keep_debug)."""
        code = {"A": 0, "P": 1, "R": 2, "S": 3, "S2": 4}[which]
        if which == "S2":
            cf = self.cf(l)
            nrows = int(np.count_nonzero((cf == 1) | (cf == -2)))   # the first-stage C points
            rp = np.empty(nrows + 1, dtype=np.int32)
            check(lib().hdk_amg_get_matrix(self.h, l, code, rp.ctypes.data, None, None))
            cj = np.empty(max(int(rp[nrows]), 1), dtype=np.int32)
            check(lib().hdk_amg_get_matrix(self.h, l, code, rp.ctypes.data, cj.ctypes.data, None))
            return rp, cj[:int(rp[nrows])], np.ones(int(rp[nrows]))
        info = self.level_info(l)
        if which == "A":
            nrows, nnz = info["rows"], info["nnz_A"]
        elif which == "P":
            nrows, nnz = info["rows"], info["nnz_P"]
        elif which == "R":
            nrows, nnz = self.level_info(l + 1)["rows"], info["nnz_P"]
        else:
            nrows, nnz = info["rows"], info["nnz_A"]
        rp = np.empty(nrows + 1, dtype=np.int32)
        cj = np.empty(max(nnz, 1), dtype=np.int32)
        va = np.zeros(max(nnz, 1), dtype=np.float64)
        check(lib().hdk_amg_get_matrix(self.h, l, code, rp.ctypes.data, cj.ctypes.data, va.ctypes.data))
        nn = int(rp[nrows])
        return rp, cj[:nn], va[:nn]

    def cf(self, l):
        out = np.empty(self.level_info(l)["rows"], dtype=np.int32)
        check(lib().hdk_amg_get_cf(self.h, l, out.ctypes.data))
        return out

    def dof_func(self, l):
        """Function labels of this rank's rows of level l (systems AMG)."""
        out = np.empty(self.level_info(l)["rows"], dtype=np.int32)
        check(lib().hdk_amg_get_dof_func(self.h, l, out.ctypes.data))
        return out

    def measure(self, l):
        out = np.empty(self.level_info(l)["rows"], dtype=np.float64)
        check(lib().hdk_amg_get_measure(self.h, l, out.ctypes.data))
        return out

    def l1(self, l):
        out = np.empty(self.level_info(l)["rows"], dtype=np.float64)
        check(lib().hdk_amg_get_l1(self.h, l, out.ctypes.data))
        return out

    def cheby(self, l):
        """Chebyshev data of level l (relax 16): dict(eig=(max_eig, min_eig), coefs=c_0.., ds=D^{-1/2})."""
        eig = np.empty(2, dtype=np.float64)
        coefs = np.empty(4, dtype=np.float64)
        ds = np.empty(self.level_info(l)["rows"], dtype=np.float64)
        check(lib().hdk_amg_get_cheby(self.h, l, eig.ctypes.data, coefs.ctypes.data, ds.ctypes.data))
        return dict(eig=(float(eig[0]), float(eig[1])), coefs=coefs[:self.params.cheby_order].copy(), ds=ds)

    def apply(self, r: DVec, z: DVec):
        check(lib().hdk_amg_apply(self.h, r.p, z.p))

    def vcycle(self, f: DVec, u: DVec):
        check(lib().hdk_amg_vcycle(self.h, f.p, u.p))

    def operator_complexity(self):
        return lib().hdk_amg_operator_complexity(self.h)

    def vcycle_bytes(self):
        return lib().hdk_amg_vcycle_bytes(self.h)

    def free(self):
        if self.h:
            lib().hdk_amg_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def pcg(A: DCsr, b: DVec, x: DVec, M: DAmg | None = None, max_iter=100, rel_tol=1e-6, abs_tol=0.0):
    k = Krylov(max_iter=max_iter, rel_tol=rel_tol, abs_tol=abs_tol)
    check(lib().hdk_pcg(A.h, M.h if M is not None else None, b.p, x.p, C.byref(k)))
    return dict(iters=k.iters, converged=bool(k.converged), rel_res_norm=k.rel_res_norm, solve_ms=k.solve_ms)


def gmres(A: DCsr, b: DVec, x: DVec, M: DAmg | None = None, max_iter=300, rel_tol=1e-6, abs_tol=0.0,
          krylov_dim=30, skip_real_res_check=0):
    k = Krylov(max_iter=max_iter, rel_tol=rel_tol, abs_tol=abs_tol, krylov_dim=krylov_dim,
               skip_real_res_check=skip_real_res_check)
    check(lib().hdk_gmres(A.h, M.h if M is not None else None, b.p, x.p, C.byref(k)))
    return dict(iters=k.iters, converged=bool(k.converged), rel_res_norm=k.rel_res_norm, solve_ms=k.solve_ms)


def fgmres(A: DCsr, b: DVec, x: DVec, M: DAmg | None = None, max_iter=300, rel_tol=1e-6, abs_tol=0.0, krylov_dim=30):
    k = Krylov(max_iter=max_iter, rel_tol=rel_tol, abs_tol=abs_tol, krylov_dim=krylov_dim)
    check(lib().hdk_fgmres(A.h, M.h if M is not None else None, b.p, x.p, C.byref(k)))
    return dict(iters=k.iters, converged=bool(k.converged), rel_res_norm=k.rel_res_norm, solve_ms=k.solve_ms)


def bicgstab(A: DCsr, b: DVec, x: DVec, M: DAmg | None = None, max_iter=100, rel_tol=1e-6, abs_tol=0.0):
    k = Krylov(max_iter=max_iter, rel_tol=rel_tol, abs_tol=abs_tol)
    check(lib().hdk_bicgstab(A.h, M.h if M is not None else None, b.p, x.p, C.byref(k)))
    return dict(iters=k.iters, converged=bool(k.converged), rel_res_norm=k.rel_res_norm, solve_ms=k.solve_ms)


def time_kernel(A: DCsr, M: DAmg | None, kernel: int, reps: int = 20):
    ms, by = C.c_double(), C.c_double()
    check(lib().hdk_time_kernel(A.h, M.h if M is not None else None, kernel, reps, C.byref(ms), C.byref(by)))
    return ms.value, by.value


def amg_rows(hM, level: int, which: int):
    """This rank's rows of A_l (which=0) / P_l (which=1) of a row-distributed hierarchy with GLOBAL
    columns in the serial storage order (needs tune("amg_keep_debug", 1) before the setup).
    Returns (row0, indptr, cols, vals)."""
    L = lib()
    L.hdk_amg_get_rows.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.POINTER(C.c_int64)] * 3 + [C.c_void_p] * 3
    r0, nr, nz = C.c_int64(), C.c_int64(), C.c_int64()
    check(L.hdk_amg_get_rows(hM, level, which, C.byref(r0), C.byref(nr), C.byref(nz), None, None, None))
    ip = np.empty(nr.value + 1, dtype=np.int64)
    cj = np.empty(max(nz.value, 1), dtype=np.int64)
    va = np.empty(max(nz.value, 1), dtype=np.float64)
    check(L.hdk_amg_get_rows(hM, level, which, None, None, None, ip.ctypes.data, cj.ctypes.data, va.ctypes.data))
    return int(r0.value), ip, cj[:nz.value], va[:nz.value]


def amg_local_levels(hM):
    """(number of row-distributed levels, total number of levels) of a hierarchy handle."""
    L = lib()
    L.hdk_amg_num_dist_levels.argtypes = [C.c_void_p]
    return int(L.hdk_amg_num_dist_levels(hM)), int(L.hdk_amg_num_levels(hM))


def tune(key: str, value: float):
    """Kernel-selection tunable (hdk_tune), e.g. tune("sell_min_rows", 0)."""
    L = lib()
    L.hdk_tune.argtypes = [C.c_char_p, C.c_double]
    check(L.hdk_tune(key.encode(), float(value)))


def launch_count_reset() -> int:
    return int(lib().hdk_launch_count_reset())


def sync():
    check(lib().hdk_sync())
