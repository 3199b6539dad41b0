"""GPU parity on unstructured matrices (tests/amg_paths.py): graph Laplacians with hubs, finite
elements with Dirichlet rows, rotated anisotropy, positive couplings, a bordered matrix, scrambled
storage, one-level and two-level hierarchies, disconnected components.

Each case is compared with the oracle built from the device's own storage (diagonal first): the
hierarchy bit for bit, the V-cycle, the Krylov solve.  Independent of the oracle, A_c, the l1 norms,
S and every level's SpMV are checked against plain numpy restatements in long double.  Each case
asserts the code paths it reaches (tests/test_amg_paths.py checks the census itself); the forced
paths run in child processes because their switches are read once per process."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import amg_paths as AP
from oracle import oracle as O
from test_gpu_kernels import _compare_hierarchy

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = np.finfo(np.float64).eps
LD = np.longdouble


def device_storage(gpu, A):
    """The matrix as the device stores it (diagonal first), as scipy CSR."""
    rp, cj, va = gpu.DCsr.from_scipy(A).diag_arrays()
    return sp.csr_matrix((va.copy(), cj.copy(), rp.copy()), shape=A.shape)


def _csr(arrays, shape):
    rp, cj, va = arrays
    return sp.csr_matrix((va.copy(), cj.copy(), rp.copy()), shape=shape)


def check_independent(M, params):
    """A_c = R A P, l1 norms and S of every level against restatements that do not use the oracle."""
    th = params.get("strong_th", 0.25)
    mrs = params.get("max_row_sum", 0.9)
    for l in range(M.nlev):
        n = M.level_info(l)["rows"]
        A = _csr(M.matrix(l, "A"), (n, n))
        # l1 norms (relaxation 18): sum of |a_ij| in the row, sign of the diagonal
        l1 = M.l1(l)
        for i in range(n):
            row = A.data[A.indptr[i]:A.indptr[i + 1]]
            ref = math.fsum(np.abs(row)) * (-1.0 if row.size and row[0] < 0 else 1.0)
            assert abs(l1[i] - ref) <= row.size * EPS * abs(ref), (l, i)
        if l == M.nlev - 1:
            break
        nc = M.level_info(l + 1)["rows"]
        # strength: hypre_BoomerAMGCreateS restated row by row on the diagonal-first storage
        rp, cj, _ = M.matrix(l, "S")
        for i in range(n):
            b, e = A.indptr[i], A.indptr[i + 1]
            strong = []
            if e > b:
                d, off = A.data[b], A.data[b + 1:e]
                row_sum = np.cumsum(A.data[b:e])[-1]          # accumulated in stored order, as hypre does
                if not (abs(row_sum) > abs(d) * mrs and mrs < 1.0):
                    scale = off.max(initial=0.0) if d < 0 else off.min(initial=0.0)
                    keep = ~(off <= th * scale) if d < 0 else ~(off >= th * scale)
                    strong = A.indices[b + 1:e][keep]
            assert np.array_equal(cj[rp[i]:rp[i + 1]], strong), (l, i)
        # Galerkin product in long double, entrywise within (terms + 2) eps (|R||A||P|)_ij
        P = _csr(M.matrix(l, "P"), (n, nc))
        R = _csr(M.matrix(l, "R"), (nc, n))
        assert (R != P.T).nnz == 0
        Ac = _csr(M.matrix(l + 1, "A"), (nc, nc)).astype(LD)
        ref = (R.astype(LD) @ A.astype(LD) @ P.astype(LD)).tocsr()
        mag = (abs(R) @ abs(A) @ abs(P)).tocsr()
        terms = ((R != 0).astype(np.float64) @ (A != 0).astype(np.float64) @ (P != 0).astype(np.float64)).tocsr()
        err = abs(Ac - ref).tocsr()
        viol = (err - (mag.multiply(terms) + 2.0 * mag).astype(LD) * EPS).tocsr()
        assert viol.nnz == 0 or viol.data.max() <= 0, f"A_c level {l + 1}"


def spmv_check(gpu, indptr, cols, vals, n, label):
    """matvec and residual of a square matrix (rectangular ones padded with empty rows) against a
    long-double product, row by row within len_i eps sum_k |a_ik x_k| (+ |b_i| for the residual)."""
    dA = gpu.DCsr.from_csr(indptr, cols, vals)
    B = sp.csr_matrix((vals, cols, indptr), shape=(n, n))
    rng = np.random.default_rng(n)
    x, b = rng.standard_normal(n), rng.standard_normal(n)
    ref = B.astype(LD) @ x.astype(LD)
    mag = abs(B) @ np.abs(x)
    lens = np.diff(indptr)
    dx, dy, db, dr = gpu.DVec(n, x), gpu.DVec(n), gpu.DVec(n, b), gpu.DVec(n)
    dA.matvec(dx, dy)
    y = dy.get().astype(LD)
    assert np.all(np.abs(y - ref) <= lens * EPS * mag), f"{label}: matvec, kind {dA.spmv_kind()}"
    dA.residual(dx, db, dr)
    r = dr.get().astype(LD)
    assert np.all(np.abs(r - (b - ref)) <= (lens + 1) * EPS * (mag + np.abs(b))), f"{label}: residual, kind {dA.spmv_kind()}"
    return dA.spmv_kind()


def _padded(rp, cj, va, n):
    """rows of a rectangular block as the first rows of an n x n matrix (empty rows below)."""
    ip = np.concatenate([rp, np.full(n + 1 - rp.size, rp[-1])]).astype(np.int64)
    return ip, cj.astype(np.int64), va


@pytest.mark.parametrize("name", list(AP.CASES))
def test_hierarchy_vcycle_and_solve_match_oracle(gpu, name):
    mk, prm, solver, want = AP.CASES[name]
    A_in = mk()
    A = device_storage(gpu, A_in)
    # the device's copy holds the input's entries (explicit zeros included), only reordered
    assert A.nnz == A_in.nnz and abs(A - A_in).max() == 0
    H, dA, M = _compare_hierarchy(gpu, A, prm)
    got = AP.paths(H, prm, A)
    assert want <= got, sorted(want - got)
    if "spmv.vector" in want and AP.census(H)[0]["max_row"] > AP.S_MAXR:
        assert dA.spmv_kind()["kind"] == 1
    check_independent(M, prm)
    n = A.shape[0]
    rng = np.random.default_rng(5)
    r = rng.standard_normal(n)
    dr, dz = gpu.DVec(n, r), gpu.DVec(n)
    M.apply(dr, dz)
    z_ref = H.precond(r)
    assert np.allclose(dz.get(), z_ref, rtol=1e-11, atol=1e-13 * np.abs(z_ref).max())
    u0 = rng.standard_normal(n)
    du = gpu.DVec(n, u0)
    M.vcycle(dr, du)
    u_ref = H.vcycle(r, u0)
    assert np.allclose(du.get(), u_ref, rtol=1e-11, atol=1e-13 * np.abs(u_ref).max())
    b = AP.rhs(n)
    tol = 1e-8
    db, dx = gpu.DVec(n, b), gpu.DVec(n)
    if solver == "pcg":
        info = gpu.pcg(dA, db, dx, M, rel_tol=tol, max_iter=200)
        x_ref, iref = O.pcg(A, b, M=H, rel_tol=tol, max_iter=200)
    else:
        info = gpu.gmres(dA, db, dx, M, rel_tol=tol, max_iter=200)
        x_ref, iref = O.gmres(A, b, M=H, rel_tol=tol, max_iter=200)
    assert info["converged"] and iref["converged"]
    assert info["iters"] == iref["iters"], (info["iters"], iref["iters"])
    if iref["iters"] > 1:                                  # (one iteration: both residuals are rounding noise)
        assert abs(info["rel_res_norm"] - iref["rel_res_norm"]) <= 1e-4 * iref["rel_res_norm"]
    x = dx.get()
    assert np.linalg.norm(x - x_ref) <= 1e-8 * np.linalg.norm(x_ref)
    assert np.linalg.norm(b - A @ x) / np.linalg.norm(b) < tol * 1.0001


def test_coarse_direct_solve_above_one_cta(gpu):
    """A coarsest level of more than 1024 rows is solved directly, as by the oracle (hypre's
    Gaussian elimination): with one level the preconditioner is the exact inverse."""
    A = device_storage(gpu, AP.diag_dominant(2000, 4))
    H, dA, M = _compare_hierarchy(gpu, A)
    assert M.nlev == 1
    n = A.shape[0]
    r = AP.rhs(n, 3)
    dr, dz = gpu.DVec(n, r), gpu.DVec(n)
    M.apply(dr, dz)
    z = dz.get()
    assert np.linalg.norm(A @ z - r) <= 1e-12 * np.linalg.norm(r)
    db, dx = gpu.DVec(n, r), gpu.DVec(n)
    assert gpu.pcg(dA, db, dx, M, rel_tol=1e-10)["iters"] == O.pcg(A, r, M=H, rel_tol=1e-10)[1]["iters"] == 1


SPMV_TUNES = [{}, {"spmv_lpr": 1}, {"spmv_lpr": 2}, {"spmv_lpr": 4}, {"spmv_lpr": 8}, {"sell_min_rows": 0}]
SPMV_DEFAULTS = {"spmv_lpr": 0, "sell_min_rows": 200000, "spmv_tgt_max": 3072}


@pytest.mark.parametrize("tune", SPMV_TUNES, ids=lambda t: ",".join(f"{k}={v}" for k, v in t.items()) or "default")
@pytest.mark.parametrize("name", ["heavy_tailed", "fe_rotated_aniso", "arrow"])
def test_level_spmv_against_long_double(gpu, name, tune):
    """A_l, P_l and R_l of every level through matvec and residual under each kernel selection."""
    mk, prm, _, _ = AP.CASES[name]
    A = device_storage(gpu, mk())
    M = gpu.DAmg(gpu.DCsr.from_scipy(A), gpu.amg_params(**prm))
    for k, v in tune.items():
        gpu.tune(k, v)
    try:
        for l in range(M.nlev):
            n = M.level_info(l)["rows"]
            rp, cj, va = M.matrix(l, "A")
            spmv_check(gpu, rp.astype(np.int64), cj.astype(np.int64), va, n, f"{name} A_{l}")
            if l < M.nlev - 1:
                spmv_check(gpu, *_padded(*M.matrix(l, "P"), n), n, f"{name} P_{l}")
                spmv_check(gpu, *_padded(*M.matrix(l, "R"), n), n, f"{name} R_{l}")
    finally:
        for k in tune:
            gpu.tune(k, SPMV_DEFAULTS[k])


@pytest.mark.parametrize("tune", SPMV_TUNES + [{"spmv_tgt_max": 8192}],
                         ids=lambda t: ",".join(f"{k}={v}" for k, v in t.items()) or "default")
@pytest.mark.parametrize("longest", [1024, 1025])
def test_spmv_rows_at_the_stream_kernel_limit(gpu, longest, tune):
    """Rows of exactly 1024 (the stream kernel's largest shared-memory stage) and 1025 entries
    (k_spmv_vector) among short rows, scattered columns."""
    n = 4000
    rng = np.random.default_rng(longest)
    lens = rng.integers(1, 30, size=n)
    lens[[7, 1999, n - 1]] = [longest, 700, longest]
    ip = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    cj = np.concatenate([np.sort(rng.choice(n, size=k, replace=False)) for k in lens]).astype(np.int64)
    va = rng.standard_normal(ip[-1])
    for k, v in tune.items():
        gpu.tune(k, v)
    try:
        kind = spmv_check(gpu, ip, cj, va, n, f"rows of {longest}")
    finally:
        for k in tune:
            gpu.tune(k, SPMV_DEFAULTS[k])
    # 1024 stays on the stream kernel, also with sell_min_rows 0: sliced ELL declines a matrix whose
    # 32-row slices would pad to more than 3 nnz (sell_build)
    assert kind["max_row"] == longest and kind["kind"] == (0 if longest <= AP.S_MAXR else 1), kind


@pytest.mark.parametrize("config", list(AP.FORCED))
def test_forced_setup_paths_match_oracle(gpu, config):
    """Interpolation one thread per row everywhere / one warp per row everywhere, count + fill
    interpolation, count + fill Galerkin product: the overflow-heavy cases with max_nnz_row 4, 0 and
    trunc_factor 0.2, hierarchy bit for bit (tests/forced_paths_check.py in a child process)."""
    env = dict(os.environ, HDK_AMG_KEEP_DEBUG="1", **AP.FORCED[config][0])
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "forced_paths_check.py"), *AP.FORCED_CASES],
                       env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("FORCED ok")]
    assert len(lines) == len(AP.FORCED_CASES) * len(AP.FORCED_SETTINGS), r.stdout[-3000:]
    for p in AP.FORCED[config][1]:
        assert any(f"'{p}'" in l for l in lines), (p, r.stdout[-3000:])
