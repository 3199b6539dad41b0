"""GPU parity of systems AMG (num_functions > 1, hypre's unknown approach) with the oracle.

For the vector-PDE cases of tests/systems_cases.py the device hierarchy is compared with the
oracle's bit for bit (S, C/F, P, every A_l, every level's function labels), then the V-cycle and
the PCG / GMRES solves.  One elasticity case is large enough (206 763 rows, 81 non-zeros a row) for
the production paths; the thread, warp and count + fill interpolation paths are forced in child
processes, which also report the SYS kernels that ran.  The HYPREDRV API runs with the
`elasticity_3d` preset, and two ranks run it on an even and a ragged split."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import systems_cases as SC
from hypredrive_b200 import driver, hdk
from oracle import oracle as O
import systems_oracle as SO

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def device_storage(A):
    """The matrix as the device stores it (diagonal first), as scipy CSR."""
    rp, cj, va = hdk.DCsr.from_scipy(A).diag_arrays()
    return sp.csr_matrix((va.copy(), cj.copy(), rp.copy()), shape=A.shape)


def compare_systems_hierarchy(A, nf, dof, params_kw):
    H = SO.Hierarchy(A, O.default_params(True, **params_kw), num_functions=nf, dof_func=dof)
    dA = hdk.DCsr.from_scipy(A)
    M = hdk.DAmg(dA, hdk.amg_params(num_functions=nf, **params_kw), dof_func=dof)
    assert M.nlev == H.nlev and M.sizes() == H.sizes(), (M.sizes(), H.sizes())
    for l in range(H.nlev):
        assert np.array_equal(M.dof_func(l), H.dof(l)), f"labels level {l}"
        if l == H.nlev - 1:
            break
        S = H.S(l)
        rp, cj, _ = M.matrix(l, "S")
        assert np.array_equal(rp, S.indptr) and np.array_equal(cj, S.indices), f"S level {l}"
        assert np.array_equal(M.cf(l), H.cf(l)), f"C/F splitting level {l}"
        P = H.P(l)
        rp, cj, va = M.matrix(l, "P")
        assert np.array_equal(rp, P.indptr) and np.array_equal(cj, P.indices), f"P pattern level {l}"
        assert np.array_equal(va, P.data), f"P values level {l}"
        Ac = H.A(l + 1)
        rp, cj, va = M.matrix(l + 1, "A")
        assert np.array_equal(rp, Ac.indptr) and np.array_equal(cj, Ac.indices), f"A_c pattern level {l + 1}"
        assert np.array_equal(va, Ac.data), f"A_c values level {l + 1}"
    for l in range(H.nlev):
        assert np.array_equal(M.l1(l), H.l1(l)), f"l1 norms level {l}"
    return H, dA, M


def _solves(H, dA, M, A, b):
    n = A.shape[0]
    r = np.random.default_rng(3).standard_normal(n)
    dr, dz = hdk.DVec(n, r), hdk.DVec(n)
    M.apply(dr, dz)
    z = H.precond(r)
    assert np.allclose(dz.get(), z, rtol=1e-11, atol=1e-11 * np.abs(z).max()), "V-cycle"
    for ofn, dfn in ((O.pcg, hdk.pcg), (O.gmres, hdk.gmres)):
        xr, info = ofn(A, b, M=H, rel_tol=1e-8, max_iter=200)
        db, dx = hdk.DVec(n, b), hdk.DVec(n)
        dx.fill(0.0)
        res = dfn(dA, db, dx, M, max_iter=200, rel_tol=1e-8)
        x = dx.get()
        assert res["converged"] and res["iters"] == info["iters"], (ofn.__name__, res, info["iters"])
        assert np.linalg.norm(x - xr) <= 1e-8 * np.linalg.norm(xr), ofn.__name__
        assert np.linalg.norm(b - A @ x) <= 1e-8 * np.linalg.norm(b) * 1.0001, ofn.__name__
    return info["iters"]


@pytest.mark.parametrize("name", list(SC.cases()))
def test_hierarchy_and_solves_match_oracle(gpu, name):
    A_in, b, nf, dof, th = SC.cases()[name]
    A = device_storage(A_in)
    H, dA, M = compare_systems_hierarchy(A, nf, dof, dict(strong_th=th))
    assert H.nlev >= 2
    _solves(H, dA, M, A, b)


def test_large_elasticity_matches_oracle(gpu):
    """3 * 41^3 = 206 763 rows: sliced-ELL SpMV and the warp interpolation on the fine level."""
    A_in, b = SC.elasticity(41, 3)
    A = device_storage(A_in)
    H, dA, M = compare_systems_hierarchy(A, 3, None, dict(strong_th=0.8))
    assert A.shape[0] > 200000 and H.nlev >= 3
    _solves(H, dA, M, A, b)


# (environment, SYS kernels that must run)
FORCED = {
    "default": ({}, {"k_strength<false, true>", "k_strength<true, true>", "k_interp_warp<true, true, true>"}),
    "thread": ({"HDK_INTERP_THREAD_AVG": "1e9"}, {"k_interp_small<true>"}),
    "count_fill": ({"HDK_INTERP_SINGLE": "0"}, {"k_interp_warp<true, false, true>"}),
    "fill_only": ({"HDK_INTERP_SINGLE": "0", "HDK_INTERP_THREAD_AVG": "1e9"}, {"k_interp_fill<true>"}),
}


@pytest.mark.parametrize("mode", list(FORCED))
def test_forced_paths_run_the_systems_kernels(gpu, mode):
    env_extra, want = FORCED[mode]
    env = dict(os.environ)
    env.update(env_extra)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "systems_paths_check.py"),
                        "elasticity_3d", "plane_strain", "block_labels", "ragged"],
                       env=env, capture_output=True, text=True, timeout=900)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("KERNELS ")]
    assert line, out[-3000:]
    ran = {k.replace("void ", "").replace("hdk::", "") for k in line[-1][8:].split("|")}
    assert want <= ran, (sorted(want - ran), sorted(ran))


def test_api_elasticity_preset(gpu):
    """HYPREDRV with `preset: elasticity_3d` builds the systems hierarchy: its iterations are the
    oracle's at num_functions = 3, strong_th = 0.8, and its level-0 strength pattern has none of the
    cross-function strong couplings that the scalar setup of the same matrix (default options) has."""
    A_in, b = SC.elasticity(12, 3)
    A = device_storage(A_in)
    tol = 1e-8

    def run(precon):
        opts = {"general": {"statistics": False}, "solver": {"pcg": {"relative_tol": tol, "max_iter": 200}},
                "preconditioner": precon}
        L = driver.api()
        with driver.HypreDrive(options=opts) as drv:
            drv.set_matrix_from_csr(A.indptr.astype(np.int64), A.indices.astype(np.int64), A.data)
            drv.set_rhs(b)
            driver._check(L.HYPREDRV_LinearSystemSetInitialGuess(drv._h, None), "SetInitialGuess")
            driver._check(L.HYPREDRV_LinearSystemResetInitialGuess(drv._h), "ResetInitialGuess")
            driver._check(L.HYPREDRV_LinearSolverCreate(drv._h), "LinearSolverCreate")
            driver._check(L.HYPREDRV_LinearSolverSetup(drv._h), "LinearSolverSetup")
            _, hM = drv.device_handles()
            n, nnz = A.shape[0], A.nnz
            rp, cj = np.empty(n + 1, np.int32), np.empty(nnz, np.int32)
            hdk.check(hdk.lib().hdk_amg_get_matrix(hM, 0, 3, rp.ctypes.data, cj.ctypes.data, None))
            driver._check(L.HYPREDRV_LinearSolverApply(drv._h), "LinearSolverApply")
            it = C.c_int()
            driver._check(L.HYPREDRV_LinearSolverGetNumIter(drv._h, C.byref(it)), "GetNumIter")
            x = drv.get_solution()
            L.HYPREDRV_LinearSolverDestroy(drv._h)
        return it.value, x, rp, cj[:rp[n]]

    lab = SC.interleaved(A.shape[0], 3)
    it_sys, x, rp, cj = run({"preset": "elasticity_3d"})
    H = SO.Hierarchy(A, O.default_params(True, strong_th=0.8), num_functions=3)
    xr, info = O.pcg(A, b, M=H, rel_tol=tol, max_iter=200)
    assert it_sys == info["iters"]
    assert np.linalg.norm(x - xr) <= 1e-8 * np.linalg.norm(xr)
    assert np.linalg.norm(b - A @ x) <= tol * np.linalg.norm(b) * 1.0001
    rows = np.repeat(np.arange(A.shape[0]), np.diff(rp))
    assert np.count_nonzero(lab[cj] != lab[rows]) == 0
    S_ref = H.S(0)
    assert np.array_equal(rp, S_ref.indptr) and np.array_equal(cj, S_ref.indices)
    # the scalar setup of the same matrix (default options) has cross-function strong couplings
    _, _, rps, cjs = run("amg")
    rows = np.repeat(np.arange(A.shape[0]), np.diff(rps))
    cross = np.count_nonzero(lab[cjs] != lab[rows])
    Ss = O.strength(A, 0.25, 0.9)
    rs = np.repeat(np.arange(A.shape[0]), np.diff(Ss.indptr))
    assert cross == np.count_nonzero(lab[Ss.indices] != lab[rs]) and cross > 0


def _digest(r):
    keep = [l for l in (r.stdout + "\n" + r.stderr).splitlines()
            if any(k in l for k in ("MPSYS", "hdk error", "HdkError", "HypreDriveError", "Error:", "error code", "NCCL WARN"))]
    return "\n".join(keep[-25:]) or (r.stdout[-1500:] + r.stderr[-1500:])


@pytest.mark.parametrize("split,full", [("even", "1"), ("ragged", "1"), ("even", "0"), ("ragged", "0")])
def test_two_ranks_match_oracle(gpu, split, full):
    """full = 1: every level replicated, the whole hierarchy is compared; full = 0: the default
    replicate_rows, the fine levels are row-distributed for the solve."""
    env = dict(os.environ)
    env["MPCHECK_HIER"] = full
    env["MPCHECK_RAGGED"] = "1" if split == "ragged" else "0"
    env["HDK_REPLICATE_ROWS"] = "100000000" if full == "1" else "2000"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29613", os.path.join(ROOT, "tests", "mp_systems_check.py"), "12"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, _digest(r)
    assert "ok=True" in r.stdout, _digest(r)
    if full == "1":
        assert "hier=bit-identical" in r.stdout, _digest(r)
    else:
        assert "dist_levels=0" not in r.stdout, _digest(r)
