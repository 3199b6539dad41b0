"""GPU parity of aggressive coarsening (two-stage PMIS, multipass interpolation) with the CPU
restatement (tests/aggressive_oracle.c).

The device hierarchy is compared with the restatement's bit for bit (S, S2, C/F including -2, P, every
A_l, l1 norms), then the V-cycle and the PCG / GMRES solves, on stencil problems (one of 128^3 rows,
so the warp kernels and sliced-ELL run on the aggressive level) and on the unstructured cases of
tests/amg_paths.py.  The one-thread-per-row S2 and product paths are forced in child processes that
report the kernels that ran; the HYPREDRV API runs with `aggressive: num_levels: 1`, and two ranks run
the replicated setup on an even and a ragged split."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import aggressive_oracle as AO
import amg_paths as AP
from hypredrive_b200 import driver, hdk
from oracle import oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def device_storage(A):
    """The matrix as the device stores it (diagonal first), as scipy CSR."""
    rp, cj, va = hdk.DCsr.from_scipy(A).diag_arrays()
    return sp.csr_matrix((va.copy(), cj.copy(), rp.copy()), shape=A.shape)


def _agg_device(agg):
    return dict(agg_num_levels=agg.get("num_levels", 1), agg_num_paths=agg.get("num_paths", 1),
                agg_max_nnz_row=agg.get("max_nnz_row", 0), agg_trunc_factor=agg.get("trunc_factor", 0.0))


def compare_aggressive_hierarchy(A, agg, params_kw=None):
    params_kw = params_kw or {}
    H = AO.Hierarchy(A, O.default_params(True, **params_kw), **agg)
    dA = hdk.DCsr.from_scipy(A)
    M = hdk.DAmg(dA, hdk.amg_params(**_agg_device(agg), **params_kw))
    assert M.nlev == H.nlev and M.sizes() == H.sizes(), (M.sizes(), H.sizes())
    for l in range(H.nlev - 1):
        S = H.S(l)
        rp, cj, _ = M.matrix(l, "S")
        assert np.array_equal(rp, S.indptr) and np.array_equal(cj, S.indices), f"S level {l}"
        assert np.array_equal(M.cf(l), H.cf(l)), f"C/F splitting level {l}"
        S2 = H.S2(l)
        if S2 is not None:
            rp, cj, _ = M.matrix(l, "S2")
            assert np.array_equal(rp, S2.indptr) and np.array_equal(cj, S2.indices), f"S2 level {l}"
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


def _solves(H, dA, M, A, b, methods=("pcg", "gmres")):
    n = A.shape[0]
    r = np.random.default_rng(3).standard_normal(n)
    dr, dz = hdk.DVec(n, r), hdk.DVec(n)
    M.apply(dr, dz)
    z = H.precond(r)
    assert np.allclose(dz.get(), z, rtol=1e-11, atol=1e-11 * np.abs(z).max()), "V-cycle"
    iters = {}
    for name in methods:
        ofn, dfn = (O.pcg, hdk.pcg) if name == "pcg" else (O.gmres, hdk.gmres)
        xr, info = ofn(A, b, M=H, rel_tol=1e-8, max_iter=300)
        db, dx = hdk.DVec(n, b), hdk.DVec(n)
        dx.fill(0.0)
        res = dfn(dA, db, dx, M, max_iter=300, rel_tol=1e-8)
        x = dx.get()
        assert res["converged"] and res["iters"] == info["iters"], (name, res, info["iters"])
        assert np.linalg.norm(x - xr) <= 1e-8 * np.linalg.norm(xr), name
        assert np.linalg.norm(b - A @ x) <= 1e-8 * np.linalg.norm(b) * 1.0001, name
        iters[name] = res["iters"]
    return iters


STENCILS = {
    "lap7": (lambda: O.gen("lap7", 30, 28, 26), ("pcg", "gmres")),
    "lap27_aniso": (lambda: O.gen("lap27", 30, 26, 22, c=(1.0, 1.0, 0.01)), ("pcg", "gmres")),
    "convdif": (lambda: O.gen("convdif", 40, 20, 16, c=(1e-3, 1.0, 0.1)), ("gmres",)),
}
AGG = {
    "l1p1": dict(num_levels=1, num_paths=1),
    "l1p2": dict(num_levels=1, num_paths=2),
    "l2p1": dict(num_levels=2, num_paths=1),
    "l2p2_mx4": dict(num_levels=2, num_paths=2, max_nnz_row=4),
    "l1_tf": dict(num_levels=1, trunc_factor=0.2),
}


@pytest.mark.parametrize("agg", list(AGG))
@pytest.mark.parametrize("name", list(STENCILS))
def test_stencil_hierarchy_and_solves_match_restatement(gpu, name, agg):
    make, methods = STENCILS[name]
    A_in, b = make()
    A = device_storage(A_in)
    H, dA, M = compare_aggressive_hierarchy(A, AGG[agg])
    assert H.nlev >= 2 and (H.cf(0) == -2).any()
    _solves(H, dA, M, A, b, methods)


UNSTRUCTURED = ["heavy_tailed", "rgg3d", "fe_dirichlet", "fe_rotated_aniso", "signed_graph", "arrow", "scrambled_fe",
                "block_diagonal"]


@pytest.mark.parametrize("agg", ["l1p1", "l2p2_mx4", "l1_tf"])
@pytest.mark.parametrize("name", UNSTRUCTURED)
def test_unstructured_hierarchy_and_solves_match_restatement(gpu, name, agg):
    make, params, solver, _ = AP.CASES[name]
    A = device_storage(make())
    b = AP.rhs(A.shape[0])
    H, dA, M = compare_aggressive_hierarchy(A, AGG[agg], params)
    _solves(H, dA, M, A, b, (solver,))


def test_lumped_row_weights(gpu):
    """signed_graph: a pass-2 row whose strong couplings are all negative while the row has positive
    ones (cpos == 0, npos != 0) lumps npos into the diagonal; its device P row equals the rule."""
    A = device_storage(AP.signed_graph(8000, 9))
    H, dA, M = compare_aggressive_hierarchy(A, dict(num_levels=1))
    S, ps, cf = H.S(0), H.passes(0), H.cf(0)
    C = np.flatnonzero(cf == 1)
    f2c = np.full(A.shape[0], -1)
    f2c[C] = np.arange(len(C))
    rp, cj, va = M.matrix(0, "P")
    checked = 0
    for i in np.flatnonzero(ps == 2):
        b, e = A.indptr[i], A.indptr[i + 1]
        off, cols = A.data[b + 1:e], A.indices[b + 1:e]
        Si = S.indices[S.indptr[i]:S.indptr[i + 1]]
        J = Si[ps[Si] == 1]
        aJ = [off[cols == j][0] for j in J]
        nneg = npos = cneg = cpos = 0.0
        for v in off:
            if v < 0:
                nneg += v
            else:
                npos += v
        for v in aJ:
            if v < 0:
                cneg += v
            else:
                cpos += v
        if not (cpos == 0.0 and npos != 0.0):
            continue
        d = A.data[b] + npos
        alfa = nneg / cneg / d
        want = [-(alfa * v) for v in aJ]
        assert np.array_equal(cj[rp[i]:rp[i + 1]], f2c[J]) and np.array_equal(va[rp[i]:rp[i + 1]], want), i
        checked += 1
        if checked == 20:
            break
    assert checked > 0


def test_large_lap7_matches_restatement(gpu):
    """128^3 = 2 097 152 rows: the warp S2 / product kernels and sliced-ELL on the aggressive level."""
    A_in, b = O.gen("lap7", 128, 128, 128)
    A = device_storage(A_in)
    H, dA, M = compare_aggressive_hierarchy(A, dict(num_levels=1))
    assert (H.passes(0) >= 3).any()
    _solves(H, dA, M, A, b, ("pcg",))


# (environment, kernels that must run): the default selection and the forced one-thread-per-row paths
FORCED = {
    "default": ({}, {"k_s2_warp<false>", "k_s2_warp<true>", "k_mp_warp<false>", "k_mp_warp<true>", "k_mp_pass2<true>"}),
    "thread": ({"HDK_AGG_THREAD": "1"}, {"k_s2_thread_count", "k_s2_thread_fill", "k_mp_thread_count", "k_mp_thread_fill"}),
}


@pytest.mark.parametrize("mode", list(FORCED))
def test_forced_paths_run_the_aggressive_kernels(gpu, mode):
    env_extra, want = FORCED[mode]
    env = dict(os.environ)
    env.update(env_extra)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "aggressive_paths_check.py"), "heavy_tailed", "arrow"],
                       env=env, capture_output=True, text=True, timeout=900)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("KERNELS ")]
    assert line, out[-3000:]
    ran = {k.replace("void ", "").replace("hdk::", "") for k in line[-1][8:].split("|")}
    assert want <= ran, (sorted(want - ran), sorted(ran))


def test_api_aggressive_yaml(gpu):
    A_in, b = O.gen("lap7", 24, 24, 24)
    A = device_storage(A_in)
    tol = 1e-8
    opts = {"general": {"statistics": False}, "solver": {"pcg": {"relative_tol": tol, "max_iter": 200}},
            "preconditioner": {"amg": {"aggressive": {"num_levels": 1}}}}
    L = driver.api()
    with driver.HypreDrive(options=opts) as drv:
        drv.set_matrix_from_csr(A.indptr.astype(np.int64), A.indices.astype(np.int64), A.data)
        drv.set_rhs(b)
        driver._check(L.HYPREDRV_LinearSystemSetInitialGuess(drv._h, None), "SetInitialGuess")
        driver._check(L.HYPREDRV_LinearSystemResetInitialGuess(drv._h), "ResetInitialGuess")
        driver._check(L.HYPREDRV_LinearSolverCreate(drv._h), "LinearSolverCreate")
        driver._check(L.HYPREDRV_LinearSolverSetup(drv._h), "LinearSolverSetup")
        driver._check(L.HYPREDRV_LinearSolverApply(drv._h), "LinearSolverApply")
        it = C.c_int()
        driver._check(L.HYPREDRV_LinearSolverGetNumIter(drv._h, C.byref(it)), "GetNumIter")
        x = drv.get_solution()
        L.HYPREDRV_LinearSolverDestroy(drv._h)
    H = AO.Hierarchy(A, O.default_params(True), num_levels=1)
    xr, info = O.pcg(A, b, M=H, rel_tol=tol, max_iter=200)
    assert it.value == info["iters"]
    assert np.linalg.norm(x - xr) <= 1e-8 * np.linalg.norm(xr)
    H0 = O.Hierarchy(A, O.default_params(True))
    assert sum(nz for _, nz in H.sizes()) < sum(nz for _, nz in H0.sizes())


def test_invalid_device_parameters(gpu):
    dA = hdk.DCsr.from_scipy(device_storage(O.gen("lap7", 8, 8, 8)[0]))
    for kw in (dict(agg_num_levels=-1), dict(agg_num_levels=1, agg_num_paths=0), dict(agg_num_levels=1, agg_trunc_factor=1.0),
               dict(agg_num_levels=1, agg_max_nnz_row=-1), dict(agg_num_levels=1, agg_interp_type=6),
               dict(agg_num_levels=1, num_functions=3)):
        with pytest.raises(hdk.HdkError):
            hdk.DAmg(dA, hdk.amg_params(**kw))
    hdk.DAmg(dA, hdk.amg_params(agg_num_levels=0, agg_num_paths=0, agg_interp_type=6))   # unused without levels


def _digest(r):
    keep = [l for l in (r.stdout + "\n" + r.stderr).splitlines()
            if any(k in l for k in ("MPAGG", "hdk error", "HdkError", "HypreDriveError", "Error:", "error code", "NCCL WARN"))]
    return "\n".join(keep[-25:]) or (r.stdout[-1500:] + r.stderr[-1500:])


@pytest.mark.parametrize("split", ["even", "ragged"])
def test_two_ranks_match_one_rank(gpu, split):
    env = dict(os.environ)
    env["MPCHECK_RAGGED"] = "1" if split == "ragged" else "0"
    env["HDK_REPLICATE_ROWS"] = "100000000"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29617", os.path.join(ROOT, "tests", "mp_aggressive_check.py"), "24"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, _digest(r)
    assert "ok=True" in r.stdout and "hier=bit-identical" in r.stdout, _digest(r)
