"""GPU parity of Chebyshev smoothing (relax 16) with the CPU restatement (tests/cheby_oracle.c).

Per level the device's D^{-1/2}, l1 norms and, with the Gershgorin estimate, the eigenvalue bounds and
coefficients are compared bit for bit; the CG-Lanczos bounds to 1e-10.  With the device's bounds injected
into the restatement, the V-cycle (zero and nonzero guess) is compared to 1e-11 and the PCG / GMRES solves
by iteration count and solution.  Cases: stencil problems, a 128^3 Laplacian (sliced-ELL), the
unstructured cases of tests/amg_paths.py (one takes the warp-per-row kernel), an elasticity problem with
num_functions = 3 and an aggressive hierarchy.  Also: graph replay against direct launches, the
kernels that ran (child process under torch.profiler), the HYPREDRV API and two ranks."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import aggressive_oracle as AO
import amg_paths as AP
import cheby_oracle as CO
import systems_cases as SC
import systems_oracle as SO
from hypredrive_b200 import driver, hdk
from oracle import oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def device_storage(A):
    """The matrix as the device stores it (diagonal first), as scipy CSR."""
    rp, cj, va = hdk.DCsr.from_scipy(A).diag_arrays()
    return sp.csr_matrix((va.copy(), cj.copy(), rp.copy()), shape=A.shape)


def compare_cheby_hierarchy(A, params_kw, cheb, base=None, dev_kw=None):
    """Device hierarchy against the restatement; returns (restatement with the device's bounds, dA, M)."""
    order, eig_est, scale = cheb.get("order", 2), cheb.get("eig_est", 10), cheb.get("scale", 1)
    if base is None:
        base = O.Hierarchy(A, O.default_params(True, **params_kw))
    dA = hdk.DCsr.from_scipy(A)
    M = hdk.DAmg(dA, hdk.amg_params(**params_kw, **(dev_kw or {}), cheby_order=order, cheby_eig_est=eig_est,
                                    cheby_scale=scale))
    assert M.nlev == base.nlev and M.sizes() == base.sizes(), (M.sizes(), base.sizes())
    ref = CO.Hierarchy(base, order=order, eig_est=eig_est, scale=scale)
    eigs = []
    for l in range(base.nlev):
        assert np.array_equal(M.l1(l), base.l1(l)), f"l1 norms level {l}"
        c = ref.cheby(l)
        if c is None:
            eigs.append(None)
            with pytest.raises(hdk.HdkError):
                M.cheby(l)
            continue
        d = M.cheby(l)
        assert np.array_equal(d["ds"], c["ds"]), f"ds level {l}"
        if eig_est == 0:
            assert d["eig"] == c["eig"], (l, d["eig"], c["eig"])
            assert np.array_equal(d["coefs"], c["coefs"]), (l, d["coefs"], c["coefs"])
        else:
            for i in range(2):
                assert abs(d["eig"][i] - c["eig"][i]) <= 1e-10 * abs(c["eig"][i]), (l, d["eig"], c["eig"])
        eigs.append(d["eig"])
    H = CO.Hierarchy(base, order=order, eig_est=eig_est, scale=scale, eigs=eigs)
    for l, e in enumerate(eigs):
        if e is not None:
            assert np.array_equal(M.cheby(l)["coefs"], H.cheby(l)["coefs"]), f"coefficients level {l}"
    return H, dA, M


def _solves(H, dA, M, A, b, methods=("pcg", "gmres")):
    n = A.shape[0]
    rng = np.random.default_rng(3)
    r, u0 = rng.standard_normal(n), rng.standard_normal(n)
    dr, dz = hdk.DVec(n, r), hdk.DVec(n)
    M.apply(dr, dz)
    z = H.precond(r)
    assert np.allclose(dz.get(), z, rtol=1e-11, atol=1e-11 * np.abs(z).max()), "V-cycle"
    du = hdk.DVec(n, u0)
    M.vcycle(dr, du)
    u = H.vcycle(r, u0)
    assert np.allclose(du.get(), u, rtol=1e-11, atol=1e-11 * np.abs(u).max()), "V-cycle, nonzero guess"
    iters = {}
    for name in methods:
        ofn, dfn = (CO.pcg, hdk.pcg) if name == "pcg" else (CO.gmres, hdk.gmres)
        xr, info = ofn(A, b, M=H, rel_tol=1e-8, max_iter=300)
        db, dx = hdk.DVec(n, b), hdk.DVec(n)
        dx.fill(0.0)
        res = dfn(dA, db, dx, M, max_iter=300, rel_tol=1e-8)
        x = dx.get()
        assert res["converged"] and res["iters"] == info["iters"], (name, res, info["iters"])
        assert np.linalg.norm(x - xr) <= 1e-8 * np.linalg.norm(xr), name
        iters[name] = res["iters"]
    return iters


BOTH = dict(relax_down=16, relax_up=16)
# (problem, Krylov methods, eigenvalue estimates: CG-Lanczos needs a symmetric operator)
STENCILS = {
    "lap7": (lambda: O.gen("lap7", 30, 28, 26), ("pcg", "gmres"), (0, 10)),
    "lap27_aniso": (lambda: O.gen("lap27", 30, 26, 22, c=(1.0, 1.0, 0.01)), ("pcg", "gmres"), (0, 10)),
    "convdif": (lambda: O.gen("convdif", 40, 20, 16, c=(1e-3, 1.0, 0.1)), ("gmres",), (0,)),
}


@pytest.mark.parametrize("name,eig_est", [(n, e) for n, (_, _, ests) in STENCILS.items() for e in ests])
def test_stencil_hierarchy_and_solves_match_restatement(gpu, name, eig_est):
    make, methods, _ = STENCILS[name]
    A_in, b = make()
    A = device_storage(A_in)
    H, dA, M = compare_cheby_hierarchy(A, BOTH, dict(eig_est=eig_est))
    assert H.nlev >= 3
    _solves(H, dA, M, A, b, methods)


# (oracle / device parameters, Chebyshev options, Krylov methods)
CONFIGS = {
    "order1": (BOTH, dict(order=1), ("pcg", "gmres")),
    "order3": (BOTH, dict(order=3), ("pcg", "gmres")),
    "order4": (BOTH, dict(order=4), ("pcg", "gmres")),
    "unscaled": (BOTH, dict(scale=0), ("pcg", "gmres")),
    "unscaled_gershgorin": (BOTH, dict(scale=0, eig_est=0), ("pcg",)),
    "two_sweeps": (dict(BOTH, sweeps_down=2, sweeps_up=2), dict(order=2), ("pcg", "gmres")),
    "down_cheby_up_l1": (dict(relax_down=16, relax_up=18), dict(order=2), ("gmres",)),
    "coarse_one_level": (dict(relax_down=16, relax_up=16, relax_coarse=16, max_levels=1, sweeps_coarse=2), dict(order=2), ("pcg",)),
    "coarse_two_levels": (dict(relax_down=16, relax_up=16, relax_coarse=16, max_levels=2), dict(order=3), ("pcg", "gmres")),
}


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_configurations_match_restatement(gpu, cfg):
    kw, cheb, methods = CONFIGS[cfg]
    A_in, b = O.gen("lap27", 24, 22, 20, c=(1.0, 1.0, 0.1))
    A = device_storage(A_in)
    H, dA, M = compare_cheby_hierarchy(A, kw, cheb)
    _solves(H, dA, M, A, b, methods)


UNSTRUCTURED = ["heavy_tailed", "fe_dirichlet", "fe_rotated_aniso", "signed_graph", "arrow", "scrambled_fe"]


@pytest.mark.parametrize("eig_est", [0, 10])
@pytest.mark.parametrize("name", UNSTRUCTURED)
def test_unstructured_hierarchy_and_solves_match_restatement(gpu, name, eig_est):
    make, params, solver, _ = AP.CASES[name]
    A = device_storage(make())
    b = AP.rhs(A.shape[0])
    H, dA, M = compare_cheby_hierarchy(A, dict(params, **BOTH), dict(eig_est=eig_est))
    _solves(H, dA, M, A, b, (solver,))


def test_long_rows_take_the_vector_kernel(gpu):
    A = device_storage(AP.CASES["arrow"][0]())
    assert hdk.DCsr.from_scipy(A).spmv_kind()["kind"] == 1


def test_elasticity_num_functions_3(gpu):
    A_in, b = SC.elasticity(10, 3)
    A = device_storage(A_in)
    kw = dict(BOTH, strong_th=0.8)
    base = SO.Hierarchy(A, O.default_params(True, **kw), num_functions=3)
    H, dA, M = compare_cheby_hierarchy(A, kw, dict(order=2), base=base, dev_kw=dict(num_functions=3))
    _solves(H, dA, M, A, b, ("pcg",))


def test_aggressive_hierarchy(gpu):
    A_in, b = O.gen("lap7", 30, 28, 26)
    A = device_storage(A_in)
    base = AO.Hierarchy(A, O.default_params(True, **BOTH), num_levels=1)
    H, dA, M = compare_cheby_hierarchy(A, BOTH, dict(order=2), base=base, dev_kw=dict(agg_num_levels=1))
    _solves(H, dA, M, A, b, ("pcg",))


def test_large_lap7_matches_restatement(gpu):
    """128^3 = 2 097 152 rows: the fine levels run the sliced-ELL Chebyshev passes."""
    A_in, b = O.gen("lap7", 128, 128, 128)
    A = device_storage(A_in)
    H, dA, M = compare_cheby_hierarchy(A, BOTH, dict(order=2))
    _solves(H, dA, M, A, b, ("pcg",))


def test_graph_replay_is_bit_identical(gpu):
    A = device_storage(O.gen("lap27", 30, 26, 22, c=(1.0, 1.0, 0.01))[0])
    dA = hdk.DCsr.from_scipy(A)
    M = hdk.DAmg(dA, hdk.amg_params(**BOTH, cheby_order=3))
    n = A.shape[0]
    rng = np.random.default_rng(5)
    r, u0 = rng.standard_normal(n), rng.standard_normal(n)
    out = []
    try:
        for rows in (150000, 0):
            hdk.tune("graph_rows", rows)
            dr, dz, du = hdk.DVec(n, r), hdk.DVec(n), hdk.DVec(n, u0)
            M.apply(dr, dz)
            M.apply(dr, dz)
            M.vcycle(dr, du)
            out.append((dz.get(), du.get()))
    finally:
        hdk.tune("graph_rows", 150000)
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])


def test_chebyshev_kernels_run_on_sliced_ell_and_stream(gpu):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "cheby_paths_check.py")],
                       capture_output=True, text=True, timeout=1800)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("KERNELS ")]
    assert line, out[-3000:]
    ran = line[-1]
    for kern in ("k_spmv_sell", "k_spmv_tma"):
        for mode in (10, 11, 12):
            assert f"{kern}<{mode}," in ran, (kern, mode, ran)


def test_time_kernel_chebyshev_sweep(gpu):
    A = device_storage(O.gen("lap7", 40, 40, 40)[0])
    dA = hdk.DCsr.from_scipy(A)
    M = hdk.DAmg(dA, hdk.amg_params(**BOTH, cheby_order=2))
    ms, by = hdk.time_kernel(dA, M, 9, reps=5)
    n, nnz = A.shape[0], A.nnz
    assert ms > 0 and by == 2 * (12.0 * nnz + 4.0 * (n + 1)) + 80.0 * n
    with pytest.raises(hdk.HdkError):
        hdk.time_kernel(dA, hdk.DAmg(dA, hdk.amg_params()), 9, reps=1)
    assert M.vcycle_bytes() > hdk.DAmg(dA, hdk.amg_params()).vcycle_bytes()


def test_invalid_device_parameters(gpu):
    dA = hdk.DCsr.from_scipy(device_storage(O.gen("lap7", 8, 8, 8)[0]))
    for kw in (dict(cheby_order=0), dict(cheby_order=5), dict(cheby_fraction=0.0), dict(cheby_fraction=1.5),
               dict(cheby_eig_est=-1), dict(cheby_variant=1), dict(cheby_variant=2), dict(cheby_scale=2)):
        with pytest.raises(hdk.HdkError):
            hdk.DAmg(dA, hdk.amg_params(**BOTH, **kw))
    hdk.DAmg(dA, hdk.amg_params(cheby_order=9, cheby_variant=1))   # unused without relaxation 16
    Z = sp.csr_matrix(np.array([[0.0, 1.0], [1.0, 2.0]]))
    with pytest.raises(hdk.HdkError):
        hdk.DAmg(hdk.DCsr.from_scipy(Z), hdk.amg_params(relax_down=16, relax_up=16, relax_coarse=16, max_levels=1))


def test_api_chebyshev_yaml(gpu, capfd):
    A_in, b = O.gen("lap7", 24, 24, 24)
    A = device_storage(A_in)
    tol = 1e-8
    opts = {"general": {"statistics": True}, "solver": {"pcg": {"relative_tol": tol, "max_iter": 200}},
            "preconditioner": {"amg": {"relaxation": {"down_type": "chebyshev", "up_type": "chebyshev",
                                                      "chebyshev": {"order": 3}}}}}
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
        drv.stats_print()
        L.HYPREDRV_LinearSolverDestroy(drv._h)
    printed = capfd.readouterr().out
    base = O.Hierarchy(A, O.default_params(True, **BOTH))
    H = CO.Hierarchy(base, order=3)
    xr, info = CO.pcg(A, b, M=H, rel_tol=tol, max_iter=200)
    assert abs(it.value - info["iters"]) <= 1
    assert np.linalg.norm(x - xr) <= 1e-7 * np.linalg.norm(xr)
    assert np.linalg.norm(b - A @ x) <= tol * np.linalg.norm(b) * 1.0001
    assert "STATISTICS SUMMARY" in printed, printed[-2000:]


def _digest(r):
    keep = [l for l in (r.stdout + "\n" + r.stderr).splitlines()
            if any(k in l for k in ("MPCHEB", "hdk error", "HdkError", "HypreDriveError", "Error:", "error code", "NCCL WARN"))]
    return "\n".join(keep[-25:]) or (r.stdout[-1500:] + r.stderr[-1500:])


@pytest.mark.parametrize("split", ["even", "ragged"])
def test_two_ranks_match_one_rank(gpu, split):
    env = dict(os.environ)
    env["MPCHECK_RAGGED"] = "1" if split == "ragged" else "0"
    env["HDK_REPLICATE_ROWS"] = "2000"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29627", os.path.join(ROOT, "tests", "mp_cheby_check.py"), "24"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, _digest(r)
    assert r.stdout.count("ok=True") == 2, _digest(r)


def test_api_elasticity_settings_with_chebyshev(gpu):
    """The `elasticity_3d` preset's settings (num_functions 3, strong_th 0.8) with Chebyshev smoothing
    through the HYPREDRV API (a preset names the whole preconditioner, so the settings are spelled out)."""
    A_in, b = SC.elasticity(10, 3)
    A = device_storage(A_in)
    tol = 1e-8
    opts = {"general": {"statistics": False}, "solver": {"pcg": {"relative_tol": tol, "max_iter": 200}},
            "preconditioner": {"amg": {"coarsening": {"num_functions": 3, "strong_th": 0.8},
                                       "relaxation": {"down_type": "chebyshev", "up_type": "chebyshev"}}}}
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
    base = SO.Hierarchy(A, O.default_params(True, strong_th=0.8, **BOTH), num_functions=3)
    H = CO.Hierarchy(base, order=2)
    xr, info = CO.pcg(A, b, M=H, rel_tol=tol, max_iter=200)
    assert abs(it.value - info["iters"]) <= 1
    assert np.linalg.norm(x - xr) <= 1e-7 * np.linalg.norm(xr)
    assert np.linalg.norm(b - A @ x) <= tol * np.linalg.norm(b) * 1.0001
