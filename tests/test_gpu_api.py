"""GPU tests through the drop-in boundary: the HYPREDRV_* C API (ctypes) driven the way the
reference's own tests drive it (tests/test_setmatrix_from_csr.c, interfaces/python/tests/
test_solve_serial.py), with results checked against the CPU oracle."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

import hypredrive_b200 as hd
from hypredrive_b200 import driver
from oracle import oracle as O

pytestmark = pytest.mark.gpu

BASE = {"general": {"statistics": False, "exec_policy": "device"}, "linear_system": {"init_guess_mode": "zeros"},
        "solver": {"pcg": {"max_iter": 100, "relative_tol": 1.0e-8, "print_level": 0}},
        "preconditioner": {"amg": {"print_level": 0}}}


def lap1d(n):
    A = sp.diags([-1.0, 2.0, -1.0], [-1, 0, 1], shape=(n, n)).tocsr()
    return A.indptr.astype(np.int64), A.indices.astype(np.int64), A.data.copy(), np.ones(n), A


def test_driver_lifecycle_and_determinism(gpu):
    indptr, cols, data, rhs, A = lap1d(32)
    with hd.HypreDrive(options=BASE) as drv:
        drv.set_matrix_from_csr(indptr, cols, data, row_start=0, row_end=31)
        drv.set_rhs(rhs)
        drv.solve()
        x1 = drv.get_solution()
        assert drv.last_converged is True and drv.last_final_res_norm >= 0.0
        with pytest.raises(ValueError, match="kind must be one of"):
            drv.solution_norm("bad")
        drv.set_rhs(rhs)
        drv.solve()
        x2 = drv.get_solution()
        assert abs(drv.solution_norm("l2") - np.linalg.norm(x2)) <= 1e-12 * np.linalg.norm(x2)
        assert abs(drv.solution_norm("inf") - np.abs(x2).max()) <= 1e-12 * np.abs(x2).max()
    np.testing.assert_allclose(x1, x2, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(A @ x1, rhs, rtol=0, atol=1e-6)


def test_input_args_override(gpu):
    indptr, cols, data, rhs, _ = lap1d(32)

    def run(input_args=None):
        with hd.HypreDrive(options=BASE, input_args=input_args) as drv:
            drv.set_matrix_from_csr(indptr, cols, data, row_start=0, row_end=31)
            drv.set_rhs(rhs)
            drv.solve()
            assert drv.last_converged is True
            return drv.last_iterations

    baseline = run()
    loose = run(["--solver:pcg:relative_tol", "1.0e-2"])
    assert loose < baseline
    assert run(["-a", "--solver:pcg:relative_tol", "1.0e-2"]) == loose
    assert run(["--general:name", "run.yml"]) == baseline


def test_known_answers_and_matrix_replacement(gpu):
    indptr = np.array([0, 1, 2], dtype=np.int64)
    cols = np.array([0, 1], dtype=np.int64)
    rhs = np.array([8.0, 16.0])
    with hd.HypreDrive(options=BASE) as drv:
        drv.set_matrix_from_csr((indptr, cols, np.array([2.0, 4.0])), row_start=0, row_end=1)
        drv.set_rhs(rhs)
        drv.solve()
        np.testing.assert_allclose(drv.get_solution(), [4.0, 4.0], atol=1e-6)
        drv.set_matrix_from_csr((indptr, cols, np.array([4.0, 8.0])), row_start=0, row_end=1)
        drv.set_rhs(rhs)
        drv.solve()
        np.testing.assert_allclose(drv.get_solution(), [2.0, 2.0], atol=1e-6)
    res = hd.solve(sp.diags([1.0, 2.0, 3.0, 4.0]).tocsr(), np.array([1.0, 4.0, 9.0, 16.0]), options=BASE)
    np.testing.assert_allclose(res.x, [1, 2, 3, 4], atol=1e-6)
    # 1x1 system 3x = 6 -> ||x|| = 2 (tests/test_setmatrix_from_csr.c:395-421), with an offset indptr slab
    ip = np.array([2, 3], dtype=np.int64)
    cj = np.array([99, 99, 0], dtype=np.int64)
    va = np.array([0.0, 0.0, 3.0])
    with hd.HypreDrive(options=BASE) as drv:
        drv.set_matrix_from_csr(ip, cj, va, row_start=0, row_end=0)
        drv.set_rhs(np.array([6.0]))
        drv.solve()
        assert abs(drv.solution_norm("l2") - 2.0) < 1e-6


def test_static_preconditioner_reuse(gpu):
    """preconditioner.reuse (static policy): rebuild when ls_index % (frequency + 1) == 0, otherwise
    keep the hierarchy of the earlier matrix (reference src/internal/precon_reuse.c:780-830)."""
    A, b = O.gen("lap7", 12, 10, 8)
    opts = {"general": {"statistics": False}, "solver": {"pcg": {"relative_tol": 1e-8, "max_iter": 100}},
            "preconditioner": {"amg": {"print_level": 0}, "reuse": {"enabled": True, "frequency": 1}}}
    setups, iters = [], []
    with hd.HypreDrive(options=opts) as drv:
        for k in range(4):
            Ak = (A + 0.05 * k * sp.eye(A.shape[0])).tocsr()        # a slowly changing operator
            drv.set_matrix_from_csr(Ak)
            drv.set_rhs(b)
            drv.solve()
            assert drv.last_converged
            x = drv.get_solution()
            assert np.linalg.norm(b - Ak @ x) <= 1e-8 * np.linalg.norm(b) * 1.0001
            setups.append(drv.last_setup_time)
            iters.append(drv.last_iterations)
    assert setups[0] > 0 and setups[2] > 0            # systems 0 and 2: rebuilt
    assert setups[1] == 0 and setups[3] == 0          # systems 1 and 3: reused
    # explicit rebuild list
    opts["preconditioner"]["reuse"] = {"enabled": True, "linear_system_ids": [0, 3]}
    setups = []
    with hd.HypreDrive(options=opts) as drv:
        for k in range(4):
            drv.set_matrix_from_csr(A)
            drv.set_rhs(b)
            drv.solve()
            assert drv.last_converged
            setups.append(drv.last_setup_time)
    assert [s > 0 for s in setups] == [True, False, False, True]


def test_unsorted_columns_and_diag_swap(gpu):
    # rows given with the diagonal last (27-pt generator style): assembly swaps it to the front
    A, b = O.gen("lap27", 8, 7, 6, c=(1.0, 1.0, 0.01), diag_first=False)
    res = hd.solve((A.indptr, A.indices, A.data), b, options=BASE, row_start=0, row_end=A.shape[0] - 1)
    Ad, _ = O.gen("lap27", 8, 7, 6, c=(1.0, 1.0, 0.01))
    H = O.Hierarchy(Ad, O.default_params(True))
    xr, ir = O.pcg(Ad, b, M=H, rel_tol=1e-8)
    assert res.iterations == ir["iters"]
    assert np.linalg.norm(res.x - xr) <= 1e-8 * np.linalg.norm(xr)


@pytest.mark.parametrize("solver,kind,dims,c,tol", [("pcg", "lap7", (20, 20, 20), (1, 1, 1), 1e-6),
                                                   ("gmres", "convdif", (32, 8, 8), (1e-3, 1.0, 0.1), 1e-8),
                                                   ("pcg", "lap27", (12, 12, 12), (1, 1, 0.01), 1e-6)])
def test_api_solve_matches_oracle(gpu, solver, kind, dims, c, tol):
    A, b = O.gen(kind, *dims, c=c)
    opts = {"solver": {solver: {"relative_tol": tol, "max_iter": 100}},
            "preconditioner": {"amg": {"coarsening": {"type": "pmis"}, "relaxation": {"down_type": "l1-jacobi", "up_type": "l1-jacobi"}}}}
    res = hd.solve(A, b, options=opts)
    H = O.Hierarchy(A, O.default_params(True))
    xr, ir = (O.pcg if solver == "pcg" else O.gmres)(A, b, M=H, rel_tol=tol, max_iter=100)
    assert res.converged and abs(res.iterations - ir["iters"]) <= 1
    assert np.linalg.norm(res.x - xr) <= 1e-8 * np.linalg.norm(xr)
    assert np.linalg.norm(b - A @ res.x) <= tol * np.linalg.norm(b) * 1.0001
    assert res.setup_time > 0 and res.solve_time > 0


def test_device_stencil_path_and_stats_table(gpu, capfd):
    with hd.HypreDrive(options={"general": {"use_millisec": True}, "solver": "pcg", "preconditioner": "amg"}) as drv:
        drv.set_stencil(7, 10, 10, 10)
        drv.solve()
        it = drv.last_iterations
        x = drv.get_solution()
        drv.stats_print()
    out = capfd.readouterr().out
    A, b = O.gen("lap7", 10, 10, 10)
    H = O.Hierarchy(A, O.default_params(True))
    xr, ir = O.pcg(A, b, M=H, rel_tol=1e-6)
    assert it == ir["iters"] and np.linalg.norm(x - xr) <= 1e-8 * np.linalg.norm(xr)
    assert "STATISTICS SUMMARY" in out and "times [ms]" in out and "1.00e+01" in out
    row = [l for l in out.splitlines() if l.startswith("|      0 |")][0]
    assert row.rstrip().endswith(f"| {it:6d} |")


def test_c_api_ij_interface_and_precon_apply(gpu):
    """HYPRE_IJMatrix/IJVector handles through SetMatrix/SetRHS and HYPREDRV_PreconApply (one V-cycle)."""
    L = driver.api()
    A, b = O.gen("lap7", 8, 8, 8)
    n = A.shape[0]
    ijA, ijb, ijx = C.c_void_p(), C.c_void_p(), C.c_void_p()
    ll = C.c_longlong
    assert L.HYPRE_IJMatrixCreate(1, ll(0), ll(n - 1), ll(0), ll(n - 1), C.byref(ijA)) == 0
    L.HYPRE_IJMatrixSetObjectType(ijA, 5555)
    L.HYPRE_IJMatrixInitialize(ijA)
    for i in range(n):
        s, e = A.indptr[i], A.indptr[i + 1]
        nc, row = C.c_int(e - s), ll(i)
        cc = (ll * (e - s))(*A.indices[s:e].tolist())
        vv = (C.c_double * (e - s))(*A.data[s:e].tolist())
        L.HYPRE_IJMatrixSetValues(ijA, 1, C.byref(nc), C.byref(row), cc, vv)
    L.HYPRE_IJMatrixAssemble(ijA)
    idx = (ll * n)(*range(n))
    for handle, vals in ((ijb, b), (ijx, np.zeros(n))):
        L.HYPRE_IJVectorCreate(1, ll(0), ll(n - 1), C.byref(handle))
        L.HYPRE_IJVectorInitialize(handle)
        L.HYPRE_IJVectorSetValues(handle, n, idx, (C.c_double * n)(*vals.tolist()))
    driver.initialize()
    h = C.c_void_p()
    assert L.HYPREDRV_Create(1, C.byref(h)) == 0
    assert L.HYPREDRV_SetLibraryMode(h) == 0
    assert L.HYPREDRV_InputArgsSetSolverPreset(h, b"pcg") == 0          # laplacian.c:370-371
    assert L.HYPREDRV_InputArgsSetPreconPreset(h, b"poisson") == 0
    L.HYPREDRV_LinearSystemSetMatrix.argtypes = [C.c_void_p, C.c_void_p]
    L.HYPREDRV_PreconApply.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    assert L.HYPREDRV_LinearSystemSetMatrix(h, ijA) == 0
    assert L.HYPREDRV_LinearSystemSetRHS(h, ijb) == 0
    assert L.HYPREDRV_LinearSystemSetInitialGuess(h, None) == 0
    assert L.HYPREDRV_LinearSystemSetPrecMatrix(h, None) == 0
    assert L.HYPREDRV_LinearSolverApply(h) != 0                         # no solver yet: error, not a crash
    L.HYPREDRV_ErrorCodeClear()
    assert L.HYPREDRV_PreconCreate(h) == 0
    assert L.HYPREDRV_PreconSetup(h) == 0
    assert L.HYPREDRV_PreconApply(h, ijb, ijx) == 0
    z = (C.c_double * n)()
    L.HYPRE_IJVectorGetValues(ijx, n, idx, z)
    H = O.Hierarchy(A, O.default_params(True))
    zr = H.precond(b)
    assert np.allclose(np.array(z), zr, rtol=1e-11, atol=1e-14)
    for _ in range(2):                                                   # repeated solves, laplacian.c:445-463
        assert L.HYPREDRV_LinearSystemResetInitialGuess(h) == 0
        assert L.HYPREDRV_LinearSolverCreate(h) == 0
        assert L.HYPREDRV_LinearSolverSetup(h) == 0
        assert L.HYPREDRV_LinearSolverApply(h) == 0
        it = C.c_int()
        L.HYPREDRV_LinearSolverGetNumIter(h, C.byref(it))
        assert L.HYPREDRV_LinearSolverDestroy(h) == 0
    _, ir = O.pcg(A, b, M=H, rel_tol=1e-6)
    assert it.value == ir["iters"]
    assert L.HYPREDRV_Destroy(C.byref(h)) == 0
    L.HYPRE_IJVectorDestroy(ijb); L.HYPRE_IJVectorDestroy(ijx); L.HYPRE_IJMatrixDestroy(ijA)


def test_unsupported_requests_fail_loudly(gpu):
    indptr, cols, data, rhs, _ = lap1d(16)
    opts = dict(BASE, preconditioner="gauss-seidel")                     # sequential GS has no device kernel
    with pytest.raises(hd.HypreDriveError):
        hd.solve((indptr, cols, data), rhs, options=opts, row_start=0, row_end=15)
    res = hd.solve((indptr, cols, data), rhs, options=dict(BASE, preconditioner="jacobi"), row_start=0, row_end=15)
    assert res.converged


@pytest.mark.parametrize("solver", ["fgmres", "bicgstab"])
def test_api_fgmres_bicgstab(gpu, solver):
    A, b = O.gen("convdif", 20, 8, 8, c=(1e-3, 1.0, 0.1))
    res = hd.solve(A, b, options={"solver": {solver: {"relative_tol": 1.0e-8, "max_iter": 60}}, "preconditioner": "amg"})
    assert res.converged and np.linalg.norm(b - A @ res.x) <= 1e-8 * np.linalg.norm(b) * 1.0001


def test_initial_guess_previous_across_two_systems(gpu):
    """init_guess_mode 'previous' (reference src/internal/linsys.c:2044-2063): the second system
    starts from the first system's solution -- a slightly perturbed operator then needs fewer
    iterations than from zeros -- and falls back to zeros when no compatible vector exists."""
    A, b = O.gen("lap7", 12, 10, 8)
    A2 = (A + 1e-3 * sp.eye(A.shape[0])).tocsr()

    def run(mode):
        opts = {"general": {"statistics": False}, "linear_system": {"init_guess_mode": mode},
                "solver": {"pcg": {"relative_tol": 1e-8, "max_iter": 100}}, "preconditioner": "amg"}
        its = []
        with hd.HypreDrive(options=opts) as drv:
            for M in (A, A2):
                drv.set_matrix_from_csr(M)
                drv.set_rhs(b)
                drv.solve()
                assert drv.last_converged
                x = drv.get_solution()
                assert np.linalg.norm(b - M @ x) <= 1e-8 * np.linalg.norm(b) * 1.0001
                its.append(drv.last_iterations)
        return its

    zeros, prev = run("zeros"), run("previous")
    assert prev[0] == zeros[0]                     # first system: no previous solution -> zeros
    assert prev[1] < zeros[1]                      # second system: warm start from the first solution
    # other generated initial guesses still converge to the same solution
    for mode in ("ones", "random"):
        res = hd.solve(A, b, options={"general": {"statistics": False}, "linear_system": {"init_guess_mode": mode},
                                      "solver": {"pcg": {"relative_tol": 1e-9, "max_iter": 100}}, "preconditioner": "amg"})
        assert res.converged and np.linalg.norm(b - A @ res.x) <= 1e-9 * np.linalg.norm(b) * 1.0001


def test_bench_dump_outputs(gpu, tmp_path):
    """`bench.py --dump-outputs DIR` writes what the last of `--steps` timed solves returned: the
    solution at the seeded sample of positions (a 104^3 grid has more than DUMP_SAMPLE rows), its
    iteration count and final relative residual norm.  `--steps` sets how many solves are timed:
    three steps launch three times the kernels of one."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    n = 104

    def run(steps):
        out = tmp_path / f"steps{steps}"
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", str(steps),
                            "--warmup", "1", "--n", str(n), "--no-cpu-baseline", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        return line, [np.load(out / f"{k}.npy") for k in ("solution", "iterations", "final_rel_res_norm")]

    line1, (x1, it1, rr1) = run(1)
    line3, (x3, it3, rr3) = run(3)
    assert line1["gpu_launches"] > 0 and line3["gpu_launches"] == 3 * line1["gpu_launches"]
    idx = bench.dump_positions(n ** 3)
    assert idx.size < n ** 3
    for x, it, rr, line in ((x1, it1, rr1, line1), (x3, it3, rr3, line3)):
        assert x.dtype == it.dtype == rr.dtype == np.float64 and x.shape == idx.shape and it.shape == rr.shape == (1,)
        assert int(it[0]) == line["iterations"] and 0 < rr[0] < 1e-6
    A, b = O.gen("lap7", n, n, n)
    xo, io = O.pcg(A, b, M=O.Hierarchy(A, O.default_params(True)), rel_tol=1e-6, max_iter=100)
    assert int(it1[0]) == int(it3[0]) == io["iters"]
    for x in (x1, x3):
        assert np.linalg.norm(x - xo[idx]) <= 1e-8 * np.linalg.norm(xo[idx])
