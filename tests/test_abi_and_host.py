"""CPU tests: the C-ABI library loads and exports every declared symbol, and the host-side
logic (YAML subset parser, option tables, presets, overrides, argument validation, error
bitfield) behaves like the reference's.  No compute call is made without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from hypredrive_b200 import driver, hdk

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID_KEY, INVALID_VAL, MISSING_KEY, TREE_INVALID = 0x100, 0x200, 0x1000, 0x20
INVALID_SOLVER, INVALID_PRECON, UNKNOWN_OBJ, NOT_INIT = 0x20000, 0x40000, 0x200000, 0x400000


def _declared(header, prefix):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = "\n".join(l for l in text.splitlines() if not l.lstrip().startswith("#"))   # macros are not exports
    return sorted(set(re.findall(r"\b(%s\w+)\s*\(" % prefix, text)))


def test_library_exports_every_declared_symbol():
    L = hdk.lib()
    names = _declared("HYPREDRV.h", "HYPREDRV_") + _declared("hdk.h", "hdk_") + _declared("HYPRE.h", "HYPRE_") + \
        _declared("mpi.h", "MPI_")
    names = [n for n in names if n not in ("HYPREDRV_SAFE_CALL", "HYPREDRV_SAFE_CALL_COMM", "HYPREDRV_SUCCESS")]
    assert len(names) > 150
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing


def test_scalar_widths():
    L = hdk.lib()
    assert L.HYPREDRV_SizeofBigInt() == 8 and L.HYPREDRV_SizeofReal() == 8 and L.HYPREDRV_SizeofInt() == 4


def _obj():
    driver.initialize()
    h = C.c_void_p()
    assert driver.api().HYPREDRV_Create(1, C.byref(h)) == 0
    assert driver.api().HYPREDRV_SetLibraryMode(h) == 0
    return h


def _parse(h, text, *over):
    argv = [text.encode()] + [o.encode() for o in over]
    arr = (C.c_char_p * len(argv))(*argv)
    code = driver.api().HYPREDRV_InputArgsParse(len(argv), arr, h)
    driver.api().HYPREDRV_ErrorCodeClear()
    return code


def test_yaml_forms_accepted():
    h = _obj()
    good = [
        "solver: pcg\npreconditioner: amg\n",
        "solver: PCG\npreconditioner: AMG\n",                                   # values are lower-cased
        "general:\n  use_millisec: on # comment\n\nsolver: gmres\npreconditioner:\n  preset: poisson\n",
        "solver:\n  pcg:\n    max_iter: 50\n    relative_tol: 1.0e-8\npreconditioner:\n  amg:\n    coarsening:\n      type: pmis\n"
        "      strong_th: 0.5\n    interpolation:\n      prolongation_type: extended+i\n      max_nnz_row: 4\n"
        "    relaxation:\n      down_type: l1-jacobi\n      up_type: 18\n      coarse_type: ge\n",
        "solver:\n    gmres:\n        krylov_dim: 20\npreconditioner: jacobi\n",  # 4-space base indent
        "solver: pcg\npreconditioner:\n  amg: { print_level: 0, coarsening: { type: pmis, max_levels: 10 } }\n",
        "solver: pcg\npreconditioner:\n  amg:\n    - print_level: 0\n      coarsening:\n        type: pmis\n",
        # static preconditioner reuse (docs/usrman-src/input_structure.rst "Static reuse")
        "solver: pcg\npreconditioner:\n  amg:\n    print_level: 0\n  reuse:\n    enabled: yes\n    frequency: 2\n",
        "solver: pcg\npreconditioner:\n  amg:\n    print_level: 0\n  reuse:\n    enabled: yes\n    linear_system_ids: [0, 10, 20]\n",
        "solver: pcg\npreconditioner:\n  amg:\n    print_level: 0\n  reuse: 3\n",
    ]
    for text in good:
        assert _parse(h, text) == 0, text
    assert _parse(h, "solver: pcg\npreconditioner: amg\n", "--solver:pcg:relative_tol", "1.0e-2") == 0
    assert _parse(h, "solver: pcg\npreconditioner: amg\n", "-a", "--solver:pcg:max_iter", "7", "--general:name", "run.yml") == 0
    driver.api().HYPREDRV_Destroy(C.byref(h))


def test_yaml_include_scalar_and_list_forms(tmp_path):
    """`include: file` splices a fragment; `include:` + a list of files makes one preconditioner
    variant per file (reference examples/ex8-multi-1.yml with ex8-amg-N.yml fragments)."""
    (tmp_path / "v1.yml").write_text("coarsening:\n  type: pmis\n  strong_th: 0.25\nrelaxation:\n  down_type: l1-jacobi\n  up_type: l1-jacobi\n")
    (tmp_path / "v2.yml").write_text("coarsening:\n  type: pmis\n  strong_th: 0.5\n")
    (tmp_path / "krylov.yml").write_text("pcg:\n  max_iter: 77\n")
    main = tmp_path / "main.yml"
    main.write_text("solver:\n  include: krylov.yml\npreconditioner:\n  amg:\n    include:\n      - v1.yml\n      - v2.yml\n")
    h = _obj()
    assert _parse(h, str(main)) == 0
    nv = C.c_int()
    driver.api().HYPREDRV_InputArgsGetNumPreconVariants(h, C.byref(nv))
    assert nv.value == 2
    (tmp_path / "bad.yml").write_text("solver: pcg\npreconditioner:\n  amg:\n    include:\n      - missing.yml\n")
    assert _parse(h, str(tmp_path / "bad.yml")) != 0          # missing fragment: FILE_NOT_FOUND bit
    driver.api().HYPREDRV_Destroy(C.byref(h))


def test_yaml_errors_set_the_reference_error_bits():
    h = _obj()
    cases = [
        ("solver: pcg\n", MISSING_KEY),                                          # preconditioner is mandatory
        ("solver: pcg\npreconditioner: amg\nbogus: 1\n", INVALID_KEY),
        ("solver:\n  pcg:\n    max_itr: 5\npreconditioner: amg\n", INVALID_KEY),
        ("solver:\n  pcg:\n    max_iter: many\npreconditioner: amg\n", INVALID_VAL),
        ("solver: pcg\npreconditioner:\n  amg:\n    coarsening:\n      type: banana\n", INVALID_VAL),
        ("solver: lgmres\npreconditioner: amg\n", INVALID_SOLVER),
        ("solver: pcg\npreconditioner: mgr\n", INVALID_PRECON),
        ("solver: pcg\n\tpreconditioner: amg\n", 0x41),                           # tab indentation
        ("solver:\n  pcg:\n   max_iter: 5\npreconditioner: amg\n", 0x4),          # inconsistent indent
        ("solver:\n      pcg:\n        max_iter: 5\n  x: 1\npreconditioner: amg\n", 0x4 | 0x80 | INVALID_KEY),
        ("solver pcg\npreconditioner: amg\n", 0x8),                               # missing divisor
        ("solver: pcg\npreconditioner:\n  amg:\n    print_level: 0\n  reuse: adaptive\n", INVALID_VAL),      # static only
        ("solver: pcg\npreconditioner:\n  amg:\n    print_level: 0\n  reuse:\n    frequency: -1\n", INVALID_VAL),
        ("solver: pcg\npreconditioner:\n  amg:\n    print_level: 0\n  reuse:\n    enabled: yes\n    cadence: 2\n", INVALID_KEY),
    ]
    for text, bits in cases:
        code = _parse(h, text)
        assert code & bits, (text, hex(code))
    assert _parse(h, "solver: pcg\npreconditioner: amg\n", "--solver:pcg:max_iter") & INVALID_VAL   # odd token count
    driver.api().HYPREDRV_Destroy(C.byref(h))


def test_guards_and_argument_validation():
    L = driver.api()
    h = _obj()
    bogus = C.c_void_p(12345)
    assert L.HYPREDRV_LinearSolverCreate(bogus) & UNKNOWN_OBJ
    L.HYPREDRV_ErrorCodeClear()
    assert L.HYPREDRV_LinearSolverCreate(h) & MISSING_KEY           # no input args parsed yet
    L.HYPREDRV_ErrorCodeClear()
    one = np.array([0], dtype=np.int64)
    # tests/test_setmatrix_from_csr.c:249-350
    assert L.HYPREDRV_LinearSystemSetMatrixFromCSR(h, 0, 4, None, None, None) & INVALID_VAL
    L.HYPREDRV_ErrorCodeClear()
    assert L.HYPREDRV_LinearSystemSetMatrixFromCSR(h, 5, 4, one.ctypes.data, None, None) & INVALID_VAL
    L.HYPREDRV_ErrorCodeClear()
    ip = np.array([0, 1], dtype=np.int64)
    assert L.HYPREDRV_LinearSystemSetMatrixFromCSR(h, 0, 0, ip.ctypes.data, None, None) & INVALID_VAL
    L.HYPREDRV_ErrorCodeClear()
    neg = np.array([-1, 0], dtype=np.int64)
    cj, va = np.array([0], dtype=np.int64), np.array([1.0])
    assert L.HYPREDRV_LinearSystemSetMatrixFromCSR(h, 0, 0, neg.ctypes.data, cj.ctypes.data, va.ctypes.data) & INVALID_VAL
    L.HYPREDRV_ErrorCodeClear()
    bad = np.array([0, 2, 1, 3], dtype=np.int64)
    c3, v3 = np.array([0, 1, 2], dtype=np.int64), np.ones(3)
    assert L.HYPREDRV_LinearSystemSetMatrixFromCSR(h, 0, 2, bad.ctypes.data, c3.ctypes.data, v3.ctypes.data) & INVALID_VAL
    L.HYPREDRV_ErrorCodeClear()
    assert L.HYPREDRV_LinearSystemSetRHSFromArray(h, 0, 4, None) & INVALID_VAL
    L.HYPREDRV_ErrorCodeClear()
    assert L.HYPREDRV_LinearSystemSetRHSFromArray(h, 5, 4, va.ctypes.data) & INVALID_VAL
    L.HYPREDRV_ErrorCodeClear()
    assert L.HYPREDRV_LinearSystemSetRHSFromArray(h, 0, 0, va.ctypes.data) & INVALID_VAL    # RHS before matrix
    L.HYPREDRV_ErrorCodeClear()
    assert L.HYPREDRV_Destroy(C.byref(h)) == 0
    assert L.HYPREDRV_Destroy(C.byref(h)) & UNKNOWN_OBJ                                      # already destroyed
    L.HYPREDRV_ErrorCodeClear()


def test_no_cpu_fallback_without_a_gpu():
    if hdk.device_count() > 0:
        pytest.skip("a GPU is visible")
    ip = np.array([0, 1], dtype=np.int64)
    cj, va = np.array([0], dtype=np.int64), np.array([3.0])
    with pytest.raises(driver.HypreDriveError) as e:
        with driver.HypreDrive() as drv:
            drv.set_matrix_from_csr(ip, cj, va)
    assert "no CUDA device" in str(e.value) and e.value.code & 0x01000000


def test_ij_shim_containers():
    L = hdk.lib()
    A = C.c_void_p()
    assert L.HYPRE_IJMatrixCreate(1, C.c_longlong(0), C.c_longlong(2), C.c_longlong(0), C.c_longlong(2), C.byref(A)) == 0
    L.HYPRE_IJMatrixSetObjectType(A, 5555)
    L.HYPRE_IJMatrixInitialize(A)
    for r, (cols, vals) in enumerate([([0, 1], [2.0, -1.0]), ([0, 1, 2], [-1.0, 2.0, -1.0]), ([1, 2], [-1.0, 2.0])]):
        n = C.c_int(len(cols))
        row = C.c_longlong(r)
        cc = (C.c_longlong * len(cols))(*cols)
        vv = (C.c_double * len(vals))(*vals)
        assert L.HYPRE_IJMatrixSetValues(A, 1, C.byref(n), C.byref(row), cc, vv) == 0
    assert L.HYPRE_IJMatrixAssemble(A) == 0
    lo, hi = C.c_longlong(), C.c_longlong()
    L.HYPRE_IJMatrixGetLocalRange(A, C.byref(lo), C.byref(hi), None, None)
    assert (lo.value, hi.value) == (0, 2)
    v = C.c_void_p()
    assert L.HYPRE_IJVectorCreate(1, C.c_longlong(0), C.c_longlong(2), C.byref(v)) == 0
    L.HYPRE_IJVectorInitialize(v)
    idx = (C.c_longlong * 3)(0, 1, 2)
    val = (C.c_double * 3)(1.0, 2.0, 3.0)
    L.HYPRE_IJVectorSetValues(v, 3, idx, val)
    out = (C.c_double * 3)()
    L.HYPRE_IJVectorGetValues(v, 3, idx, out)
    assert list(out) == [1.0, 2.0, 3.0]
    assert L.HYPRE_IJVectorDestroy(v) == 0 and L.HYPRE_IJMatrixDestroy(A) == 0


def test_mpi_shim_cartesian_and_point_to_point(monkeypatch):
    """include/mpi.h without an MPI library: one process is exact (every Cartesian neighbour is
    MPI_PROC_NULL, point-to-point calls to it succeed and move nothing); with several processes of
    the launcher environment the Cartesian calls follow MPI's row-major rank order, and a
    point-to-point call to a real peer fails instead of returning wrong data."""
    L = hdk.lib()
    WORLD, PROC_NULL, INT = 1, -2, 1
    I3 = C.c_int * 3
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    monkeypatch.delenv("RANK", raising=False)
    cart, src, dst, req, coords = C.c_int(), C.c_int(), C.c_int(), C.c_int(7), I3()
    assert L.MPI_Cart_create(WORLD, 3, I3(1, 1, 1), I3(0, 0, 0), 0, C.byref(cart)) == 0
    for d in range(3):
        assert L.MPI_Cart_shift(cart, d, 1, C.byref(src), C.byref(dst)) == 0
        assert (src.value, dst.value) == (PROC_NULL, PROC_NULL)
    buf = (C.c_int * 4)(1, 2, 3, 4)
    assert L.MPI_Isend(buf, 4, INT, PROC_NULL, 0, cart, C.byref(req)) == 0 and req.value == 0
    assert L.MPI_Irecv(buf, 4, INT, PROC_NULL, 0, cart, C.byref(req)) == 0 and list(buf) == [1, 2, 3, 4]
    assert L.MPI_Waitall(0, None, None) == 0
    assert L.MPI_Comm_free(C.byref(cart)) == 0 and cart.value == 0
    # rank 1 of a 1 x 1 x 2 grid
    monkeypatch.setenv("WORLD_SIZE", "2")
    monkeypatch.setenv("RANK", "1")
    assert L.MPI_Cart_create(WORLD, 3, I3(1, 1, 3), I3(0, 0, 0), 0, C.byref(cart)) != 0   # 3 processes on 2
    assert L.MPI_Cart_create(WORLD, 3, I3(1, 1, 2), I3(0, 0, 0), 0, C.byref(cart)) == 0
    assert L.MPI_Cart_coords(cart, 1, 3, coords) == 0 and list(coords) == [0, 0, 1]
    r = C.c_int()
    assert L.MPI_Cart_rank(cart, I3(0, 0, 0), C.byref(r)) == 0 and r.value == 0
    assert L.MPI_Cart_shift(cart, 2, 1, C.byref(src), C.byref(dst)) == 0 and (src.value, dst.value) == (0, PROC_NULL)
    assert L.MPI_Cart_shift(cart, 0, 1, C.byref(src), C.byref(dst)) == 0 and (src.value, dst.value) == (PROC_NULL, PROC_NULL)
    assert L.MPI_Isend(buf, 4, INT, 0, 0, cart, C.byref(req)) != 0
    assert L.MPI_Irecv(buf, 4, INT, 0, 0, cart, C.byref(req)) != 0
    assert L.MPI_Isend(buf, 4, INT, PROC_NULL, 0, cart, C.byref(req)) == 0
    assert L.MPI_Comm_free(C.byref(cart)) == 0


def test_options_dict_to_yaml():
    y = driver.normalize_options({"general": {"statistics": False}, "solver": {"pcg": {"max_iter": 10}},
                                  "preconditioner": {"amg": {"print_level": 0}}})
    assert "statistics: off" in y and "    max_iter: 10" in y and y.startswith("general:")


def test_sliced_ell_kernel_register_budget():
    """Occupancy guard for the kernel that is 80 % of a solve: the plain sliced-ELL variants must
    compile to <= 32 registers (8 CTAs of 256 threads per SM) and the fused-dot / fused-offd
    variants to <= 40 (6 CTAs), without spills -- ptxas is touchy here (DESIGN.md section 4)."""
    import re
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    lib = os.path.join(ROOT, "hypredrive_b200", "lib", "libHYPREDRV.so")
    out = subprocess.run([cuobjdump, "--dump-resource-usage", lib], capture_output=True, text=True).stdout
    found = re.findall(r"Function _ZN3hdk11k_spmv_sellILi(\d)ELb([01])ELb([01])ELb([01])EEEvNS_7SpmvDevE:\s*\n\s*REG:(\d+) STACK:(\d+)", out)
    assert len(found) >= 54, len(found)     # 9 epilogue modes x fused dot x {one rank, multi-rank, multi-rank + folded export}
    for mode, dot, offd, exp, reg, stack in found:
        # 32 registers = 8 CTAs per SM: every plain variant, and the multi-rank variants of the three modes
        # without smoother operands (SET, RESIDUAL, ADD) -- also when they fold the halo export, which is
        # why every product folds; mode 7 (two-stage GS first stage) writes two vectors per row: 40 also
        # when plain
        lean = dot == "0" and mode != "7" and (offd == "0" or mode in "013")
        limit = 32 if lean else 40
        assert int(reg) <= limit, (mode, dot, offd, exp, reg)
        assert int(stack) <= 8, (mode, dot, offd, exp, stack)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the restated reference on the host cores) prints one JSON line
    with the contract's keys; a small sample keeps the test short."""
    import json
    import subprocess
    import sys
    # torchrun exports OMP_NUM_THREADS=1 to its children: the arm must override it by assignment
    env = dict(os.environ, OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--n", "40"], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "DOF*iters/s" and line["value"] > 0
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["dtype"] == "f64"
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and "40x40x40" in line["config"]["workload"]
    assert line["steps"] == 2 and line["warmup"] == 1
    assert line["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    # the two arms must print the same metric / unit / direction or the driver cannot form a ratio
    sys.path.insert(0, ROOT)
    import bench
    assert line["metric"] == bench.CONFIGS["lap7_256"]["metric"]
    for name, cfg in bench.CONFIGS.items():
        assert cfg["scaling"] in ("weak", "strong") and cfg["solver"] in ("pcg", "gmres"), name
