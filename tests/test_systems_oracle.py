"""CPU tests of systems AMG (num_functions > 1, hypre's unknown approach) in the CPU restatement
(tests/systems_oracle.c, built on the parity oracle) and in the host option layer.  Its strength pattern is checked against a restatement of the rule in
numpy; P, the coarse labels and the coarse operators are checked for the structure the rule
implies; on decoupled functions the systems hierarchy must equal the scalar one bit for bit."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

import systems_cases as SC
from hypredrive_b200 import driver, hdk
from oracle import oracle as O
import systems_oracle as SO

INVALID_VAL = 0x200


def strength_restated(A, dof, theta, mrs):
    """hypre_BoomerAMGCreateS, num_functions > 1, on diagonal-first storage, one row at a time."""
    rows = []
    for i in range(A.shape[0]):
        b, e = A.indptr[i], A.indptr[i + 1]
        cols, vals = A.indices[b + 1:e], A.data[b + 1:e]
        d = A.data[b]
        same = dof[cols] == dof[i]
        row_sum = d
        for v in vals[same]:                          # stored order, separately rounded additions
            row_sum += v
        scale = vals[same].max(initial=0.0) if d < 0 else vals[same].min(initial=0.0)
        if abs(row_sum) > abs(d) * mrs and mrs < 1.0:
            rows.append(np.zeros(0, dtype=cols.dtype))
            continue
        keep = ~(vals <= theta * scale) if d < 0 else ~(vals >= theta * scale)
        rows.append(cols[keep & same])
    return rows


def _stored(H):
    return H.A(0)                                     # the oracle's diagonal-first copy of the input


@pytest.mark.parametrize("name", ["elasticity_3d", "plane_strain", "block_labels", "ragged"])
@pytest.mark.parametrize("sign", [1.0, -1.0])
def test_strength_matches_restatement(name, sign):
    A, _, nf, dof, th = SC.cases()[name]
    A = (sign * A).tocsr()
    H = SO.Hierarchy(A, O.default_params(True, strong_th=th, max_levels=2), num_functions=nf, dof_func=dof)
    A0 = _stored(H)
    lab = H.dof(0)
    assert np.array_equal(lab, dof if dof is not None else SC.interleaved(A.shape[0], nf))
    S = H.S(0)
    ref = strength_restated(A0, lab, th, 0.9)
    for i, r in enumerate(ref):
        assert np.array_equal(S.indices[S.indptr[i]:S.indptr[i + 1]], r), (name, i)
    # the stand-alone entry gives the same pattern
    S2 = SO.strength(A0, nf, lab, th, 0.9)
    assert np.array_equal(S2.indptr, S.indptr) and np.array_equal(S2.indices, S.indices)
    # no strong cross-function coupling, while the scalar rule has some at the default threshold
    r = np.repeat(np.arange(A.shape[0]), np.diff(S.indptr))
    assert np.all(lab[S.indices] == lab[r])
    Ss = O.strength(A0, 0.25, 0.9)
    rs = np.repeat(np.arange(A.shape[0]), np.diff(Ss.indptr))
    assert np.any(lab[Ss.indices] != lab[rs])


def test_max_row_sum_makes_a_row_weak_only_for_its_own_function():
    """A row whose couplings to its own function are tiny: its own-function row sum is close to the
    diagonal, so max_row_sum = 0.9 makes the whole row weak (it has strong entries before)."""
    A, _, nf, _, _ = SC.cases()["elasticity_3d"]
    H0 = SO.Hierarchy(A, O.default_params(True, strong_th=0.25, max_levels=2), num_functions=nf)
    A = A.tolil()
    i = 3 * 40 + 1
    lab = SC.interleaved(A.shape[0], nf)
    for j in A.rows[i]:
        if j != i and lab[j] == lab[i]:
            A[i, j] = A[i, j] * 1e-3
    A = A.tocsr()
    H = SO.Hierarchy(A, O.default_params(True, strong_th=0.25, max_levels=2), num_functions=nf)
    S = H.S(0)
    assert S.indptr[i + 1] == S.indptr[i]
    ref = strength_restated(_stored(H), lab, 0.25, 0.9)
    assert ref[i].size == 0
    S0 = H0.S(0)
    assert S0.indptr[i + 1] > S0.indptr[i]


@pytest.mark.parametrize("name", list(SC.cases()))
def test_interpolation_and_coarse_labels_keep_functions_apart(name):
    A, b, nf, dof, th = SC.cases()[name]
    H = SO.Hierarchy(A, O.default_params(True, strong_th=th), num_functions=nf, dof_func=dof)
    assert H.nlev >= 2
    for l in range(H.nlev - 1):
        lab, labc = H.dof(l), H.dof(l + 1)
        cf = H.cf(l)
        assert np.array_equal(labc, lab[cf == 1])             # labels of the C points, in coarse order
        assert set(np.unique(labc)) <= set(range(nf))
        P = H.P(l)
        r = np.repeat(np.arange(P.shape[0]), np.diff(P.indptr))
        assert np.all(lab[r] == labc[P.indices]), (name, l)
        if name == "vector_laplacian":
            Ac = H.A(l + 1)
            rc = np.repeat(np.arange(Ac.shape[0]), np.diff(Ac.indptr))
            assert np.all(labc[rc] == labc[Ac.indices])
    # the hierarchy is a working preconditioner
    x, info = O.pcg(A, b, M=H, rel_tol=1e-8, max_iter=200)
    assert info["converged"] and np.linalg.norm(b - A @ x) <= 1e-8 * np.linalg.norm(b) * 1.0001


def test_decoupled_systems_hierarchy_equals_scalar():
    """kron(L7, I_3): no coupling between functions, so the systems rule changes nothing."""
    A, _, nf, _, th = SC.cases()["vector_laplacian"]
    p = O.default_params(True, strong_th=th)
    Hs = O.Hierarchy(A, p)
    Hv = SO.Hierarchy(A, O.default_params(True, strong_th=th), num_functions=nf)
    assert Hs.nlev == Hv.nlev and Hs.sizes() == Hv.sizes()
    for l in range(Hs.nlev):
        a, c = Hs.A(l), Hv.A(l)
        assert np.array_equal(a.indptr, c.indptr) and np.array_equal(a.indices, c.indices) and np.array_equal(a.data, c.data)
        if l == Hs.nlev - 1:
            break
        for get in (Hs.S, Hs.P):
            a, c = get(l), getattr(Hv, get.__name__)(l)
            assert np.array_equal(a.indptr, c.indptr) and np.array_equal(a.indices, c.indices) and np.array_equal(a.data, c.data)
        assert np.array_equal(Hs.cf(l), Hv.cf(l))


def test_restatement_with_one_function_is_the_oracle_setup():
    """num_functions = 1 through the systems restatement reproduces the oracle's scalar setup."""
    A, _, _, _, _ = SC.cases()["elasticity_3d"]
    Hs = O.Hierarchy(A, O.default_params(True))
    H1 = SO.Hierarchy(A, O.default_params(True), num_functions=1)
    assert Hs.sizes() == H1.sizes()
    for l in range(Hs.nlev):
        for get in ("A", "P", "S") if l < Hs.nlev - 1 else ("A",):
            a, c = getattr(Hs, get)(l), getattr(H1, get)(l)
            assert np.array_equal(a.indptr, c.indptr) and np.array_equal(a.indices, c.indices) and np.array_equal(a.data, c.data)
        assert np.array_equal(Hs.l1(l), H1.l1(l))
    r = np.random.default_rng(0).standard_normal(A.shape[0])
    assert np.array_equal(Hs.precond(r), H1.precond(r))


# ---- host options -----------------------------------------------------------------------------
def _params(text):
    driver.initialize()
    L = driver.api()
    h = C.c_void_p()
    assert L.HYPREDRV_Create(1, C.byref(h)) == 0
    assert L.HYPREDRV_SetLibraryMode(h) == 0
    argv = (C.c_char_p * 1)(text.encode())
    code = L.HYPREDRV_InputArgsParse(1, argv, h)
    L.HYPREDRV_ErrorCodeClear()
    assert code == 0, hex(code)
    p = hdk.AmgParams()
    code = L.HYPREDRV_PreconGetDeviceParams(h, C.byref(p))
    L.HYPREDRV_ErrorCodeClear()
    L.HYPREDRV_Destroy(C.byref(h))
    return code, p


def test_presets_set_num_functions():
    for preset, nf in (("elasticity_3d", 3), ("elasticity_2d", 2), ("poisson", 1)):
        code, p = _params(f"solver: pcg\npreconditioner:\n  preset: {preset}\n")
        assert code == 0 and p.num_functions == nf and not p.dof_func
        assert p.strong_th == (0.8 if nf > 1 else 0.25)
    code, p = _params("solver: pcg\npreconditioner:\n  amg:\n    coarsening:\n      num_functions: 4\n")
    assert code == 0 and p.num_functions == 4


@pytest.mark.parametrize("key", ["nodal: 1", "filter_functions: on"])
def test_unsupported_companions_are_rejected(key):
    code, _ = _params(f"solver: pcg\npreconditioner:\n  amg:\n    coarsening:\n      num_functions: 3\n      {key}\n")
    assert code & INVALID_VAL
    code, p = _params(f"solver: pcg\npreconditioner:\n  amg:\n    coarsening:\n      num_functions: 1\n      {key}\n")
    assert code == 0 and p.num_functions == 1


def test_num_functions_below_one_is_rejected():
    for v in (0, -2):
        code, _ = _params(f"solver: pcg\npreconditioner:\n  amg:\n    coarsening:\n      num_functions: {v}\n")
        assert code & INVALID_VAL
