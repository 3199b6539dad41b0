"""CPU tests of aggressive coarsening (two-stage PMIS, multipass interpolation) in the CPU restatement
(tests/aggressive_oracle.c, built on the parity oracle) and in the host option layer.  S2 is checked
against a scipy statement of the rule; C/F and P are checked for the structure the rule implies,
independently of the restatement; with agg_num_levels = 0 the hierarchy must equal the oracle's."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.csgraph import shortest_path

import aggressive_oracle as AO
import amg_paths as AP
from hypredrive_b200 import driver, hdk
from oracle import oracle as O

INVALID_VAL = 0x200


def cases():
    return {
        "lap7": lambda: O.gen("lap7", 14, 13, 12)[0],
        "lap27_aniso": lambda: O.gen("lap27", 14, 12, 10, c=(1.0, 1.0, 0.01))[0],
        "convdif": lambda: O.gen("convdif", 24, 10, 8, c=(1e-3, 1.0, 0.1))[0],
        "heavy_tailed": lambda: AP.heavy_tailed(6000, 11),
        "signed_graph": lambda: AP.signed_graph(4000, 9),
        "fe_dirichlet": lambda: AP.fe_dirichlet(60, 50, 5),
    }


def s2_scipy(S, cf1, num_paths):
    """S2 as sparse algebra: path counts S_CC + S_CF S_FC over the C points, diagonal removed."""
    S = sp.csr_matrix((np.ones(S.nnz), S.indices, S.indptr), shape=S.shape)
    c, f = cf1 == 1, cf1 != 1
    SC = S[c]
    paths = (SC[:, c] + SC[:, f] @ S[f][:, c]).tolil()
    paths.setdiag(0)
    paths = paths.tocsr()
    paths.data = (paths.data >= num_paths).astype(float)
    paths.eliminate_zeros()
    paths.sort_indices()
    return paths


def _first_stage(A):
    """strength pattern and first-stage C/F (today's strength and PMIS) of level 0"""
    H = O.Hierarchy(A, O.default_params(True, max_levels=2))
    return H.S(0), H.cf(0, raw=True), H


@pytest.mark.parametrize("paths", [1, 2])
@pytest.mark.parametrize("name", list(cases()))
def test_s2_matches_sparse_statement(name, paths):
    A = cases()[name]()
    S, cf1, _ = _first_stage(A)
    ref = s2_scipy(S, cf1, paths)
    got = AO.s2(S, cf1, paths)
    assert np.array_equal(got.indptr, ref.indptr) and np.array_equal(got.indices, ref.indices), name
    H = AO.Hierarchy(A, O.default_params(True, max_levels=2), num_levels=1, num_paths=paths)
    S2 = H.S2(0)
    assert np.array_equal(S2.indptr, ref.indptr) and np.array_equal(S2.indices, ref.indices)
    # the hierarchy's first stage is the oracle's
    assert np.array_equal(H.S(0).indices, S.indices) and np.array_equal(H.measure(0), _first_stage(A)[2].measure(0))


@pytest.mark.parametrize("paths", [1, 2])
@pytest.mark.parametrize("name", list(cases()))
def test_cf_is_a_second_pmis_over_s2(name, paths):
    A = cases()[name]()
    _, cf1, _ = _first_stage(A)
    H = AO.Hierarchy(A, O.default_params(True, max_levels=2), num_levels=1, num_paths=paths)
    cf = H.cf(0, raw=True)
    c1 = np.flatnonzero(cf1 == 1)
    # final C points are first-stage C points; -2 exactly on first-stage C points made F; rest unchanged
    assert set(np.flatnonzero(cf == 1)) <= set(c1)
    assert np.array_equal(np.flatnonzero(cf == -2), c1[cf[c1] != 1])
    other = cf1 != 1
    assert np.array_equal(cf[other], cf1[other])
    # PMIS makes a point F only if it has a C point in its S2 row, or if no S2 row points to it
    S2 = H.S2(0)
    final_c = cf[c1] == 1
    pointed = np.zeros(len(c1), bool)
    pointed[S2.indices] = True
    for ic in np.flatnonzero(cf[c1] == -2):
        row = S2.indices[S2.indptr[ic]:S2.indptr[ic + 1]]
        assert final_c[row].any() or not pointed[ic], (name, ic)
    # after P is built -3 is reported as -1 and -2 stays
    fin = H.cf(0)
    assert not (fin == -3).any() and np.array_equal(fin == -2, cf == -2)


def _reversed_with_source(G, C):
    """edges j -> i for j in S_i, plus a virtual source n -> every C point"""
    n = G.shape[0]
    E = G.T.tocoo()
    rows = np.concatenate([E.row, np.full(len(C), n)])
    cols = np.concatenate([E.col, C])
    return sp.csr_matrix((np.ones(len(rows)), (rows, cols)), shape=(n + 1, n + 1))


def _levels(H, trunc):
    for l in range(H.nlev - 1):
        if H.passes(l) is not None:
            yield l


@pytest.mark.parametrize("trunc", [dict(), dict(max_nnz_row=4), dict(trunc_factor=0.2)], ids=["none", "mx4", "tf0.2"])
@pytest.mark.parametrize("name", list(cases()))
def test_multipass_structure(name, trunc):
    A = cases()[name]()
    H = AO.Hierarchy(A, O.default_params(True), num_levels=2, num_paths=1, **trunc)
    assert H.nlev > 1
    for l in _levels(H, trunc):
        A0, S, P, cf, ps = H.A(l), H.S(l), H.P(l), H.cf(l), H.passes(l)
        n = A0.shape[0]
        C = np.flatnonzero(cf == 1)
        f2c = np.full(n, -1)
        f2c[C] = np.arange(len(C))
        # pass numbers: 1 + breadth-first distance along S edges to a C point (0: unreachable)
        G = sp.csr_matrix((np.ones(S.nnz), S.indices, S.indptr), shape=(n, n))
        d = shortest_path(_reversed_with_source(G, C), unweighted=True, directed=True, indices=n)[:n]
        want = np.where(np.isfinite(d), d, 0).astype(int)   # distance from the virtual source = 1 + BFS distance
        assert np.array_equal(ps, want), (name, l)
        rows = [P.indices[P.indptr[i]:P.indptr[i + 1]] for i in range(n)]
        for i in range(n):
            Si = S.indices[S.indptr[i]:S.indptr[i + 1]]
            if ps[i] == 1:
                assert np.array_equal(rows[i], [f2c[i]]) and P.data[P.indptr[i]] == 1.0
            elif ps[i] == 0:
                assert len(rows[i]) == 0
            elif ps[i] == 2:
                strong_c = f2c[Si[ps[Si] == 1]]
                if not trunc:
                    assert np.array_equal(rows[i], strong_c) or len(rows[i]) == 0
                assert set(rows[i]) <= set(strong_c)
            else:
                allowed = set()
                for j in Si[ps[Si] == ps[i] - 1]:
                    allowed |= set(rows[j])
                assert set(rows[i]) <= allowed, (name, l, i)
            if "max_nnz_row" in trunc:
                assert len(rows[i]) <= trunc["max_nnz_row"]


def test_zero_row_sum_laplacian_preserves_constants():
    A = AP.rgg(5000, 3, 16, 3, shift=0.0)
    for np_ in (1, 2):
        H = AO.Hierarchy(A, O.default_params(True), num_levels=1, num_paths=np_)
        P = H.P(0)
        s = np.asarray(P.sum(axis=1)).ravel()
        live = np.diff(P.indptr) > 0
        assert live.sum() > 0.9 * A.shape[0]
        assert np.abs(s[live] - 1.0).max() < 1e-12
        assert (H.passes(0) >= 3).any()         # the product passes are reached


def test_positive_offdiagonal_rows_take_the_beta_and_lumping_branches():
    """signed_graph has positive off-diagonals: they are weak, so rows lump them (cpos == 0,
    npos != 0).  With the sign flipped (negative diagonal) the strong couplings are the positive
    ones and the rows take the beta branch."""
    seen = {}
    for sign in (1.0, -1.0):
        A = (sign * AP.signed_graph(4000, 9)).tocsr()
        H = AO.Hierarchy(A, O.default_params(True), num_levels=1)
        A0, S, P, ps = H.A(0), H.S(0), H.P(0), H.passes(0)
        lump = beta = 0
        for i in np.flatnonzero(ps >= 2):
            b, e = A0.indptr[i], A0.indptr[i + 1]
            off = A0.data[b + 1:e]
            npos = off[off > 0].sum()
            Si = S.indices[S.indptr[i]:S.indptr[i + 1]]
            J = Si[ps[Si] == ps[i] - 1]
            aJ = np.array([off[A0.indices[b + 1:e] == j][0] for j in J])
            cpos = aJ[aJ > 0].sum()
            lump += (cpos == 0 and npos != 0)
            beta += cpos != 0
        seen[sign] = (lump, beta)
    assert seen[1.0][0] > 0 and seen[-1.0][1] > 0, seen


@pytest.mark.parametrize("name", ["lap7", "convdif", "heavy_tailed", "fe_dirichlet"])
def test_no_aggressive_level_is_the_oracle(name):
    A = cases()[name]()
    prm = O.default_params(True)
    H1, Ha = O.Hierarchy(A, prm), AO.Hierarchy(A, O.default_params(True), num_levels=0)
    assert Ha.nlev == H1.nlev
    for l in range(H1.nlev):
        for get in ("A", "P", "S") if l < H1.nlev - 1 else ("A",):
            a, c = getattr(Ha, get)(l), getattr(H1, get)(l)
            assert np.array_equal(a.indptr, c.indptr) and np.array_equal(a.indices, c.indices) and np.array_equal(a.data, c.data)
        if l < H1.nlev - 1:
            assert np.array_equal(Ha.cf(l), H1.cf(l)) and Ha.S2(l) is None
        assert np.array_equal(Ha.l1(l), H1.l1(l))
    r = np.random.default_rng(0).standard_normal(A.shape[0])
    assert np.array_equal(Ha.precond(r), H1.precond(r))


def test_aggressive_lowers_operator_complexity():
    A = cases()["lap27_aniso"]()
    sizes = [sum(nnz for _, nnz in AO.Hierarchy(A, O.default_params(True), num_levels=k).sizes()) for k in (0, 1)]
    assert sizes[1] < sizes[0]


# ---- host options -----------------------------------------------------------------------------
def _params(text, capfd=None):
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
    msg = ""
    if code and capfd is not None:
        capfd.readouterr()
        L.HYPREDRV_ErrorCodeDescribe(code)
        msg = capfd.readouterr().err
    L.HYPREDRV_ErrorCodeClear()
    L.HYPREDRV_Destroy(C.byref(h))
    return code, p, msg


def _agg_yaml(body):
    lines = "".join(f"      {kv}\n" for kv in body)
    return f"solver: pcg\npreconditioner:\n  amg:\n    aggressive:\n{lines}"


def test_aggressive_keys_reach_the_device_parameters():
    code, p, _ = _params(_agg_yaml(["num_levels: 2", "num_paths: 2", "prolongation_type: multipass",
                                    "max_nnz_row: 4", "trunc_factor: 0.2"]))
    assert code == 0
    assert (p.agg_num_levels, p.agg_num_paths, p.agg_interp_type, p.agg_max_nnz_row) == (2, 2, 4, 4)
    assert p.agg_trunc_factor == 0.2
    code, p, _ = _params("solver: pcg\npreconditioner:\n  amg:\n    max_iter: 1\n")
    assert code == 0 and (p.agg_num_levels, p.agg_num_paths, p.agg_interp_type, p.agg_max_nnz_row, p.agg_trunc_factor) == (0, 1, 4, 0, 0.0)


@pytest.mark.parametrize("keys", [["num_levels: -1"], ["num_levels: 1", "num_paths: 0"], ["num_levels: 1", "max_nnz_row: -1"],
                                  ["num_levels: 1", "trunc_factor: 1.0"], ["num_levels: 1", "trunc_factor: -0.1"],
                                  ["num_levels: 1", "prolongation_type: 2_stage_extended+i"]],
                         ids=["levels", "paths", "max_nnz", "trunc_hi", "trunc_lo", "interp"])
def test_rejected_aggressive_options(keys, capfd):
    code, _, msg = _params(_agg_yaml(keys), capfd)
    assert code & INVALID_VAL and "amg:aggressive" in msg


def test_aggressive_with_systems_is_rejected(capfd):
    text = ("solver: pcg\npreconditioner:\n  amg:\n    coarsening:\n      num_functions: 3\n"
            "    aggressive:\n      num_levels: 1\n")
    code, _, msg = _params(text, capfd)
    assert code & INVALID_VAL and "num_functions" in msg


@pytest.mark.parametrize("keys", [["num_paths: 0"], ["prolongation_type: 2_stage_extended+i", "trunc_factor: 1.5"],
                                  ["max_nnz_row: -3"]], ids=["paths", "interp_trunc", "max_nnz"])
def test_aggressive_keys_without_levels_are_still_accepted(keys):
    code, p, _ = _params(_agg_yaml(["num_levels: 0"] + keys))
    assert code == 0 and p.agg_num_levels == 0
