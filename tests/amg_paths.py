"""Unstructured test matrices and the code-path census of the device AMG setup.

The matrices are what finite-element and graph callers pass and no stencil produces: Dirichlet
identity rows, strongly diagonally dominant rows, positive off-diagonal entries, rows coupled to
hundreds of others, scattered columns.  Every generator is numpy/scipy with a fixed seed.

`census()` computes, from an oracle hierarchy, the quantities each kernel-selection decision of
the device setup depends on, and `paths()` names the code paths a hierarchy reaches.  The
thresholds below mirror the library's constants; each cites where it is defined.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp
from scipy.spatial import cKDTree

# ---- thresholds of hypredrive_b200/csrc/hdk_amg_setup.cu ---------------------------------------
INTERP_THREAD_AVG = 10.0   # HDK_INTERP_THREAD_AVG default: one thread per row when nnz/n <= this (build_interp)
IS_CAP = 48                # k_interp_small: |C-hat| held in thread-local arrays
IS_F = 24                  # k_interp_small: strong F neighbours held in thread-local arrays
IW_LIST = 120              # k_interp_warp: longest C-hat
IW_INS = 192               # k_interp_warp: inserts (C-hat plus strong F neighbours), 3/4 of IW_CAP = 256
RAP_256 = 160              # k_rap_warp<.., 256, true>: rows of A_c up to 5/8 of 256 slots
RW_LIMIT = 320             # k_rap_warp: longest row of A_c; longer rows go to k_rap_count / k_rap_fill
RAP_BANDS = (80, 160, 320)  # count + fill product (HDK_RAP_SINGLE=0): 128-, 256-, 512-slot tables
GE_ONE_CTA = 1024          # GJ_ONE_CTA: dense coarse inverse in one CTA up to this many rows
GE_MAX_N2 = 2.0e8          # dense coarse inverse while n^2 < 2e8 (also oracle/amg_setup.c)
# ---- hypredrive_b200/csrc/hdk_spmv.cu (csr_analyze) ---------------------------------------------
S_MAXR = 1024              # longest row of the stream kernel; longer rows select k_spmv_vector


def lanes_per_row(avg):
    """csr_analyze: lanes per row of the stream kernel from the average row length."""
    return 1 if avg <= 12.0 else (2 if avg <= 24.0 else (4 if avg <= 56.0 else 8))


# ---- matrix families ---------------------------------------------------------------------------
def _sym_from_edges(n, i, j, w, shift):
    """Graph Laplacian-like SPD matrix: off-diagonal -w (or +w for negative w), diagonal sum|w| + shift."""
    W = sp.coo_matrix((np.concatenate([w, w]), (np.concatenate([i, j]), np.concatenate([j, i]))), shape=(n, n)).tocsr()
    W.sum_duplicates()
    d = np.asarray(abs(W).sum(axis=1)).ravel() + shift
    return (sp.diags(d) - W).tocsr()


def rgg(n, dim, degree, seed, shift=1e-2):
    """Random geometric graph Laplacian in the unit square / cube, mean degree about `degree`."""
    rng = np.random.default_rng(seed)
    pts = rng.random((n, dim))
    vol = np.pi if dim == 2 else 4.0 * np.pi / 3.0
    r = (degree / (n * vol)) ** (1.0 / dim)
    pairs = cKDTree(pts).query_pairs(r, output_type="ndarray")
    w = 1.0 / (1e-3 + np.linalg.norm(pts[pairs[:, 0]] - pts[pairs[:, 1]], axis=1) / r)
    return _sym_from_edges(n, pairs[:, 0], pairs[:, 1], w, shift)


def heavy_tailed(n, seed):
    """2-D geometric graph plus hubs with a heavy-tailed degree distribution.  'Strong' hubs
    (couplings as strong as the base graph) become C points whose rows of A_c reach hundreds of
    entries; 'weak' hubs (couplings weak from the neighbours' side, strong from the hub's) become
    F points with a C-hat of hundreds of points."""
    rng = np.random.default_rng(seed)
    A = rgg(n, 2, 7, seed).tocoo()
    mask = A.row < A.col
    i, j, w = list(A.row[mask]), list(A.col[mask]), list(-A.data[mask])
    hubs = rng.choice(n, size=48, replace=False)
    degs = np.concatenate([np.full(8, 30), np.full(8, 60), np.full(8, 120), np.full(6, 250), np.full(4, 500),
                           np.full(2, 1100), np.full(12, 400)])
    weights = np.concatenate([np.full(36, 1.0), np.full(12, 0.05)])
    for h, dg, hw in zip(hubs, degs, weights):
        nb = rng.choice(n, size=int(dg), replace=False)
        nb = nb[nb != h]
        i += [int(h)] * nb.size
        j += list(nb)
        w += [hw] * nb.size
    i, j, w = np.array(i), np.array(j), np.array(w, dtype=np.float64)
    lo, hi = np.minimum(i, j), np.maximum(i, j)
    key = lo * n + hi
    _, first = np.unique(key, return_index=True)
    return _sym_from_edges(n, lo[first], hi[first], w[first], 1e-2)


def _p1_stiffness(nx, ny, seed, K=((1.0, 0.0), (0.0, 1.0)), jitter=0.3):
    """P1 stiffness matrix of a jittered, triangulated nx x ny grid on the unit square with the
    diffusion tensor K; returns (A, boundary mask)."""
    rng = np.random.default_rng(seed)
    hx, hy = 1.0 / (nx - 1), 1.0 / (ny - 1)
    X, Y = np.meshgrid(np.linspace(0, 1, nx), np.linspace(0, 1, ny), indexing="ij")
    bnd = (X == 0) | (X == 1) | (Y == 0) | (Y == 1)
    X = X + np.where(bnd, 0.0, jitter * hx * (rng.random(X.shape) - 0.5))
    Y = Y + np.where(bnd, 0.0, jitter * hy * (rng.random(Y.shape) - 0.5))
    pts = np.stack([X.ravel(), Y.ravel()], axis=1)
    idx = np.arange(nx * ny).reshape(nx, ny)
    a, b, c, d = idx[:-1, :-1].ravel(), idx[1:, :-1].ravel(), idx[:-1, 1:].ravel(), idx[1:, 1:].ravel()
    flip = rng.random(a.size) < 0.5   # random diagonal of every quad: an unstructured triangulation
    t1 = np.where(flip[:, None], np.stack([a, b, d], 1), np.stack([a, b, c], 1))
    t2 = np.where(flip[:, None], np.stack([a, d, c], 1), np.stack([b, d, c], 1))
    tri = np.concatenate([t1, t2])
    p = pts[tri]                                            # (T, 3, 2)
    e1, e2 = p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]
    det = e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0]
    ginv = np.stack([np.stack([e2[:, 1], -e1[:, 1]], 1), np.stack([-e2[:, 0], e1[:, 0]], 1)], 1) / det[:, None, None]
    G = np.einsum("tij,kj->tki", ginv, np.array([[-1.0, -1.0], [1.0, 0.0], [0.0, 1.0]]))   # gradients (T, 3, 2)
    Ke = 0.5 * np.abs(det)[:, None, None] * np.einsum("tai,ij,tbj->tab", G, np.asarray(K), G)
    rows = np.repeat(tri, 3, axis=1).ravel()
    cols = np.tile(tri, (1, 3)).ravel()
    A = sp.coo_matrix((Ke.ravel(), (rows, cols)), shape=(nx * ny,) * 2).tocsr()
    A.sum_duplicates()
    return A, bnd.ravel()


def _dirichlet(A, bnd):
    """Identity rows (and zero columns, so the matrix stays symmetric) at the boundary nodes."""
    keep = sp.diags((~bnd).astype(np.float64))
    A = (keep @ A @ keep + sp.diags(bnd.astype(np.float64))).tocsr()
    A.eliminate_zeros()
    return A


def fe_dirichlet(nx, ny, seed):
    A, bnd = _p1_stiffness(nx, ny, seed)
    return _dirichlet(A, bnd)


def fe_rotated_aniso(nx, ny, seed, eps=1e-3, theta=np.pi / 6):
    """Rotated anisotropic diffusion on a triangulated grid: positive off-diagonal entries."""
    R = np.array([[np.cos(theta), -np.sin(theta)], [np.sin(theta), np.cos(theta)]])
    A, bnd = _p1_stiffness(nx, ny, seed, K=R @ np.diag([1.0, eps]) @ R.T)
    return _dirichlet(A, bnd)


def signed_graph(n, seed, frac=0.25):
    """3-D geometric graph with a share of positive off-diagonal couplings, diagonally dominant."""
    A = rgg(n, 3, 14, seed).tocoo()
    rng = np.random.default_rng(seed + 1)
    mask = A.row < A.col
    w = -A.data[mask]
    w = np.where(rng.random(w.size) < frac, -w, w)
    return _sym_from_edges(n, A.row[mask], A.col[mask], w, 1e-2)


def arrow(n, seed):
    """2-D geometric graph bordered by one dense row and column (the last one): the level-0 SpMV
    has a row of n entries (k_spmv_vector)."""
    A = rgg(n - 1, 2, 8, seed)
    rng = np.random.default_rng(seed)
    border = -0.01 * (0.5 + rng.random(n - 1))
    B = sp.bmat([[A, sp.csr_matrix(border[:, None])], [sp.csr_matrix(border[None, :]), None]]).tocsr()
    B = (B + sp.diags(np.concatenate([np.abs(border), [np.abs(border).sum() + 1.0]]))).tocsr()
    return B


def diag_dominant(n, seed):
    """Every row fails the max_row_sum test (|row sum| > 0.9 |a_ii|): S is empty, one level."""
    A = rgg(n, 3, 12, seed).tocoo()
    mask = A.row != A.col
    off = sp.coo_matrix((A.data[mask], (A.row[mask], A.col[mask])), shape=A.shape).tocsr()
    d = 20.0 * np.asarray(abs(off).sum(axis=1)).ravel() + 1.0
    return (off + sp.diags(d)).tocsr()


def block_diagonal(seed):
    """Disconnected components of different kinds and sizes, and isolated 1x1 blocks."""
    rng = np.random.default_rng(seed)
    blocks = [rgg(1500, 2, 8, seed), fe_dirichlet(30, 40, seed + 1), rgg(900, 3, 14, seed + 2),
              sp.csr_matrix(np.array([[2.0]])), rgg(40, 2, 6, seed + 3), sp.csr_matrix(np.array([[5.0]]))]
    A = sp.block_diag(blocks, format="csr")
    p = rng.permutation(A.shape[0])        # components interleaved in the row order
    return A[p][:, p].tocsr()


def scrambled(A, seed, zeros_per_row=2):
    """The same matrix stored with unsorted rows, the diagonal not first and explicit zeros."""
    rng = np.random.default_rng(seed)
    A = A.tocsr()
    n = A.shape[0]
    rows, cols, vals = [], [], []
    for i in range(n):
        c = A.indices[A.indptr[i]:A.indptr[i + 1]]
        v = A.data[A.indptr[i]:A.indptr[i + 1]]
        extra = np.setdiff1d(rng.choice(n, size=zeros_per_row, replace=False), c)
        c = np.concatenate([c, extra])
        v = np.concatenate([v, np.zeros(extra.size)])
        o = rng.permutation(c.size)
        rows.append(np.full(c.size, i)); cols.append(c[o]); vals.append(v[o])
    indptr = np.concatenate([[0], np.cumsum([r.size for r in rows])]).astype(np.int64)
    B = sp.csr_matrix((n, n))
    B.indptr, B.indices, B.data = indptr, np.concatenate(cols).astype(np.int64), np.concatenate(vals)
    B._shape = (n, n)
    return B


def rhs(n, seed=7):
    return np.random.default_rng(seed).standard_normal(n)


# (name, matrix builder, AMG parameters, solver, paths the case reaches with the default selection)
CASES = {
    "heavy_tailed": (lambda: heavy_tailed(20000, 11), {}, "pcg",
                     {"interp.staged", "interp.thread", "interp.thread_overflow", "interp.warp", "interp.warp_overflow",
                      "rap.single256", "rap.single512", "rap.global", "spmv.vector"}),
    "heavy_tailed_no_trunc": (lambda: heavy_tailed(20000, 11), dict(max_nnz_row=0), "pcg",
                              {"interp.count_fill", "interp.warp_overflow", "interp.warp_insert_overflow",
                               "rap.global", "spmv.lpr8"}),
    "rgg3d": (lambda: rgg(12000, 3, 16, 3), {}, "pcg", {"interp.warp", "spmv.lpr2"}),
    "fe_dirichlet": (lambda: fe_dirichlet(120, 110, 5), {}, "pcg", {"interp.thread", "sf_rows", "spmv.lpr1"}),
    "fe_rotated_aniso": (lambda: fe_rotated_aniso(110, 100, 6), dict(trunc_factor=0.2), "pcg",
                         {"positive_offdiag", "interp.count_fill", "sf_rows"}),
    "signed_graph": (lambda: signed_graph(8000, 9), {}, "gmres", {"positive_offdiag", "interp.warp"}),
    "arrow": (lambda: arrow(3000, 13), {}, "pcg", {"spmv.vector"}),
    "scrambled_fe": (lambda: scrambled(fe_dirichlet(60, 50, 8), 8), {}, "pcg", {"sf_rows"}),
    "diag_dominant": (lambda: diag_dominant(2000, 4), {}, "pcg", {"one_level", "coarse.dense_grid"}),
    "two_levels": (lambda: rgg(12000, 3, 24, 21), dict(max_levels=2), "pcg", {"coarse.dense_grid", "spmv.lpr4"}),
    "block_diagonal": (lambda: block_diagonal(17), {}, "pcg", {"sf_rows", "coarse.dense_cta"}),
    # the hierarchy of rgg3d has levels of 12000, 1621, 248 and 36 rows: max_coarse_size at and just
    # below the third level's size stops the coarsening there or one level further
    "coarse_size_at": (lambda: rgg(12000, 3, 16, 3), dict(max_coarse_size=248), "pcg", {"coarse.dense_cta"}),
    "coarse_size_below": (lambda: rgg(12000, 3, 16, 3), dict(max_coarse_size=247), "pcg", {"coarse.dense_cta"}),
}

# Path switches read once per process (child processes of test_forced_setup_paths_match_oracle):
# name -> (environment, paths reached by FORCED_CASES over FORCED_SETTINGS)
FORCED = {
    "thread": ({"HDK_INTERP_THREAD_AVG": "1e9"}, {"interp.thread", "interp.thread_overflow"}),
    "warp": ({"HDK_INTERP_THREAD_AVG": "0"}, {"interp.warp", "interp.warp_overflow", "interp.warp_insert_overflow"}),
    "interp_count_fill": ({"HDK_INTERP_SINGLE": "0"}, {"interp.count_fill", "interp.warp_overflow"}),
    "rap_count_fill": ({"HDK_RAP_SINGLE": "0"}, {"rap.band80", "rap.band160", "rap.band320", "rap.global"}),
}
FORCED_CASES = ("heavy_tailed", "arrow")
FORCED_SETTINGS = (dict(max_nnz_row=4), dict(max_nnz_row=0), dict(trunc_factor=0.2))


def knobs(env):
    """The path switches of an environment (the library's defaults where unset)."""
    return dict(thread_avg=float(env.get("HDK_INTERP_THREAD_AVG", INTERP_THREAD_AVG)),
                interp_single=env.get("HDK_INTERP_SINGLE", "1").strip() != "0",
                rap_single=env.get("HDK_RAP_SINGLE", "1").strip() != "0")


# counts() of every case (oracle hierarchy of the input as generated): which rows pass which limit
COUNTS = {
    'heavy_tailed': {'rows': [20000, 4111, 1174, 64], 'chat': 652, 'nf': 321, 'inserts': 973, 'ac_len': 3587, 'over_is': 406, 'over_iw': 228, 'ac_over_320': 101},
    'heavy_tailed_no_trunc': {'rows': [20000, 4111, 1231, 135, 2], 'chat': 652, 'nf': 321, 'inserts': 973, 'ac_len': 3809, 'over_is': 421, 'over_iw': 231, 'ac_over_320': 2580},
    'rgg3d': {'rows': [12000, 1621, 248, 36], 'chat': 17, 'nf': 29, 'inserts': 40, 'ac_len': 101, 'over_is': 10, 'over_iw': 0, 'ac_over_320': 0},
    'fe_dirichlet': {'rows': [13200, 4621, 962, 179, 30], 'chat': 8, 'nf': 10, 'inserts': 17, 'ac_len': 36, 'over_is': 0, 'over_iw': 0, 'ac_over_320': 0},
    'fe_rotated_aniso': {'rows': [11000, 3361, 986, 225, 47], 'chat': 9, 'nf': 8, 'inserts': 16, 'ac_len': 33, 'over_is': 0, 'over_iw': 0, 'ac_over_320': 0},
    'signed_graph': {'rows': [8000, 1401, 50], 'chat': 17, 'nf': 18, 'inserts': 30, 'ac_len': 64, 'over_is': 0, 'over_iw': 0, 'ac_over_320': 0},
    'arrow': {'rows': [3000, 611, 178, 55], 'chat': 611, 'nf': 2388, 'inserts': 2999, 'ac_len': 611, 'over_is': 1, 'over_iw': 1, 'ac_over_320': 4},
    'scrambled_fe': {'rows': [3000, 1023, 218, 45], 'chat': 8, 'nf': 8, 'inserts': 14, 'ac_len': 216, 'over_is': 0, 'over_iw': 0, 'ac_over_320': 0},
    'diag_dominant': {'rows': [2000], 'chat': 0, 'nf': 0, 'inserts': 0, 'ac_len': 0, 'over_is': 0, 'over_iw': 0, 'ac_over_320': 0},
    'two_levels': {'rows': [12000, 1353], 'chat': 21, 'nf': 42, 'inserts': 60, 'ac_len': 72, 'over_is': 1238, 'over_iw': 0, 'ac_over_320': 0},
    'block_diagonal': {'rows': [3642, 849, 197, 47], 'chat': 14, 'nf': 20, 'inserts': 31, 'ac_len': 50, 'over_is': 0, 'over_iw': 0, 'ac_over_320': 0},
    'coarse_size_at': {'rows': [12000, 1621, 248], 'chat': 17, 'nf': 29, 'inserts': 40, 'ac_len': 101, 'over_is': 10, 'over_iw': 0, 'ac_over_320': 0},
    'coarse_size_below': {'rows': [12000, 1621, 248, 36], 'chat': 17, 'nf': 29, 'inserts': 40, 'ac_len': 101, 'over_is': 10, 'over_iw': 0, 'ac_over_320': 0},
}


# ---- census ------------------------------------------------------------------------------------
def row_census(S, cf):
    """Per row of a level: |C-hat_i| (extended+i), the number of strong F neighbours and the table
    inserts (their sum), for F rows; 0 for C and SF rows.  cf is the oracle's raw splitting
    (1 C, -1 F, -3 SF)."""
    S = sp.csr_matrix((np.ones(S.nnz), S.indices, S.indptr), shape=S.shape)
    isC = (cf > 0).astype(np.float64)
    isF = (cf == -1).astype(np.float64)
    SC = (S @ sp.diags(isC)).tocsr()
    SF = (S @ sp.diags(isF)).tocsr()
    SC.eliminate_zeros()
    SF.eliminate_zeros()
    chat_m = (SC + SF @ SC).tocsr()
    chat_m.eliminate_zeros()
    frow = cf == -1
    chat = np.where(frow, np.diff(chat_m.indptr), 0)
    nf = np.where(frow, np.diff(SF.indptr), 0)
    return chat, nf, chat + nf


def census(H):
    """Per level of an oracle hierarchy: the quantities the device setup's path choices depend on."""
    out = []
    for l in range(H.nlev):
        A = H.A(l)
        n = A.shape[0]
        lens = np.diff(A.indptr)
        e = dict(level=l, rows=n, avg_row=A.nnz / max(n, 1), max_row=int(lens.max()) if n else 0)
        if l < H.nlev - 1:
            chat, nf, ins = row_census(H.S(l), H.cf(l, raw=True))
            Ac = H.A(l + 1)
            e.update(chat=chat, nf=nf, inserts=ins, ac_len=np.diff(Ac.indptr), sf_rows=int((H.cf(l, raw=True) == -3).sum()))
        out.append(e)
    return out


def counts(H):
    """The census in a few numbers: level sizes, largest |C-hat|, strong F neighbours, table
    inserts and A_c row, and the number of rows past each interpolation limit."""
    cen = census(H)
    fine = [e for e in cen if "chat" in e]
    mx = lambda k: max((int(e[k].max()) for e in fine), default=0)
    tot = lambda m: sum(int(np.sum(m(e))) for e in fine)
    return dict(rows=[e["rows"] for e in cen], chat=mx("chat"), nf=mx("nf"), inserts=mx("inserts"), ac_len=mx("ac_len"),
                over_is=tot(lambda e: (e["chat"] > IS_CAP) | (e["nf"] > IS_F)),
                over_iw=tot(lambda e: (e["chat"] > IW_LIST) | (e["inserts"] > IW_INS)),
                ac_over_320=tot(lambda e: e["ac_len"] > RW_LIMIT))


def paths(H, params, A0=None, knob=None):
    """Names of the code paths a hierarchy with these AMG parameters reaches on the device under
    the path switches `knob` (knobs(env); the defaults when None), following build_interp,
    build_rap, build_dense_inverse and csr_analyze."""
    k = knob or knobs({})
    got = set()
    cen = census(H)
    staged = k["interp_single"] and params.get("max_nnz_row", 4) > 0 and params.get("trunc_factor", 0.0) == 0.0
    if len(cen) == 1:
        got.add("one_level")
    for e in cen:
        got.add("spmv.vector" if e["max_row"] > S_MAXR else f"spmv.lpr{lanes_per_row(e['avg_row'])}")
        if "chat" not in e:
            continue
        got.add("interp.staged" if staged else "interp.count_fill")
        if e["sf_rows"]:
            got.add("sf_rows")
        if e["avg_row"] <= k["thread_avg"]:
            # one thread per row only in the single pass; otherwise every row of the level is flagged
            # for k_interp_count / k_interp_fill
            if staged:
                got.add("interp.thread")
                if np.any((e["chat"] > IS_CAP) | (e["nf"] > IS_F)):
                    got.add("interp.thread_overflow")
        else:
            got.add("interp.warp")
            over = (e["chat"] > IW_LIST) | (e["inserts"] > IW_INS)
            if np.any(over):
                got.add("interp.warp_overflow")
            if np.any((e["chat"] <= IW_LIST) & (e["inserts"] > IW_INS)):
                got.add("interp.warp_insert_overflow")   # flagged by the insert bound alone
        L = e["ac_len"]
        if k["rap_single"]:
            if np.any(L <= RAP_256):
                got.add("rap.single256")
            if np.any((L > RAP_256) & (L <= RW_LIMIT)):
                got.add("rap.single512")
        else:
            for j, b in enumerate(RAP_BANDS):
                if np.any((L > (RAP_BANDS[j - 1] if j else 0)) & (L <= b)):
                    got.add(f"rap.band{b}")
        if np.any(L > RW_LIMIT):
            got.add("rap.global")
    nc = cen[-1]["rows"]
    if params.get("relax_coarse", 9) in (9, 99) and nc * nc < GE_MAX_N2:
        got.add("coarse.dense_cta" if nc <= GE_ONE_CTA else "coarse.dense_grid")
    if A0 is not None and np.any(sp.triu(A0, 1).data > 0):
        got.add("positive_offdiag")
    return got


# every decision of the device setup and SpMV that a test must reach
REQUIRED = {"interp.thread", "interp.thread_overflow", "interp.warp", "interp.warp_overflow",
            "interp.warp_insert_overflow", "interp.staged", "interp.count_fill", "rap.single256", "rap.single512",
            "rap.global", "rap.band80", "rap.band160", "rap.band320", "spmv.vector", "spmv.lpr1", "spmv.lpr2",
            "spmv.lpr4", "spmv.lpr8", "coarse.dense_cta", "coarse.dense_grid", "sf_rows", "positive_offdiag",
            "one_level"}
