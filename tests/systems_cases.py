"""Vector-PDE matrices for the systems AMG tests (num_functions > 1), numpy/scipy only.

* Q1 linear elasticity (E = 1, nu = 0.3, full 2x2x2 or 2x2 Gauss integration) on a box of unit
  cells; the nodes of the face x = 0 are clamped and removed, the load is a unit body force in every
  direction, the unknowns are interleaved per node (ux, uy[, uz]).  3-D, and 2-D plane strain.
  The operator is assembled in structured form: for every one of the 27 (3-D) node offsets the
  d x d block is the sum of the element-stiffness blocks of the cells the two nodes share, so the
  assembly needs O(rows x 81) memory and also serves bench_systems.py at millions of rows.
* the decoupled vector Laplacian kron(L7, I_3), interleaved;
* the elasticity matrix permuted to block (contiguous) order with matching labels;
* a ragged size: the last node keeps only part of its unknowns.
"""
from __future__ import annotations

import itertools

import numpy as np
import scipy.sparse as sp


def _elasticity_D(dim: int, E: float = 1.0, nu: float = 0.3) -> np.ndarray:
    lam, mu = E * nu / ((1 + nu) * (1 - 2 * nu)), E / (2 * (1 + nu))
    if dim == 3:
        D = np.zeros((6, 6))
        D[:3, :3] = lam
        D[np.arange(3), np.arange(3)] += 2 * mu
        D[np.arange(3, 6), np.arange(3, 6)] = mu
    else:                                               # plane strain
        D = np.array([[lam + 2 * mu, lam, 0.0], [lam, lam + 2 * mu, 0.0], [0.0, 0.0, mu]])
    return D


def element_stiffness(dim: int) -> np.ndarray:
    """Stiffness of the unit Q1 cell, unknowns ordered (corner, component); corners in the order
    of itertools.product((0, 1), repeat=dim) read as (x, y[, z])."""
    corners = np.array(list(itertools.product((0, 1), repeat=dim)), dtype=float)   # (2^d, d)
    D = _elasticity_D(dim)
    g = np.array([0.5 - 0.5 / np.sqrt(3.0), 0.5 + 0.5 / np.sqrt(3.0)])
    nd = corners.shape[0] * dim
    K = np.zeros((nd, nd))
    for q in itertools.product(g, repeat=dim):
        q = np.array(q)
        # dN_a/dx_k for N_a = prod_j (c_aj x_j + (1 - c_aj)(1 - x_j))
        f = np.where(corners > 0, q, 1.0 - q)                        # (2^d, d)
        s = np.where(corners > 0, 1.0, -1.0)
        dN = np.empty_like(f)
        for k in range(dim):
            dN[:, k] = s[:, k] * np.prod(np.delete(f, k, axis=1), axis=1)
        nv = 6 if dim == 3 else 3
        B = np.zeros((nv, nd))
        for a in range(corners.shape[0]):
            for k in range(dim):
                B[k, a * dim + k] = dN[a, k]
            if dim == 3:
                B[3, a * 3 + 0], B[3, a * 3 + 1] = dN[a, 1], dN[a, 0]
                B[4, a * 3 + 1], B[4, a * 3 + 2] = dN[a, 2], dN[a, 1]
                B[5, a * 3 + 0], B[5, a * 3 + 2] = dN[a, 2], dN[a, 0]
            else:
                B[2, a * 2 + 0], B[2, a * 2 + 1] = dN[a, 1], dN[a, 0]
        K += B.T @ D @ B / 2 ** dim                                    # Gauss weights (1/2)^d
    return K


def elasticity(m: int, dim: int = 3):
    """Clamped Q1 elasticity with m^dim free nodes (m cells in x, m - 1 in the other directions,
    the m + 1-st node plane x = 0 clamped).  Returns (A scipy CSR with sorted columns, b)."""
    Ke = element_stiffness(dim)
    corners = list(itertools.product((0, 1), repeat=dim))
    ncell = [m] + [m - 1] * (dim - 1)                 # cells per direction
    shape = [m] * dim                                  # free nodes per direction (x index 1..m)
    nn = m ** dim
    idx = np.indices(shape[::-1]).reshape(dim, -1)[::-1]   # (x, y[, z]) of every free node, x fastest
    pos = idx.copy()
    pos[0] += 1                                        # grid coordinate including the clamped plane
    offsets = list(itertools.product((-1, 0, 1), repeat=dim))
    offsets = [o[::-1] for o in offsets]               # (ox, oy[, oz]) with oz slowest: increasing neighbour index
    blocks = np.zeros((nn, len(offsets), dim, dim))
    conn = np.zeros((nn, len(offsets)), dtype=bool)
    ncells_at = np.zeros(nn)
    for a_i, a in enumerate(corners):
        # cell whose corner a is this node: cell coordinate pos - a must exist
        ok = np.ones(nn, dtype=bool)
        for k in range(dim):
            c = pos[k] - a[k]
            ok &= (c >= 0) & (c < ncell[k])
        ncells_at += ok
        for o_i, o in enumerate(offsets):
            b = tuple(a[k] + o[k] for k in range(dim))
            if any(v not in (0, 1) for v in b):
                continue
            b_i = corners.index(b)
            valid = ok & (pos[0] + o[0] >= 1)           # the neighbour is not clamped
            blocks[valid, o_i] += Ke[a_i * dim:(a_i + 1) * dim, b_i * dim:(b_i + 1) * dim]
            conn[valid, o_i] = True
    stride = np.cumprod([1] + shape[:-1])
    nbr = np.zeros((nn, len(offsets)), dtype=np.int64)
    for o_i, o in enumerate(offsets):
        nbr[:, o_i] = sum((idx[k] + o[k]) * stride[k] for k in range(dim))
    # rows d*node + c: columns d*nbr + c' over the connected offsets, in increasing order
    cols = (dim * nbr[:, :, None, None] + np.arange(dim)[None, None, None, :]).repeat(dim, axis=2)
    vals = blocks                                          # (nn, off, c, c')
    mask = np.broadcast_to(conn[:, :, None, None], vals.shape)
    cols = np.transpose(cols, (0, 2, 1, 3))                # (nn, c, off, c')
    vals = np.transpose(vals, (0, 2, 1, 3))
    mask = np.transpose(mask, (0, 2, 1, 3))
    n = dim * nn
    cols, vals, mask = cols.reshape(n, -1), vals.reshape(n, -1), mask.reshape(n, -1)
    indptr = np.concatenate([[0], np.cumsum(mask.sum(axis=1))]).astype(np.int64)
    A = sp.csr_matrix((vals[mask], cols[mask].astype(np.int32), indptr), shape=(n, n))
    b = np.repeat(ncells_at / 2 ** dim, dim)               # unit body force in every direction
    return A, b


def lap7(nx: int, ny: int, nz: int) -> sp.csr_matrix:
    def l1(k):
        return sp.diags([-np.ones(k - 1), 2 * np.ones(k), -np.ones(k - 1)], [-1, 0, 1])
    I = sp.identity
    return (sp.kron(I(nz), sp.kron(I(ny), l1(nx))) + sp.kron(I(nz), sp.kron(l1(ny), I(nx)))
            + sp.kron(l1(nz), sp.kron(I(ny), I(nx)))).tocsr()


def vector_laplacian(nx: int, ny: int, nz: int, nf: int = 3):
    """kron(L7, I_nf): nf decoupled Laplacians, unknowns interleaved per node."""
    A = sp.kron(lap7(nx, ny, nz), sp.identity(nf)).tocsr()
    A.sort_indices()
    return A, np.ones(A.shape[0])


def interleaved(n: int, nf: int) -> np.ndarray:
    return (np.arange(n) % nf).astype(np.int32)


def block_order(A: sp.csr_matrix, b: np.ndarray, nf: int):
    """The interleaved system permuted to block order (all u_0, then all u_1, ...) and its labels."""
    n = A.shape[0]
    perm = np.concatenate([np.arange(f, n, nf) for f in range(nf)])
    Ab = A[perm][:, perm].tocsr()
    Ab.sort_indices()
    return Ab, b[perm], interleaved(n, nf)[perm]


def ragged(A: sp.csr_matrix, b: np.ndarray, drop: int = 1):
    """The last `drop` unknowns removed: the last node keeps only part of its components."""
    n = A.shape[0] - drop
    return A[:n][:, :n].tocsr(), b[:n].copy()


def cases():
    """name -> (A, b, num_functions, dof_func or None, strong_th)."""
    A3, b3 = elasticity(6, 3)
    A2, b2 = elasticity(12, 2)
    Av, bv = vector_laplacian(7, 6, 5)
    Ab, bb, db = block_order(A3, b3, 3)
    Ar, br = ragged(A3, b3, 1)
    return {
        "elasticity_3d": (A3, b3, 3, None, 0.8),
        "elasticity_3d_th025": (A3, b3, 3, None, 0.25),
        "plane_strain": (A2, b2, 2, None, 0.8),
        "vector_laplacian": (Av, bv, 3, None, 0.25),
        "block_labels": (Ab, bb, 3, db, 0.8),
        "ragged": (Ar, br, 3, None, 0.8),
    }
