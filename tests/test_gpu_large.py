"""GPU parity at sizes where the production code paths are the ones that run (>= 10^6 rows):
natural sliced-ELL selection (>= 200 000 rows), the warp-per-row setup kernels, every level of a
7-8 level hierarchy.  (The setup's scratch stays below one chunk at these sizes; the fall-back
paths for long rows are reached by tests/test_gpu_unstructured.py.)  The CUDA hierarchy is
compared with an oracle run of the same problem level by level -- sizes, C/F splitting,
interpolation and Galerkin operators bit for bit (pattern, storage order and values) -- and the
Krylov solve by iteration count (north star: +-1), solution difference <= 1e-8 and true residual."""
import hashlib
import os

import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu


def _sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


LARGE = [("lap7", (128, 128, 128), (1.0, 1.0, 1.0), "pcg", 1e-6),
         ("lap27", (128, 128, 128), (1.0, 1.0, 0.01), "pcg", 1e-6),
         ("convdif", (128, 64, 64), (1e-3, 1.0, 0.1), "gmres", 1e-8),
         # not a cube, not a multiple of 32: ragged last slices / blocks on every level
         ("lap7", (150, 131, 67), (1.0, 2.0, 0.5), "pcg", 1e-6)]


@pytest.mark.parametrize("kind,dims,c,solver,tol", LARGE)
def test_large_grid_hierarchy_and_solve_match_oracle(gpu, kind, dims, c, solver, tol):
    O.set_threads(len(os.sched_getaffinity(0)))
    A, b = O.gen(kind, *dims, c=c)
    n = A.shape[0]
    assert n >= 5 * 10 ** 5
    H = O.Hierarchy(A, O.default_params(True))
    dA, db = gpu.DCsr.stencil({"lap7": 7, "lap27": 27, "convdif": 107}[kind], *dims, c=c)   # device assembly
    assert np.array_equal(db.get(), b)
    assert dA.spmv_kind()["kind"] == 2                       # sliced ELL chosen by the row count itself
    M = gpu.DAmg(dA)
    assert M.nlev == H.nlev and M.sizes() == H.sizes(), (M.sizes(), H.sizes())
    rp, cj, va = dA.diag_arrays()
    assert _sha(rp, cj, va) == _sha(A.indptr.astype(np.int32), A.indices.astype(np.int32), A.data)
    for l in range(H.nlev - 1):
        assert _sha(M.cf(l).astype(np.int32)) == _sha(H.cf(l).astype(np.int32)), f"C/F splitting level {l}"
        P = H.P(l)
        rp, cj, va = M.matrix(l, "P")
        assert _sha(rp, cj) == _sha(P.indptr.astype(np.int32), P.indices.astype(np.int32)), f"P pattern level {l}"
        assert _sha(va) == _sha(P.data), f"P values level {l}"
        del P
        Ac = H.A(l + 1)
        rp, cj, va = M.matrix(l + 1, "A")
        assert _sha(rp, cj) == _sha(Ac.indptr.astype(np.int32), Ac.indices.astype(np.int32)), f"A_c pattern level {l + 1}"
        assert _sha(va) == _sha(Ac.data), f"A_c values level {l + 1}"
        del Ac
    for l in range(H.nlev):
        assert np.array_equal(M.l1(l), H.l1(l)), f"l1 norms level {l}"
    # V-cycle and Krylov solve
    r = np.random.default_rng(3).standard_normal(n)
    dr, dz = gpu.DVec(n, r), gpu.DVec(n)
    M.apply(dr, dz)
    z_ref = H.precond(r)
    assert np.allclose(dz.get(), z_ref, rtol=1e-10, atol=1e-12 * np.abs(z_ref).max())
    dx = gpu.DVec(n)
    if solver == "pcg":
        info = gpu.pcg(dA, db, dx, M, rel_tol=tol, max_iter=100)
        xo, io = O.pcg(A, b, M=H, rel_tol=tol, max_iter=100)
    else:
        info = gpu.gmres(dA, db, dx, M, rel_tol=tol, max_iter=100)
        xo, io = O.gmres(A, b, M=H, rel_tol=tol, max_iter=100)
    assert info["converged"] and io["converged"]
    assert abs(info["iters"] - io["iters"]) <= 1, (info["iters"], io["iters"])
    x = dx.get()
    assert np.linalg.norm(x - xo) <= 1e-8 * np.linalg.norm(xo)
    assert np.linalg.norm(b - A @ x) / np.linalg.norm(b) < tol * 1.0001
