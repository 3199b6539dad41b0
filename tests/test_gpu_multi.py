"""GPU test of the N > 1 path: spawns one process per rank with torchrun and checks parity of the
row-distributed setup (hierarchy bit-identical to the oracle's, slab by slab) and of the
distributed solve (halo exchange, allreduce, replicated tail) against the oracle.  With fewer GPUs
than ranks (the driver's 1-GPU box) the ranks share cuda:0 and talk through NCCL's socket
transport (tests/mp_gpu_check.py), so nothing here is skipped."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _digest(r):
    """The lines that say what happened (the torchrun banner and traceback are noise)."""
    keep = [l for l in (r.stdout + "\n" + r.stderr).splitlines()
            if any(k in l for k in ("MPCHECK", "hdk error", "HdkError", "HypreDriveError", "Error:", "error code", "NCCL WARN"))]
    return "\n".join(keep[-25:]) or (r.stdout[-1500:] + r.stderr[-1500:])


def _run(world, args, env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", "29611", os.path.join(ROOT, "tests", "mp_gpu_check.py")] + args
    return subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)


@pytest.mark.parametrize("kind,dims,rep,share", [
    ("lap7", ("12", "11", "6"), "40", "0"), ("lap7", ("16", "16", "10"), "262144", "0"),
    ("lap27", ("8", "8", "6"), "30", "0"), ("convdif", ("16", "8", "6"), "40", "0"),
    # replicated setup only (no work sharing between the ranks)
    ("lap7", ("12", "11", "6"), "40", "off"),
    # NCCL send/recv halo exchange instead of the peer-memory (CUDA IPC) path
    ("lap7", ("12", "11", "6"), "40", "nccl"),
    # sliced-ELL kernel on every level: off-rank block fused into the SpMV kernel, and the same layout
    # with the separate correction kernel
    ("lap7", ("16", "16", "10"), "40", "sell-fused"), ("lap27", ("8", "8", "6"), "30", "sell-fused"),
    ("convdif", ("16", "8", "6"), "40", "sell-fused"), ("lap7", ("16", "16", "10"), "40", "sell-unfused"),
    ("lap7", ("12", "11", "6"), "40", "sell-nccl"),
    # uneven row slabs that cut through grid planes (asymmetric halo sizes), all three exchange paths
    ("lap7", ("14", "9", "7"), "40", "ragged"), ("lap27", ("8", "8", "6"), "30", "ragged-sell"),
    ("convdif", ("16", "8", "6"), "40", "ragged-nccl")])
def test_two_rank_solve_matches_oracle(gpu, kind, dims, rep, share):
    env = {"HDK_REPLICATE_ROWS": rep}
    if share == "off":
        env["HDK_SETUP_REPLICATED"] = "1"        # the round-1 scheme: global hierarchy rebuilt on every rank
    elif share == "nccl":
        env["HDK_HALO_IPC"] = "0"
    elif share.startswith("ragged"):
        env["MPCHECK_RAGGED"] = "1"
        env["HDK_SHARE_MIN_ROWS"] = "0"
        if share == "ragged-sell":
            env["HDK_SELL_MIN_ROWS"] = "0"
            env["HDK_SELL_MIN_ROWS_DIST"] = "0"
        if share == "ragged-nccl":
            env["HDK_HALO_IPC"] = "0"
    elif share.startswith("sell"):
        env["HDK_SELL_MIN_ROWS"] = "0"
        env["HDK_SELL_MIN_ROWS_DIST"] = "0"
        if share == "sell-unfused":
            env["HDK_FUSE_OFFD"] = "0"
        if share == "sell-nccl":
            env["HDK_HALO_IPC"] = "0"
    else:
        env["HDK_SHARE_MIN_ROWS"] = share  # share the interpolation / RAP rows even on these tiny levels
    r = _run(2, [kind, *dims], env)
    assert r.returncode == 0, _digest(r)
    assert "ok=True" in r.stdout, _digest(r)
    if share != "off":
        assert "hier=bit-identical" in r.stdout, _digest(r)


@pytest.mark.parametrize("world,kind,dims,rep,ragged", [
    (3, "lap7", ("16", "14", "7"), "60", "1"), (4, "lap27", ("10", "9", "5"), "50", "0"),
    (4, "convdif", ("16", "10", "5"), "60", "1"), (2, "lap7", ("40", "36", "20"), "2000", "0"),
    # every level distributed down to the coarsest (replicate_rows below max_coarse_size)
    (2, "lap7", ("20", "18", "9"), "10", "1"),
    # the whole hierarchy replicated (fine level below replicate_rows)
    (2, "lap7", ("10", "9", "4"), "100000", "0")])
def test_row_distributed_setup_matches_oracle(gpu, world, kind, dims, rep, ragged):
    _row_distributed_case(world, kind, dims, rep, ragged, {})


@pytest.mark.parametrize("knob", ["HDK_RAP_SINGLE", "HDK_INTERP_SINGLE", "HDK_HALO_EXPORT", "HDK_MAILBOX", "HDK_GRAPH_ROWS",
                                  "HDK_FUSE_OFFD", "HDK_EXPORT_MAX_ROWS=100"])
def test_fallback_paths_match_oracle(gpu, knob):
    """Every default-on optimisation switched off in turn (count + fill Galerkin product and interpolation,
    pack kernels instead of folded halo exports, NCCL all-reduce instead of the mailbox, no CUDA graph,
    off-rank block in a kernel of its own, big operators packing while small ones fold): same bits."""
    name, _, value = knob.partition("=")
    extra = {name: value or "0", "HDK_SELL_MIN_ROWS": "0", "HDK_SELL_MIN_ROWS_DIST": "0"}
    if gpu.device_count() < 2:
        extra["MPCHECK_SHARED_IPC"] = "1"        # keep the peer-memory path on (two processes, one GPU)
    _row_distributed_case(2, "lap7", ("16", "16", "10"), "40", "0", extra)


def test_peer_memory_path_with_folded_exports(gpu):
    """The default multi-rank solve path (peer-memory halo, exports folded into the producers, mailbox
    reductions, all-gather of the tail's right-hand side) on sliced-ELL levels, also when the ranks
    share one GPU."""
    extra = {"HDK_SELL_MIN_ROWS": "0", "HDK_SELL_MIN_ROWS_DIST": "0", "MPCHECK_SHARED_IPC": "1"}
    _row_distributed_case(2, "lap27", ("8", "8", "6"), "30", "0", extra)
    _row_distributed_case(3, "lap7", ("16", "14", "7"), "60", "1", extra)


def _row_distributed_case(world, kind, dims, rep, ragged, extra):
    """Row-distributed setup on 2-4 ranks: per-level C/F splitting, P and A_c slabs (global columns)
    concatenate to the oracle's matrices bit for bit; solve parity as above."""
    env = {"HDK_REPLICATE_ROWS": rep, "MPCHECK_RAGGED": ragged, "MPCHECK_HIER": "1"}
    env.update(extra)
    r = _run(world, [kind, *dims], env)
    assert r.returncode == 0, _digest(r)
    assert "ok=True" in r.stdout and "hier=bit-identical" in r.stdout, _digest(r)


def _npz_system(path, name, max_levels=None):
    """One of tests/amg_paths.py's cases in hypre's storage (diagonal first, as the oracle orders
    it), with a random right-hand side, written for the ranks of mp_gpu_check.py."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import amg_paths as AP
    A = AP.CASES[name][0]().tocsr()
    for i in range(A.shape[0]):                  # ocsr_diag_first: swap the diagonal into first place
        b, e = A.indptr[i], A.indptr[i + 1]
        k = b + int(np.nonzero(A.indices[b:e] == i)[0][0])
        A.indices[[b, k]], A.data[[b, k]] = A.indices[[k, b]], A.data[[k, b]]
    extra = {} if max_levels is None else {"max_levels": np.int64(max_levels)}
    np.savez(path, indptr=A.indptr.astype(np.int64), indices=A.indices.astype(np.int64), data=A.data,
             b=AP.rhs(A.shape[0]), **extra)


@pytest.mark.parametrize("world,ragged", [(2, "0"), (3, "1")])
@pytest.mark.parametrize("mode", ["share", "sell-fused"])
def test_heavy_tailed_graph_on_several_ranks(gpu, tmp_path, world, ragged, mode):
    """The heavy-tailed graph (hubs with hundreds of scattered columns) through the CSR API on 2
    ranks and on 3 ragged slabs: the exported rows are spread over every slab, the setup's long-row
    fallbacks run on distributed levels.  Hierarchy bit-identical to the oracle's, solve parity."""
    path = str(tmp_path / "system.npz")
    _npz_system(path, "heavy_tailed")
    env = {"HDK_REPLICATE_ROWS": "2000", "MPCHECK_RAGGED": ragged, "MPCHECK_HIER": "1"}
    if mode == "share":
        env["HDK_SHARE_MIN_ROWS"] = "0"
    else:
        env.update(HDK_SELL_MIN_ROWS="0", HDK_SELL_MIN_ROWS_DIST="0")
    r = _run(world, ["npz", path], env)
    assert r.returncode == 0, _digest(r)
    assert "ok=True" in r.stdout and "hier=bit-identical" in r.stdout, _digest(r)


def test_coarse_direct_solve_above_one_cta_on_two_ranks(gpu, tmp_path):
    """max_levels 2 on a 12 000-row graph: a replicated coarsest level of more than 1024 rows, whose
    dense inverse every rank builds with the grid-wide Gauss-Jordan elimination."""
    path = str(tmp_path / "system.npz")
    _npz_system(path, "two_levels", max_levels=2)
    r = _run(2, ["npz", path], {"HDK_REPLICATE_ROWS": "2000", "MPCHECK_RAGGED": "1", "MPCHECK_HIER": "1",
                               "HDK_SHARE_MIN_ROWS": "0"})
    assert r.returncode == 0, _digest(r)
    assert "ok=True" in r.stdout and "hier=bit-identical" in r.stdout, _digest(r)
