"""CPU test of the N > 1 host logic with torch.distributed (gloo, world_size 2, 127.0.0.1):
slab ranges, ParCSR diag/offd split, halo plan negotiation and a halo-exchanged SpMV, checked
against the oracle's serial SpMV.  The device implementation of the same steps is covered on
GPUs by tests/test_gpu_multi.py."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _worker(rank, world, port, kind, dims, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import partition_mirror as P
    from oracle import oracle as O
    A, _ = O.gen(kind, *dims, c=(1.0, 1.0, 0.5), diag_first=False)
    n = A.shape[0]
    x = np.random.default_rng(3).standard_normal(n)
    starts = P.row_starts(n, world)
    rs, re = P.slab_range(n, rank, world)
    assert rs == starts[rank] and re == starts[rank + 1] - 1
    ip = A.indptr[rs:re + 2].astype(np.int64)
    sl = slice(ip[0], ip[-1])
    (dp, dc, dv), (op, oc, ov), col_map = P.split_diag_offd(ip - ip[0], A.indices[sl], A.data[sl], rs, re)
    assert all(dc[dp[r]] == r for r in range(re - rs + 1) if dp[r + 1] > dp[r])      # diagonal first
    plan = P.halo_plan(col_map, starts, rank)
    # negotiate: tell every owner how many of its rows I need, then which ones
    want = torch.zeros(world, dtype=torch.int64)
    for r, (_, c) in plan.items():
        want[r] = c
    all_want = [torch.zeros(world, dtype=torch.int64) for _ in range(world)]
    dist.all_gather(all_want, want)
    reqs = []
    for r, (o, c) in plan.items():
        reqs.append(dist.isend(torch.from_numpy(col_map[o:o + c].copy()), dst=r))
    send_idx = {}
    for r in range(world):
        c = int(all_want[r][rank])
        if r != rank and c > 0:
            buf = torch.zeros(c, dtype=torch.int64)
            dist.recv(buf, src=r)
            send_idx[r] = buf.numpy() - rs
    for q in reqs:
        q.wait()
    # halo exchange of x, then y = A_diag x_loc + A_offd x_halo
    x_loc = x[rs:re + 1]
    reqs = [dist.isend(torch.from_numpy(x_loc[idx].copy()), dst=r) for r, idx in send_idx.items()]
    x_halo = np.zeros(col_map.size)
    for r, (o, c) in plan.items():
        buf = torch.zeros(c, dtype=torch.float64)
        dist.recv(buf, src=r)
        x_halo[o:o + c] = buf.numpy()
    for q in reqs:
        q.wait()
    y = np.zeros(re - rs + 1)
    for r in range(re - rs + 1):
        y[r] = dv[dp[r]:dp[r + 1]] @ x_loc[dc[dp[r]:dp[r + 1]]] + ov[op[r]:op[r + 1]] @ x_halo[oc[op[r]:op[r + 1]]]
    ys = [torch.zeros(starts[r + 1] - starts[r], dtype=torch.float64) for r in range(world)]
    dist.all_gather(ys, torch.from_numpy(y))
    # allreduce of a dot product (Krylov scalar)
    d = torch.tensor([float(x_loc @ x_loc)], dtype=torch.float64)
    dist.all_reduce(d)
    if rank == 0:
        Ad, _ = O.gen(kind, *dims, c=(1.0, 1.0, 0.5), diag_first=True)
        ref = O.matvec(Ad, x)
        got = torch.cat(ys).numpy()
        out.put((float(np.abs(got - ref).max()), float(abs(d.item() - x @ x)), len(plan)))
    dist.barrier()
    dist.destroy_process_group()


def _run(kind, dims, port):
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, kind, dims, out)) for r in range(2)]
    for p in procs:
        p.start()
    res = out.get(timeout=180)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


def test_two_rank_partition_halo_spmv_gloo():
    err, derr, nplan = _run("lap7", (6, 5, 8), 29731)
    assert err < 1e-12 and derr < 1e-10 and nplan == 1


def test_two_rank_27pt_gloo():
    err, derr, nplan = _run("lap27", (5, 4, 6), 29733)
    assert err < 1e-12 and derr < 1e-10


def test_slab_ranges_cover_everything():
    import partition_mirror as P
    for n, w in ((10, 3), (7, 7), (1000, 8), (5, 2)):
        rng = [P.slab_range(n, r, w) for r in range(w)]
        assert rng[0][0] == 0 and rng[-1][1] == n - 1
        assert all(rng[r][1] + 1 == rng[r + 1][0] for r in range(w - 1))
        assert all(e >= s for s, e in rng)


def _dump_worker(rank, world, port, n_glob, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import bench
    x = np.random.default_rng(5).standard_normal(n_glob)
    cuts = [n_glob * r // world for r in range(world + 1)]             # uneven consecutive slabs
    got = bench.gather_dump_sample(x[cuts[rank]:cuts[rank + 1]], cuts[rank], n_glob, dist)
    if rank == 0:
        out.put(bool(np.array_equal(got, x[bench.dump_positions(n_glob)])))
    dist.barrier()
    dist.destroy_process_group()


def test_bench_dump_sample_gathered_over_two_ranks_gloo():
    """bench.py --dump-outputs at N > 1: each rank contributes its slab's entries of the seeded
    sample, and rank 0 receives them in global order."""
    n_glob = 3_000_001
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    procs = [ctx.Process(target=_dump_worker, args=(r, 2, 29735, n_glob, out)) for r in range(2)]
    for p in procs:
        p.start()
    assert out.get(timeout=180) is True
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0


def test_bench_dump_positions(monkeypatch):
    """Whole solution up to DUMP_SAMPLE entries; beyond, a seeded sample: sorted, unique, in range,
    the same on every call, and at most DUMP_SAMPLE positions."""
    import bench
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    assert np.array_equal(bench.dump_positions(1000), np.arange(1000))
    idx = bench.dump_positions(50_000)
    assert 900 < idx.size <= 1000 and idx[0] >= 0 and idx[-1] < 50_000 and np.all(np.diff(idx) > 0)
    assert np.array_equal(idx, bench.dump_positions(50_000))
    x = np.arange(50_000) * 0.5
    assert np.array_equal(bench.gather_dump_sample(x, 0, 50_000), x[idx])
    assert np.array_equal(bench.gather_dump_sample(x[20_000:], 20_000, 50_000), x[idx[idx >= 20_000]])
