"""Two-rank check of aggressive coarsening (launched by torchrun; see test_gpu_aggressive.py).  Every
rank passes its slab of rows of the 7-point Laplacian through the HYPREDRV CSR API with
`aggressive: num_levels: 1`; the ranks rebuild the global hierarchy (the replicated setup that N > 1
uses for aggressive coarsening) and solve together.  With every level replicated
(HDK_REPLICATE_ROWS large) rank 0 compares A_l, S_l, S2_l, C/F and P_l of every level with the CPU
restatement run on the global problem -- the hierarchy the one-rank device setup builds -- bit for
bit, and checks equal iterations, a solution difference <= 1e-8 and the true residual.
MPCHECK_RAGGED=1 cuts the rows unevenly.  With fewer GPUs than ranks the ranks share cuda:0 as in
mp_gpu_check.py."""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)


def _level(hM, l, which, nrows, nnz):
    from hypredrive_b200 import hdk
    rp, cj, va = np.empty(nrows + 1, np.int32), np.empty(max(nnz, 1), np.int32), np.zeros(max(nnz, 1))
    hdk.check(hdk.lib().hdk_amg_get_matrix(hM, l, which, rp.ctypes.data, cj.ctypes.data, va.ctypes.data))
    k = int(rp[nrows])
    return rp, cj[:k], va[:k]


def main():
    import torch
    import torch.distributed as dist
    from hypredrive_b200 import hdk, driver
    from oracle import oracle as O

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    if torch.cuda.device_count() < world:
        local = local % max(torch.cuda.device_count(), 1)
        os.environ["NCCL_HOSTID"] = f"hdk-one-gpu-rank{rank}"
        os.environ.setdefault("NCCL_SOCKET_IFNAME", "lo")
        os.environ["NCCL_IB_DISABLE"] = "1"
        os.environ["HDK_HALO_IPC"] = "0"
    torch.cuda.set_device(local)
    dist.init_process_group(backend="gloo")
    hdk.init(local)
    uid = torch.zeros(128, dtype=torch.uint8)
    if rank == 0:
        buf = (C.c_ubyte * 128)()
        hdk.check(hdk.lib().hdk_comm_unique_id(buf))
        uid = torch.tensor(list(buf), dtype=torch.uint8)
    dist.broadcast(uid, 0)
    hdk.check(hdk.lib().hdk_comm_init(rank, world, bytes(uid.tolist())))
    hdk.tune("amg_keep_debug", 1)

    m = int(sys.argv[1]) if len(sys.argv) > 1 else 12
    A, b = O.gen("lap7", m, m, m)
    n = A.shape[0]
    if os.environ.get("MPCHECK_RAGGED") == "1":
        cuts = np.array([0, n // 3 + 7, n])
    else:
        cuts = np.arange(world + 1, dtype=np.int64) * n // world
    rs, re = int(cuts[rank]), int(cuts[rank + 1]) - 1
    tol = 1e-8
    opts = {"general": {"statistics": False}, "solver": {"pcg": {"relative_tol": tol, "max_iter": 200}},
            "preconditioner": {"amg": {"aggressive": {"num_levels": 1}}}}
    L = driver.api()
    mine = {}
    with driver.HypreDrive(options=opts) as drv:
        lo, hi = int(A.indptr[rs]), int(A.indptr[re + 1])
        drv.set_matrix_from_csr(A.indptr[rs:re + 2] - lo, A.indices[lo:hi], A.data[lo:hi], row_start=rs, row_end=re)
        drv.set_rhs(b[rs:re + 1])
        driver._check(L.HYPREDRV_LinearSystemSetInitialGuess(drv._h, None), "SetInitialGuess")
        driver._check(L.HYPREDRV_LinearSystemResetInitialGuess(drv._h), "ResetInitialGuess")
        driver._check(L.HYPREDRV_LinearSolverCreate(drv._h), "LinearSolverCreate")
        driver._check(L.HYPREDRV_LinearSolverSetup(drv._h), "LinearSolverSetup")
        _, hM = drv.device_handles()
        ndist, nlev = hdk.amg_local_levels(hM)
        mine = {"ndist": ndist, "nlev": nlev, "tail": []}
        for l in range(nlev):
            r, a, p = C.c_int64(), C.c_int64(), C.c_int64()
            hdk.check(hdk.lib().hdk_amg_level_info(hM, l, C.byref(r), C.byref(a), C.byref(p)))
            if rank == 0 and l >= ndist:
                e = {"A": _level(hM, l, 0, r.value, a.value)}
                if l + 1 < nlev:
                    cf = np.empty(r.value, np.int32)
                    hdk.check(hdk.lib().hdk_amg_get_cf(hM, l, cf.ctypes.data))
                    e.update(cf=cf, P=_level(hM, l, 1, r.value, p.value), S=_level(hM, l, 3, r.value, a.value))
                    if l == 0:
                        nc1 = int(np.count_nonzero((cf == 1) | (cf == -2)))
                        rp = np.empty(nc1 + 1, np.int32)
                        hdk.check(hdk.lib().hdk_amg_get_matrix(hM, l, 4, rp.ctypes.data, None, None))
                        e["S2"] = _level(hM, l, 4, nc1, int(rp[nc1]))
                mine["tail"].append(e)
        driver._check(L.HYPREDRV_LinearSolverApply(drv._h), "LinearSolverApply")
        it, cv = C.c_int(), C.c_int()
        driver._check(L.HYPREDRV_LinearSolverGetNumIter(drv._h, C.byref(it)), "GetNumIter")
        driver._check(L.HYPREDRV_LinearSolverGetConverged(drv._h, C.byref(cv)), "GetConverged")
        x_loc = drv.get_solution()
        L.HYPREDRV_LinearSolverDestroy(drv._h)
    xs = [torch.zeros(int(cuts[r + 1] - cuts[r]), dtype=torch.float64) for r in range(world)]
    for r in range(world):
        if r == rank:
            xs[r].copy_(torch.from_numpy(np.ascontiguousarray(x_loc)))
        dist.broadcast(xs[r], r)
    allh = [None] * world
    dist.gather_object(mine, allh if rank == 0 else None, dst=0)
    ok = True
    if rank == 0:
        from oracle import oracle as O
        import aggressive_oracle as AO
        x = torch.cat(xs).numpy()
        H = AO.Hierarchy(A, O.default_params(True), num_levels=1)
        xr, ir = O.pcg(A, b, M=H, rel_tol=tol, max_iter=200)
        rel = np.linalg.norm(x - xr) / np.linalg.norm(xr)
        res = np.linalg.norm(b - A @ x) / np.linalg.norm(b)
        ok = bool(cv.value) and it.value == ir["iters"] and rel <= 1e-8 and res < tol * 1.0001
        msg = "hier=ok"
        h0 = allh[0]
        if h0["nlev"] != H.nlev:
            ok, msg = False, f"hier=levels {h0['nlev']} vs oracle {H.nlev}"
        else:
            if h0["ndist"] != 0:
                ok, msg = False, f"hier={h0['ndist']} row-distributed levels"
            for k, e in enumerate(h0["tail"]):
                l = h0["ndist"] + k
                refs = {"A": H.A(l)}
                if "P" in e:
                    refs.update(P=H.P(l), S=H.S(l))
                    if "S2" in e:
                        refs["S2"] = H.S2(l)
                    if not np.array_equal(e["cf"], H.cf(l)):
                        ok, msg = False, f"hier=C/F differs on level {l}"
                for w, ref in refs.items():
                    rp, cj, va = e[w]
                    same = np.array_equal(rp, ref.indptr) and np.array_equal(cj, ref.indices)
                    if w not in ("S", "S2"):
                        same = same and np.array_equal(va, ref.data)
                    if not same:
                        ok, msg = False, f"hier={w} differs on level {l}"
            if ok:
                msg = f"hier=bit-identical({H.nlev} levels)"
        print(f"MPAGG world={world} n={n} cuts={list(map(int, cuts))} levels={H.sizes()} dist_levels={h0['ndist']} "
              f"iters={it.value} oracle_iters={ir['iters']} rel_diff={rel:.2e} true_res={res:.2e} {msg} ok={ok}", flush=True)
    flag = torch.tensor([1 if ok else 0])
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
