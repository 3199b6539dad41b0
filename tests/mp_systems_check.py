"""Two-rank check of systems AMG (launched by torchrun; see test_gpu_systems.py).  Every rank passes
its slab of rows of the clamped Q1 elasticity matrix through the HYPREDRV CSR API with the
`elasticity_3d` preconditioner preset; the ranks rebuild the global hierarchy (the replicated setup
that N > 1 uses for num_functions > 1) and solve together.  Rank 0 compares with the CPU oracle run
on the global problem:
  * with MPCHECK_HIER=1 (every level replicated): A_l, S_l, C/F, P_l and the labels of every level,
    bit for bit;
  * otherwise: the labels of the row-distributed levels (the ranks' slabs, concatenated);
  * iterations equal, solution difference <= 1e-8, true residual below the tolerance.
MPCHECK_RAGGED=1 cuts the rows so that a node's three unknowns are split between the ranks.
With fewer GPUs than ranks the ranks share cuda:0 as in mp_gpu_check.py."""
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
    import systems_cases as SC

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
    A, b = SC.elasticity(m, 3)
    n = A.shape[0]
    if os.environ.get("MPCHECK_RAGGED") == "1":
        cuts = np.array([0, 3 * (n // 3 // world) + 1, n])          # through the middle of a node
    else:
        cuts = np.arange(world + 1, dtype=np.int64) * n // world
    rs, re = int(cuts[rank]), int(cuts[rank + 1]) - 1
    tol = 1e-8
    opts = {"general": {"statistics": False}, "solver": {"pcg": {"relative_tol": tol, "max_iter": 200}},
            "preconditioner": {"preset": "elasticity_3d"}}
    L = driver.api()
    full = os.environ.get("MPCHECK_HIER") == "1"
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
        mine = {"ndist": ndist, "nlev": nlev, "dof": [], "tail": []}
        for l in range(nlev):
            r, a, p = C.c_int64(), C.c_int64(), C.c_int64()
            hdk.check(hdk.lib().hdk_amg_level_info(hM, l, C.byref(r), C.byref(a), C.byref(p)))
            d = np.empty(r.value, np.int32)
            hdk.check(hdk.lib().hdk_amg_get_dof_func(hM, l, d.ctypes.data))
            mine["dof"].append(d)
            if full and rank == 0 and l >= ndist:
                e = {"A": _level(hM, l, 0, r.value, a.value)}
                if l + 1 < nlev:
                    cf = np.empty(r.value, np.int32)
                    hdk.check(hdk.lib().hdk_amg_get_cf(hM, l, cf.ctypes.data))
                    e.update(cf=cf, P=_level(hM, l, 1, r.value, p.value), S=_level(hM, l, 3, r.value, a.value))
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
        import systems_oracle as SO
        x = torch.cat(xs).numpy()
        H = SO.Hierarchy(A, O.default_params(True, strong_th=0.8), num_functions=3)
        xr, ir = O.pcg(A, b, M=H, rel_tol=tol, max_iter=200)
        rel = np.linalg.norm(x - xr) / np.linalg.norm(xr)
        res = np.linalg.norm(b - A @ x) / np.linalg.norm(b)
        ok = bool(cv.value) and it.value == ir["iters"] and rel <= 1e-8 and res < tol * 1.0001
        msg = "hier=ok"
        h0 = allh[0]
        if h0["nlev"] != H.nlev:
            ok, msg = False, f"hier=levels {h0['nlev']} vs oracle {H.nlev}"
        else:
            for l in range(H.nlev):
                d = np.concatenate([h["dof"][l] for h in allh]) if l < h0["ndist"] else h0["dof"][l]
                if not np.array_equal(d, H.dof(l)):
                    ok, msg = False, f"hier=labels differ on level {l}"
            for k, e in enumerate(h0["tail"]):
                l = h0["ndist"] + k
                refs = {"A": H.A(l)}
                if "P" in e:
                    refs.update(P=H.P(l), S=H.S(l))
                    if not np.array_equal(e["cf"], H.cf(l)):
                        ok, msg = False, f"hier=C/F differs on level {l}"
                for w, ref in refs.items():
                    rp, cj, va = e[w]
                    same = np.array_equal(rp, ref.indptr) and np.array_equal(cj, ref.indices)
                    if w != "S":
                        same = same and np.array_equal(va, ref.data)
                    if not same:
                        ok, msg = False, f"hier={w} differs on level {l}"
            if full and ok:
                msg = f"hier=bit-identical({H.nlev} levels)"
        print(f"MPSYS world={world} n={n} cuts={list(map(int, cuts))} levels={H.sizes()} dist_levels={h0['ndist']} "
              f"iters={it.value} oracle_iters={ir['iters']} rel_diff={rel:.2e} true_res={res:.2e} {msg} ok={ok}", flush=True)
    flag = torch.tensor([1 if ok else 0])
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
