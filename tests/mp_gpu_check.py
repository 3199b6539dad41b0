"""Multi-rank parity check, one process per rank (launched by torchrun; see test_gpu_multi.py).
Every rank assembles its slab of the system on its GPU, the ranks set up the AMG hierarchy and
solve together (row-distributed setup, halo exchange, allreduce) through the HYPREDRV C API, and
rank 0 compares with the CPU oracle run on the global problem:
  * the hierarchy, level by level: C/F splitting, interpolation and Galerkin operators of the
    row-distributed levels (the ranks' slabs with global columns, concatenated) and of the
    replicated tail -- bit for bit (pattern, storage order, values);
  * iterations (+-1), solution difference <= 1e-8, true residual below the tolerance.
With fewer GPUs than ranks (the driver's 1-GPU box) the ranks share cuda:0."""
import ctypes as C
import os
import sys

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist
    from hypredrive_b200 import hdk, driver

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    shared = torch.cuda.device_count() < world
    if shared:
        # fewer GPUs than ranks: the ranks share cuda:0.  NCCL refuses two ranks on one device of one
        # host, so every rank reports its own host id and the ranks talk through NCCL's socket
        # transport on the loopback interface.  The peer-memory halo path (kernels waiting on another
        # process of the same GPU) is switched off unless MPCHECK_SHARED_IPC=1.
        local = local % max(torch.cuda.device_count(), 1)
        os.environ["NCCL_HOSTID"] = f"hdk-one-gpu-rank{rank}"
        os.environ.setdefault("NCCL_SOCKET_IFNAME", "lo")
        os.environ["NCCL_IB_DISABLE"] = "1"
        if os.environ.get("MPCHECK_SHARED_IPC") != "1":
            os.environ["HDK_HALO_IPC"] = "0"
    torch.cuda.set_device(local)
    dist.init_process_group(backend="gloo")      # control plane of this script only (uid, results)
    hdk.init(local)
    uid = torch.zeros(128, dtype=torch.uint8)
    if rank == 0:
        buf = (C.c_ubyte * 128)()
        hdk.check(hdk.lib().hdk_comm_unique_id(buf))
        uid = torch.tensor(list(buf), dtype=torch.uint8)
    dist.broadcast(uid, 0)
    hdk.check(hdk.lib().hdk_comm_init(rank, world, bytes(uid.tolist())))

    kind = sys.argv[1] if len(sys.argv) > 1 else "lap7"
    amg_kw = {}
    if kind == "npz":
        # a general matrix and right-hand side written by the parent: npz <file> (indptr, indices,
        # data, b; optional max_levels), every rank passes its slab of rows through the CSR API
        sysdat = np.load(sys.argv[2])
        A_ip, A_cj, A_va, b_all = sysdat["indptr"], sysdat["indices"], sysdat["data"], sysdat["b"]
        if "max_levels" in sysdat:
            amg_kw["max_levels"] = int(sysdat["max_levels"])
        n_tot = b_all.size
        solver, tol = "pcg", 1e-8
        grid = f"n={n_tot}"
    else:
        nx, ny, nzl = (int(v) for v in (sys.argv[2:5] if len(sys.argv) > 4 else (12, 11, 6)))
        nz = nzl * world
        code, c, solver, tol = {"lap7": (7, (1.0, 1.0, 1.0), "pcg", 1e-6), "lap27": (27, (1.0, 1.0, 0.01), "pcg", 1e-6),
                                "convdif": (107, (1e-3, 1.0, 0.1), "gmres", 1e-8)}[kind]
        n_tot = nx * ny * nz
        grid = f"grid={nx}x{ny}x{nz}"
    if os.environ.get("MPCHECK_RAGGED") == "1":
        # uneven slabs that cut through grid planes: rank r owns rows [cuts[r], cuts[r+1])
        w = np.array([1.0 + 0.7 * ((r * 37) % 5) for r in range(world)])
        cuts = np.concatenate([[0], np.floor(np.cumsum(w) / w.sum() * n_tot).astype(np.int64)])
        cuts[-1] = n_tot
    elif kind == "npz":
        cuts = np.arange(world + 1, dtype=np.int64) * n_tot // world
    else:
        cuts = np.arange(world + 1, dtype=np.int64) * (nx * ny * nzl)
    rs, re = int(cuts[rank]), int(cuts[rank + 1]) - 1
    check_hier = os.environ.get("MPCHECK_HIER", "1") == "1" and os.environ.get("HDK_SETUP_REPLICATED") != "1"
    if check_hier:
        hdk.tune("amg_keep_debug", 1)
    opts = {"general": {"statistics": False}, "solver": {solver: {"relative_tol": tol, "max_iter": 100}},
            "preconditioner": {"amg": {"coarsening": amg_kw}} if amg_kw else "amg"}
    L = driver.api()
    hier = None
    with driver.HypreDrive(options=opts) as drv:
        if kind == "npz":
            lo, hi = int(A_ip[rs]), int(A_ip[re + 1])
            drv.set_matrix_from_csr(A_ip[rs:re + 2] - lo, A_cj[lo:hi], A_va[lo:hi], row_start=rs, row_end=re)
            drv.set_rhs(b_all[rs:re + 1])
        else:
            drv.set_stencil(code, nx, ny, nz, c, rs, re)
        driver._check(L.HYPREDRV_LinearSystemSetInitialGuess(drv._h, None), "SetInitialGuess")
        driver._check(L.HYPREDRV_LinearSystemResetInitialGuess(drv._h), "ResetInitialGuess")
        driver._check(L.HYPREDRV_LinearSolverCreate(drv._h), "LinearSolverCreate")
        driver._check(L.HYPREDRV_LinearSolverSetup(drv._h), "LinearSolverSetup")
        if check_hier:
            _, hM = drv.device_handles()
            ndist, nlev = hdk.amg_local_levels(hM)
            hier = {"ndist": ndist, "nlev": nlev, "levels": []}
            for l in range(ndist):
                r = C.c_int64()
                hdk.check(hdk.lib().hdk_amg_level_info(hM, l, C.byref(r), None, None))
                cf = np.empty(r.value, dtype=np.int32)
                hdk.check(hdk.lib().hdk_amg_get_cf(hM, l, cf.ctypes.data))
                hier["levels"].append({"cf": cf, "A": hdk.amg_rows(hM, l, 0), "P": hdk.amg_rows(hM, l, 1)})
            if rank == 0:                        # replicated tail: complete matrices on every rank
                hier["tail"] = []
                for l in range(ndist, nlev):
                    r, a, p = C.c_int64(), C.c_int64(), C.c_int64()
                    hdk.check(hdk.lib().hdk_amg_level_info(hM, l, C.byref(r), C.byref(a), C.byref(p)))
                    rp, cj, va = np.empty(r.value + 1, np.int32), np.empty(max(a.value, 1), np.int32), np.empty(max(a.value, 1))
                    hdk.check(hdk.lib().hdk_amg_get_matrix(hM, l, 0, rp.ctypes.data, cj.ctypes.data, va.ctypes.data))
                    e = {"A": (rp, cj[:a.value], va[:a.value])}
                    if l + 1 < nlev:
                        cf = np.empty(r.value, dtype=np.int32)
                        hdk.check(hdk.lib().hdk_amg_get_cf(hM, l, cf.ctypes.data))
                        prp, pcj, pva = np.empty(r.value + 1, np.int32), np.empty(max(p.value, 1), np.int32), np.empty(max(p.value, 1))
                        hdk.check(hdk.lib().hdk_amg_get_matrix(hM, l, 1, prp.ctypes.data, pcj.ctypes.data, pva.ctypes.data))
                        e.update(cf=cf, P=(prp, pcj[:p.value], pva[:p.value]))
                    hier["tail"].append(e)
        driver._check(L.HYPREDRV_LinearSolverApply(drv._h), "LinearSolverApply")
        it, cv = C.c_int(), C.c_int()
        driver._check(L.HYPREDRV_LinearSolverGetNumIter(drv._h, C.byref(it)), "GetNumIter")
        driver._check(L.HYPREDRV_LinearSolverGetConverged(drv._h, C.byref(cv)), "GetConverged")
        iters, conv = it.value, bool(cv.value)
        x_loc = drv.get_solution()
        L.HYPREDRV_LinearSolverDestroy(drv._h)
    xs = [torch.zeros(int(cuts[r + 1] - cuts[r]), dtype=torch.float64) for r in range(world)]
    for r in range(world):                       # uneven pieces: one broadcast per owner
        if r == rank:
            xs[r].copy_(torch.from_numpy(np.ascontiguousarray(x_loc)))
        dist.broadcast(xs[r], r)
    hiers = [None] * world
    dist.gather_object(hier, hiers if rank == 0 else None, dst=0)
    ok = True
    if rank == 0:
        from oracle import oracle as O
        x = torch.cat(xs).numpy()
        if kind == "npz":
            A, b = sp.csr_matrix((A_va, A_cj, A_ip), shape=(n_tot, n_tot)), b_all
        else:
            A, b = O.gen(kind, nx, ny, nz, c=c)
        H = O.Hierarchy(A, O.default_params(True, **amg_kw))
        xr, ir = (O.pcg if solver == "pcg" else O.gmres)(A, b, M=H, rel_tol=tol, max_iter=100)
        rel = np.linalg.norm(x - xr) / np.linalg.norm(xr)
        res = np.linalg.norm(b - A @ x) / np.linalg.norm(b)
        ok = bool(conv) and abs(iters - ir["iters"]) <= 1 and rel <= 1e-8 and res < tol * 1.0001
        hmsg = "hier=skipped"
        if check_hier:
            hok, hmsg = compare_hierarchy(hiers, H)
            ok = ok and hok
        print(f"MPCHECK kind={kind} world={world} {grid} levels={H.sizes()} iters={iters} oracle_iters={ir['iters']} "
              f"rel_diff={rel:.2e} true_res={res:.2e} {hmsg} ok={ok}", flush=True)
    flag = torch.tensor([1 if ok else 0])
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


def _cat_rows(parts):
    """Concatenate the ranks' (row0, indptr, cols, vals) slabs into one global CSR triple."""
    parts = sorted(parts, key=lambda p: p[0])
    ip = [np.zeros(1, dtype=np.int64)]
    off = 0
    for _, pip, _, _ in parts:
        ip.append(pip[1:] + off)
        off += int(pip[-1])
    return np.concatenate(ip), np.concatenate([p[2] for p in parts]), np.concatenate([p[3] for p in parts])


def compare_hierarchy(hiers, H):
    h0 = hiers[0]
    ndist, nlev = h0["ndist"], h0["nlev"]
    if nlev != H.nlev:
        return False, f"hier=levels {nlev} vs oracle {H.nlev}"
    for l in range(ndist):
        cf = np.concatenate([h["levels"][l]["cf"] for h in hiers])
        if not np.array_equal(cf, H.cf(l)):
            return False, f"hier=C/F splitting differs on distributed level {l}"
        for which, ref in (("A", H.A(l)), ("P", H.P(l))):
            ip, cj, va = _cat_rows([h["levels"][l][which] for h in hiers])
            if not (np.array_equal(ip, ref.indptr) and np.array_equal(cj, ref.indices)):
                return False, f"hier={which} pattern differs on distributed level {l}"
            if not np.array_equal(va, ref.data):
                return False, f"hier={which} values differ on distributed level {l}"
    for k, e in enumerate(h0["tail"]):
        l = ndist + k
        rp, cj, va = e["A"]
        ref = H.A(l)
        if not (np.array_equal(rp, ref.indptr) and np.array_equal(cj, ref.indices) and np.array_equal(va, ref.data)):
            return False, f"hier=A differs on replicated level {l}"
        if "P" in e:
            rp, cj, va = e["P"]
            ref = H.P(l)
            if not (np.array_equal(e["cf"], H.cf(l)) and np.array_equal(rp, ref.indptr) and np.array_equal(cj, ref.indices)
                    and np.array_equal(va, ref.data)):
                return False, f"hier=C/F or P differs on replicated level {l}"
    return True, f"hier=bit-identical({ndist} distributed + {nlev - ndist} replicated levels)"


if __name__ == "__main__":
    main()
