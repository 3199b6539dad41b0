"""Two-rank check of Chebyshev smoothing (launched by torchrun; see test_gpu_chebyshev.py).  Every rank
passes its slab of rows of the 7-point Laplacian through the HYPREDRV CSR API with Chebyshev down and
up; with a small HDK_REPLICATE_ROWS the first levels are row-distributed, so their Gershgorin bounds
and CG-Lanczos dots are reduced over the ranks.  Rank 0 compares the eigenvalue bounds of every level
with the CPU restatement on the global problem (the one-rank values): Gershgorin to 1e-14, CG-Lanczos
to 1e-10; and the solve: iterations within one, solution difference <= 1e-8.  MPCHECK_RAGGED=1 cuts
the rows unevenly.  With fewer GPUs than ranks the ranks share cuda:0 as in mp_gpu_check.py."""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)


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

    m = int(sys.argv[1]) if len(sys.argv) > 1 else 24
    A, b = O.gen("lap7", m, m, m)
    n = A.shape[0]
    if os.environ.get("MPCHECK_RAGGED") == "1":
        cuts = np.array([0, n // 3 + 7, n])
    else:
        cuts = np.arange(world + 1, dtype=np.int64) * n // world
    rs, re = int(cuts[rank]), int(cuts[rank + 1]) - 1
    tol = 1e-8
    L = driver.api()
    ok = True
    for eig_est in (0, 10):
        opts = {"general": {"statistics": False}, "solver": {"pcg": {"relative_tol": tol, "max_iter": 200}},
                "preconditioner": {"amg": {"relaxation": {"down_type": "chebyshev", "up_type": "chebyshev",
                                                          "chebyshev": {"order": 2, "eig_est": eig_est}}}}}
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
            eigs = []
            for l in range(nlev - 1):
                e, c = np.zeros(2), np.zeros(4)
                hdk.check(hdk.lib().hdk_amg_get_cheby(hM, l, e.ctypes.data, c.ctypes.data, None))
                eigs.append((float(e[0]), float(e[1])))
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
        if rank == 0:
            import cheby_oracle as CO
            x = torch.cat(xs).numpy()
            base = O.Hierarchy(A, O.default_params(True, relax_down=16, relax_up=16))
            H = CO.Hierarchy(base, order=2, eig_est=eig_est)
            xr, ir = CO.pcg(A, b, M=H, rel_tol=tol, max_iter=200)
            rel = np.linalg.norm(x - xr) / np.linalg.norm(xr)
            rtol = 1e-14 if eig_est == 0 else 1e-10
            worst = 0.0
            good = nlev == base.nlev and ndist > 0
            for l, e in enumerate(eigs):
                ref = H.cheby(l)["eig"]
                worst = max(worst, max(abs(e[i] - ref[i]) / max(abs(ref[i]), 1e-300) for i in range(2)))
            good = good and worst <= rtol and bool(cv.value) and abs(it.value - ir["iters"]) <= 1 and rel <= 1e-8
            ok = ok and good
            print(f"MPCHEB world={world} n={n} cuts={list(map(int, cuts))} eig_est={eig_est} dist_levels={ndist} "
                  f"levels={nlev}/{base.nlev} eig_rel={worst:.2e} iters={it.value} oracle_iters={ir['iters']} "
                  f"rel_diff={rel:.2e} ok={good}", flush=True)
    flag = torch.tensor([1 if ok else 0])
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
