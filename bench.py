#!/usr/bin/env python
"""bench.py -- headline benchmark of hypredrive_b200.

Metric (BASELINE.json): AMG-PCG solve DOF*iterations/s on the synthetic 3-D 7-point Poisson
system, 256^3 unknowns per GPU, BoomerAMG(PMIS, extended+i, l1-Jacobi)-PCG, fp64, tol 1e-6.
`--config` selects the other BASELINE.json configurations (C3 512^3 strong scaling, C4 27-point
anisotropic 256^3, C5 convection-diffusion GMRES(30) 256^3); the default stays the headline.

A "step" is one Krylov solve (the reference's "solve" timer region, src/internal/solver.c:668-683
of the reference) on an already set-up hierarchy.
  value : N_global * iterations / solve_seconds, operands resident in HBM, CUDA-event timed on
          the library's compute stream, max over ranks.
  e2e   : the same metric through the HYPREDRV_* C-ABI with HOST buffers: every step uploads the
          right-hand side from pinned host memory (SetRHSFromArray), solves (LinearSolverApply,
          including the reference's untimed r0 / final-residual evaluations) and downloads the
          solution (GetSolutionValues).
  roofline     : the fine-level fused residual SpMV (the kernel with the largest share of a
                 solve), algorithmic bytes / CUDA-event time, against MEASURED_PEAKS.json.
  cpu_baseline : the CPU oracle (restated reference, OpenMP) on the SAME configuration, rank 0,
                 N=1; its hierarchy and solution are also the parity check of the line
                 (`parity`: iterations, per-level sizes, SHA-256 of the C/F splittings and of
                 the coarse operators, solution difference).
  parity_companion (N > 1): a small companion grid solved by all ranks together and compared
                 with the oracle on rank 0 (iterations, solution difference).

`--impl reference` times the restated reference (oracle/) on the host cores with every thread
the box has; the real hypredrive+hypre cannot be built here (no hypre sources, no MPI, no
network).  Same `metric` string, same configuration; at N > 1 rank 0 runs one rank's share of
the weak-scaled problem and says so in `cpu_baseline.sample`.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

AMG_YAML = """preconditioner:
  amg:
    coarsening:
      type: pmis
      strong_th: 0.25
    interpolation:
      prolongation_type: extended+i
      max_nnz_row: 4
    relaxation:
      down_type: l1-jacobi
      up_type: l1-jacobi
      coarse_type: ge
      num_sweeps: 1
"""
PCG_YAML = "general:\n  statistics: off\nsolver:\n  pcg:\n    max_iter: 100\n    relative_tol: 1.0e-6\n" + AMG_YAML
GMRES_YAML = ("general:\n  statistics: off\nsolver:\n  gmres:\n    max_iter: 100\n    krylov_dim: 30\n"
              "    relative_tol: 1.0e-8\n" + AMG_YAML)
NORTH_STAR_YAML = PCG_YAML

# BASELINE.json configs.  edge = (nx, ny, nz) of ONE GPU's slab under weak scaling, of the whole
# problem under strong scaling (z-slabs either way: nz is split / multiplied)
CONFIGS = {
    "lap7_256": dict(kind="lap7", code=7, edge=(256, 256, 256), c=(1.0, 1.0, 1.0), solver="pcg", tol=1e-6,
                     scaling="weak", yaml=PCG_YAML,
                     metric="AMG-PCG solve DOF-iters/s, 7pt Poisson 256^3 per GPU",
                     what="synthetic 3D 7-point Poisson"),
    "lap7_512_strong": dict(kind="lap7", code=7, edge=(512, 512, 512), c=(1.0, 1.0, 1.0), solver="pcg", tol=1e-6,
                            scaling="strong", yaml=PCG_YAML,
                            metric="AMG-PCG solve DOF-iters/s, 7pt Poisson 512^3 total (strong scaling)",
                            what="synthetic 3D 7-point Poisson"),
    "lap27_aniso_256": dict(kind="lap27", code=27, edge=(256, 256, 256), c=(1.0, 1.0, 0.01), solver="pcg", tol=1e-6,
                            scaling="weak", yaml=PCG_YAML,
                            metric="AMG-PCG solve DOF-iters/s, 27pt anisotropic diffusion 256^3 per GPU",
                            what="synthetic 3D 27-point anisotropic diffusion c=(1,1,0.01)"),
    "convdif_gmres_256": dict(kind="convdif", code=107, edge=(256, 256, 256), c=(1e-3, 1.0, 0.1), solver="gmres",
                              tol=1e-8, scaling="strong", yaml=GMRES_YAML,
                              metric="AMG-GMRES(30) solve DOF-iters/s, convection-diffusion 256^3 total",
                              what="synthetic nonsymmetric 3D upwind convection-diffusion (kappa 1e-3, umax 1, dt 0.1)"),
}
SOLVER_DESC = {"pcg": "BoomerAMG(PMIS, ext+i, max_nnz_row 4, l1-Jacobi, GE coarse)-PCG tol 1e-6, x0 = 0",
               "gmres": "BoomerAMG(PMIS, ext+i, max_nnz_row 4, l1-Jacobi, GE coarse)-GMRES(30) tol 1e-8, x0 = 0"}

# dram__bytes_read.sum + dram__bytes_write.sum per launch of the fine-level residual SpMV at the
# headline workload (256^3 7-point rows per GPU), from the `ncu --set full` capture summarised
# under profiles/ (see profiles/README.md); None when no capture exists for the selected kernel
NCU_TRAFFIC_BYTES = {"lap7_256": {"k_spmv_sell": 1.7438e9 + 0.1177e9,   # profiles/r02_spmv_sell_ncu_full.csv, first launch
                                   "k_spmv_tma": 1.7404e9 + 0.1303e9}}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            return json.load(fh).get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


def global_dims(cfg, world):
    nx, ny, nz = cfg["edge"]
    if cfg["scaling"] == "weak":
        return nx, ny, nz * world
    return nx, ny, nz


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        self.tmp.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.tmp.read().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.tmp.name)
        except OSError:
            pass
        if sm:
            sm.sort()
            out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        return out


# ---------------------------------------------------------------------------------------------
# CPU legs (oracle/): the only place bench.py executes the oracle -- as the baseline and checker
# ---------------------------------------------------------------------------------------------
def oracle_threads():
    """All host cores, set by assignment (torchrun exports OMP_NUM_THREADS=1 to its children) and
    through omp_set_num_threads; returns the team size the oracle really runs with."""
    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0)) or cores
    except Exception:
        pass
    os.environ["OMP_NUM_THREADS"] = str(cores)
    from oracle import oracle as O
    return O.set_threads(cores)


def run_cpu_oracle(cfg, dims, steps, warmup, keep=False, budget_s=900.0):
    """Restated reference on the host cores.  Returns a dict (value, per-solve seconds, iterations,
    setup seconds, and -- keep=True -- the hierarchy and solution for the parity check)."""
    from oracle import oracle as O
    nx, ny, nz = dims
    t0 = time.time()
    A, b = O.gen(cfg["kind"], nx, ny, nz, c=cfg["c"])
    gen_s = time.time() - t0
    t0 = time.time()
    H = O.Hierarchy(A, O.default_params(True))
    setup_s = time.time() - t0
    solve = O.pcg if cfg["solver"] == "pcg" else O.gmres
    times, iters, x, done = [], 0, None, 0
    t_start = time.time()
    for s in range(warmup + steps):
        t0 = time.time()
        x, info = solve(A, b, M=H, rel_tol=cfg["tol"], max_iter=100)
        dt = time.time() - t0
        iters = info["iters"]
        if s >= warmup:
            times.append(dt)
            done += 1
            # bounded: stop early (and say so through `steps`) if the run would exceed the budget
            if done < steps and (time.time() - t_start) + dt > budget_s:
                break
    per = sum(times) / max(len(times), 1)
    n = nx * ny * nz
    out = dict(value=n * iters / per, per=per, iters=iters, setup_s=setup_s, gen_s=gen_s, steps=done, n=n)
    if keep:
        out.update(H=H, x=x, A=A, b=b)
    return out


def sha(*arrays):
    import numpy as np
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def parity_against_oracle(hdk, hM, orc, x_gpu, iters_gpu, max_hash_nnz=30_000_000):
    """GPU hierarchy and solution against the oracle run of the same configuration."""
    import numpy as np
    H = orc["H"]
    L = hdk.lib()
    nlev = int(L.hdk_amg_num_levels(hM))
    sizes_gpu = []
    for l in range(nlev):
        r, a, p = C.c_int64(), C.c_int64(), C.c_int64()
        hdk.check(L.hdk_amg_level_info(hM, l, C.byref(r), C.byref(a), C.byref(p)))
        sizes_gpu.append((int(r.value), int(a.value)))
    sizes_orc = [tuple(int(v) for v in s) for s in H.sizes()]
    out = {"iters_gpu": int(iters_gpu), "iters_oracle": int(orc["iters"]), "levels_gpu": nlev, "levels_oracle": H.nlev,
           "level_sizes_equal": sizes_gpu == sizes_orc}
    cf_ok, ops_ok, hashed = True, True, []
    if out["level_sizes_equal"]:
        for l in range(nlev - 1):
            n = sizes_gpu[l][0]
            cf = np.empty(n, dtype=np.int32)
            hdk.check(L.hdk_amg_get_cf(hM, l, cf.ctypes.data))
            cf_ok = cf_ok and sha(cf) == sha(H.cf(l).astype(np.int32))
        for l in range(1, nlev):
            n, nnz = sizes_gpu[l]
            if nnz > max_hash_nnz:
                continue
            rp, cj, va = np.empty(n + 1, np.int32), np.empty(nnz, np.int32), np.empty(nnz, np.float64)
            hdk.check(L.hdk_amg_get_matrix(hM, l, 0, rp.ctypes.data, cj.ctypes.data, va.ctypes.data))
            Ao = H.A(l)
            ops_ok = ops_ok and sha(rp, cj, va) == sha(Ao.indptr.astype(np.int32), Ao.indices.astype(np.int32),
                                                       Ao.data.astype(np.float64))
            hashed.append(l)
    else:
        cf_ok = ops_ok = False
    xo = orc["x"]
    out.update(cf_sha_equal=bool(cf_ok), coarse_ops_sha_equal=bool(ops_ok), coarse_ops_levels_hashed=hashed,
               rel_diff=float(np.linalg.norm(x_gpu - xo) / np.linalg.norm(xo)),
               true_rel_res_gpu=float(np.linalg.norm(orc["b"] - orc["A"] @ x_gpu) / np.linalg.norm(orc["b"])))
    out["ok"] = bool(abs(out["iters_gpu"] - out["iters_oracle"]) <= 1 and out["level_sizes_equal"] and cf_ok and ops_ok
                     and out["rel_diff"] <= 1e-8)
    return out


def cpu_sample_dims(gdims, world):
    """The CPU legs run the complete configuration when it is at most ~1.5 x 256^3 rows; beyond that a
    bounded 256^3-sized slab of the same grid (the CPU's DOF*iters/s does not grow with the problem)."""
    if gdims[0] * gdims[1] * gdims[2] <= 256 ** 3 * 1.5:
        return gdims, "the complete configuration"
    dims = (gdims[0], gdims[1], max(1, (256 ** 3) // (gdims[0] * gdims[1])))
    return dims, (f"bounded sample: {dims[0]}x{dims[1]}x{dims[2]} slab of the {gdims[0]}x{gdims[1]}x{gdims[2]} problem "
                  f"(about one rank's share at N={world}); the CPU rate does not grow with N")


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg = args.cfg
    threads = oracle_threads()
    world = args.gpus
    gdims = global_dims(cfg, world)
    dims, sample_note = cpu_sample_dims(gdims, world)
    r = run_cpu_oracle(cfg, dims, max(1, args.steps), max(0, args.warmup))
    sample = (f"{cfg['what']} {dims[0]}x{dims[1]}x{dims[2]} ({sample_note}), same solver options, oracle/ (C + OpenMP, "
              f"{threads} threads), {r['steps']} solves after {args.warmup} warm-up")
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": r["value"], "unit": "DOF*iters/s",
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["per"] * 1e3,
        "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{cfg['what']} {gdims[0]}x{gdims[1]}x{gdims[2]} fp64, {SOLVER_DESC[cfg['solver']]}",
                   "name": args.config, "cpu_problem": f"{dims[0]}x{dims[1]}x{dims[2]}",
                   "note": "restated reference (oracle/, C + OpenMP) on the host cores; hypredrive+hypre itself "
                           "cannot be built in this image (hypre not vendored, no MPI, no network)"},
        "iterations": r["iters"], "setup_s": r["setup_s"], "solve_s": r["per"],
        "cpu_baseline": {"value": r["value"], "unit": "DOF*iters/s", "cores": threads, "kind": "port", "sample": sample,
                         "iterations": r["iters"], "setup_s": r["setup_s"], "solve_s": r["per"]},
        "e2e": {"value": r["value"], "unit": "DOF*iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def bind_to_gpu_numa(local):
    """N > 1: run this rank on the CPUs next to its GPU (NVML's ideal CPU set), so that the pinned host
    buffers of the end-to-end leg are first-touched on the GPU's NUMA node and the 8 concurrent
    H2D / D2H streams do not cross sockets.  Returns the number of CPUs bound to (0: left unchanged)."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(torch.cuda.get_device_properties(local).uuid)).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * i + b for i, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if cpus and len(cpus) < len(allowed):
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


def ours(args):
    import numpy as np
    from hypredrive_b200 import hdk, driver

    cfg = args.cfg
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    numa_cpus = 0
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        numa_cpus = bind_to_gpu_numa(local)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    if hdk.device_count() <= 0:
        raise SystemExit("bench.py: no CUDA device visible and there is no CPU fallback "
                         "(use --impl reference for the host-core baseline)")
    hdk.init(local)
    if world > 1:
        import torch
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            buf = (C.c_ubyte * 128)()
            hdk.check(hdk.lib().hdk_comm_unique_id(buf))
            uid = torch.tensor(list(buf), dtype=torch.uint8, device="cuda")
        dist.broadcast(uid, 0)
        raw = bytes(uid.cpu().tolist())
        hdk.check(hdk.lib().hdk_comm_init(rank, world, raw))

    nx, ny, nz_total = global_dims(cfg, world)
    plane = nx * ny
    cuts = [plane * ((nz_total * r) // world) for r in range(world + 1)]
    row_start, row_end = cuts[rank], cuts[rank + 1] - 1
    n_loc = row_end - row_start + 1
    n_glob = plane * nz_total
    L = driver.api()
    d = C.c_double()

    def barrier():
        hdk.sync()
        if dist is not None:
            dist.barrier()
        hdk.sync()

    drv = driver.HypreDrive(options=cfg["yaml"])
    t0 = time.time()
    drv.set_stencil(cfg["code"], nx, ny, nz_total, cfg["c"], row_start, row_end)   # assembled in HBM
    hdk.sync()
    build_s = time.time() - t0
    driver._check(L.HYPREDRV_LinearSystemSetInitialGuess(drv._h, None), "SetInitialGuess")
    driver._check(L.HYPREDRV_LinearSolverCreate(drv._h), "LinearSolverCreate")
    for _ in range(2):                                                            # warm-up setups: the stream-ordered pool
        driver._check(L.HYPREDRV_LinearSolverSetup(drv._h), "LinearSolverSetup")  # reaches its steady state (old + new hierarchy)
    setups = []
    for _ in range(3):
        barrier()
        driver._check(L.HYPREDRV_LinearSolverSetup(drv._h), "LinearSolverSetup")
        driver._check(L.HYPREDRV_LinearSolverGetSetupTime(drv._h, C.byref(d)), "GetSetupTime")
        setups.append(d.value)
    setup_s = sorted(setups)[1]
    if dist is not None:
        import torch
        t = torch.tensor([setup_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        setup_s = float(t[0])

    def one_solve():
        driver._check(L.HYPREDRV_LinearSystemResetInitialGuess(drv._h), "ResetInitialGuess")
        driver._check(L.HYPREDRV_LinearSolverApply(drv._h), "LinearSolverApply")
        it = C.c_int()
        driver._check(L.HYPREDRV_LinearSolverGetNumIter(drv._h, C.byref(it)), "GetNumIter")
        driver._check(L.HYPREDRV_LinearSolverGetSolveTime(drv._h, C.byref(d)), "GetSolveTime")
        return it.value, d.value

    # ---- device-resident leg -----------------------------------------------------------
    for _ in range(args.warmup):
        one_solve()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    prof = os.environ.get("HDK_PROFILE_RANGE") == "1"     # ncu --profile-from-start off
    if prof:
        hdk.lib().hdk_profiler_range(1)
    hdk.launch_count_reset()
    wall0 = time.time()
    solve_s, iters = 0.0, 0
    for _ in range(args.steps):
        it, s = one_solve()
        iters = it
        solve_s += s
    barrier()
    wall = time.time() - wall0
    if prof:
        hdk.lib().hdk_profiler_range(0)
    launches = hdk.launch_count_reset()
    if dist is not None:
        import torch
        t = torch.tensor([solve_s, wall], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        solve_s, wall = float(t[0]), float(t[1])
    per_step = solve_s / args.steps
    value = n_glob * iters / per_step
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, drv, driver, dist, rank, row_start, n_loc, n_glob)
    if os.environ.get("HDK_TIMELINE") == "1":             # diagnostics: per-operation times of one more solve, to stderr
        hdk.tune("timeline", 1)
        one_solve()
        hdk.tune("timeline", 0)

    # ---- end-to-end leg: host buffers through the C-ABI ---------------------------------
    import torch
    b_host = torch.empty(n_loc, dtype=torch.float64).pin_memory().numpy()
    pv = C.POINTER(C.c_double)()
    # fetch the generated right-hand side once so each step re-uploads the same data
    rhs_p = C.POINTER(C.c_double)()
    hdk.lib().HYPREDRV_LinearSystemGetRHSValues.argtypes = [C.c_void_p, C.POINTER(C.POINTER(C.c_double))]
    hdk.lib().HYPREDRV_LinearSystemGetRHSValues.restype = C.c_uint32
    driver._check(hdk.lib().HYPREDRV_LinearSystemGetRHSValues(drv._h, C.byref(rhs_p)), "GetRHSValues")
    b_host[:] = np.ctypeslib.as_array(rhs_p, shape=(n_loc,))

    def e2e_step():
        driver._check(L.HYPREDRV_LinearSystemSetRHSFromArray(drv._h, row_start, row_end, b_host.ctypes.data), "SetRHS")
        driver._check(L.HYPREDRV_LinearSystemResetInitialGuess(drv._h), "ResetInitialGuess")
        driver._check(L.HYPREDRV_LinearSolverApply(drv._h), "LinearSolverApply")
        driver._check(L.HYPREDRV_LinearSystemGetSolutionValues(drv._h, C.byref(pv)), "GetSolutionValues")
        it = C.c_int()
        driver._check(L.HYPREDRV_LinearSolverGetNumIter(drv._h, C.byref(it)), "GetNumIter")
        return it.value

    e2e_warm = min(args.warmup, 2)
    for _ in range(e2e_warm):
        e2e_step()
    barrier()
    t0 = time.time()
    for _ in range(args.steps):
        e2e_it = e2e_step()
    barrier()
    e2e_wall = time.time() - t0
    if dist is not None:
        t = torch.tensor([e2e_wall], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_wall = float(t[0])
    e2e_value = n_glob * e2e_it / (e2e_wall / args.steps)
    clocks = sampler.stop() if sampler else None
    x_gpu = np.ctypeslib.as_array(pv, shape=(n_loc,)).copy() if (rank == 0 and world == 1) else None

    # ---- roofline of the dominant kernel (fine-level SpMV), live -----------------------------
    hA, hM = drv.device_handles()
    peak, peak_src = measured_peaks()
    roof = None
    extra_kernels = {}
    ms, by = C.c_double(), C.c_double()
    names = {0: "spmv", 1: "l1_jacobi_fused", 2: "residual", 3: "pcg_xr_update", 4: "vcycle", 5: "pcg_p_update"}
    if world > 1:                            # what the multi-rank products add: the exchange alone, the product without it
        names.update({7: "halo_exchange", 8: "spmv_without_exchange"})
    for kid, name in names.items():          # collective at N > 1 (halo exchange inside): every rank runs it
        hdk.check(hdk.lib().hdk_time_kernel(hA, hM, kid, 20, C.byref(ms), C.byref(by)))
        extra_kernels[name] = {"ms": ms.value, "GBps": by.value / ms.value / 1e6, "bytes": by.value}
    if rank == 0:
        k0 = extra_kernels["residual"]   # largest share of a solve (profiles/r01_launch_shares.csv)
        kk, ka, km = C.c_int(), C.c_double(), C.c_int()
        hdk.check(hdk.lib().hdk_csr_spmv_kind(hA, C.byref(kk), C.byref(ka), C.byref(km)))
        kname = {0: "k_spmv_tma", 1: "k_spmv_vector", 2: "k_spmv_sell"}.get(kk.value, "k_spmv")
        traffic = NCU_TRAFFIC_BYTES.get(args.config, {}).get(kname) if not args.n and world == 1 else None
        roof = {"bound": "hbm", "achieved": k0["GBps"], "peak": peak, "unit": "GB/s", "frac": k0["GBps"] / peak,
                "traffic": traffic, "kernel": kname + "<RESIDUAL> (fine level, r = b - A x, per GPU)",
                "peak_source": peak_src,
                "note": "peak is the measured copy bandwidth (half reads, half writes); this kernel is 94% reads",
                "algorithmic_bytes": k0["bytes"], "ms": k0["ms"]}
    levels = []
    nlev = int(hdk.lib().hdk_amg_num_levels(hM))
    if dist is not None:
        dist.barrier()

    # ---- CPU baseline + parity on the SAME configuration (rank 0, N = 1 only) ----------------
    cpu, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = oracle_threads()
        cdims, cnote = cpu_sample_dims((nx, ny, nz_total), world)
        full = cdims == (nx, ny, nz_total)
        orc = run_cpu_oracle(cfg, cdims, 2, 1, keep=full)
        cpu = {"value": orc["value"], "unit": "DOF*iters/s", "cores": threads, "kind": "port",
               "sample": f"{cfg['what']} {cdims[0]}x{cdims[1]}x{cdims[2]} ({cnote}), same solver options, oracle/ "
                         f"(C + OpenMP, {threads} threads), {orc['steps']} solves after 1 warm-up",
               "iterations": orc["iters"], "setup_s": orc["setup_s"], "solve_s": orc["per"]}
        # the oracle of the complete configuration is also the parity check of this line
        parity = parity_against_oracle(hdk, hM, orc, x_gpu, e2e_it) if full else None
        del orc

    # ---- N > 1: companion grid solved by all ranks together, checked against the oracle --------
    companion = None
    if world > 1 and not args.no_cpu_baseline:
        companion = companion_parity(hdk, driver, dist, cfg, rank, world)

    if rank == 0:
        if True:                                  # (N > 1: rank 0's slabs of the distributed levels, then the replicated tail)
            for l in range(nlev):
                r_, a_, p_ = C.c_int64(), C.c_int64(), C.c_int64()
                hdk.check(hdk.lib().hdk_amg_level_info(hM, l, C.byref(r_), C.byref(a_), C.byref(p_)))
                levels.append([int(r_.value), int(a_.value), int(p_.value)])
        line = {
            "metric": cfg["metric"], "value": value, "unit": "DOF*iters/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3,
            "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{cfg['what']} {nx}x{ny}x{nz_total} fp64 ({n_loc} rows on rank 0, z-slabs), "
                                   f"{SOLVER_DESC[cfg['solver']]}",
                       "name": args.config,
                       "inputs_vs_L2": "operator and vectors exceed the 126 MB L2 (7-pt 256^3: 1.4 GB + 134 MB each); no flush needed",
                       "assembly": "device (HYPREDRV_LinearSystemSetStencil)",
                       "host_cpus_bound_to_gpu_numa_node": numa_cpus},
            "iterations": iters, "solve_s": per_step, "setup_s": setup_s, "setup_s_all": setups, "build_s": build_s,
            "wall_s_timed_region": wall, "levels": nlev, "level_rows_nnzA_nnzP": levels,
            "e2e": {"value": e2e_value, "unit": "DOF*iters/s", "h2d_bytes_per_step": 8 * n_glob,
                    "d2h_bytes_per_step": 8 * n_glob, "ms_per_step": e2e_wall / args.steps * 1e3,
                    "iterations": e2e_it},
            "gpu_launches": int(launches),
            "halo_exchange": {0: "none (1 rank)", 1: "nccl send/recv",
                              2: "peer-memory stores (CUDA IPC)"}.get(int(hdk.lib().hdk_comm_halo_mode()), "?"),
            "clocks": clocks, "roofline": roof, "kernels": extra_kernels,
            "cpu_baseline": cpu, "parity": parity, "parity_companion": companion,
            "published_reference": {"what": "hypre CUDA driven by hypredrive, 8xB200, lap-7 256^3 (docs figure, +-10%)",
                                    "setup_s": 0.10, "solve_s": 0.076},
        }
        print(json.dumps(line), flush=True)
    drv.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


def companion_parity(hdk, driver, dist, cfg, rank, world):
    """N > 1 parity where the driver can see it: a small grid of the same operator family, solved by
    all ranks together through the same distributed code (halo exchange, distributed hierarchy,
    allreduce), compared on rank 0 with the oracle on the global problem."""
    import numpy as np
    import torch
    nx, ny, nzl = 40, 36, 12
    nz = nzl * world
    plane = nx * ny
    rs, re = plane * nzl * rank, plane * nzl * (rank + 1) - 1
    hdk.tune("replicate_rows", 3000)        # keep the first levels of this small grid distributed
    try:
        with driver.HypreDrive(options=cfg["yaml"]) as drv:
            drv.set_stencil(cfg["code"], nx, ny, nz, cfg["c"], rs, re)
            drv.solve()
            x_loc = drv.get_solution()
            iters, conv = drv.last_iterations, drv.last_converged
    finally:
        hdk.tune("replicate_rows", 262144)
    xs = [torch.zeros(plane * nzl, dtype=torch.float64, device="cuda") for _ in range(world)]
    dist.all_gather(xs, torch.from_numpy(np.ascontiguousarray(x_loc)).cuda())
    out = None
    if rank == 0:
        from oracle import oracle as O
        oracle_threads()
        x = torch.cat(xs).cpu().numpy()
        A, b = O.gen(cfg["kind"], nx, ny, nz, c=cfg["c"])
        H = O.Hierarchy(A, O.default_params(True))
        xo, io = (O.pcg if cfg["solver"] == "pcg" else O.gmres)(A, b, M=H, rel_tol=cfg["tol"], max_iter=100)
        rel = float(np.linalg.norm(x - xo) / np.linalg.norm(xo))
        res = float(np.linalg.norm(b - A @ x) / np.linalg.norm(b))
        out = {"grid": f"{nx}x{ny}x{nz}", "ranks": world, "iters_gpu": int(iters), "iters_oracle": int(io["iters"]),
               "rel_diff": rel, "true_rel_res_gpu": res,
               "ok": bool(conv and abs(iters - io["iters"]) <= 1 and rel <= 1e-8 and res < cfg["tol"] * 1.0001)}
    return out


DUMP_SAMPLE = 1 << 20    # solution entries written by --dump-outputs (8 MB in float64)


def dump_positions(n_glob):
    """Global solution positions written by --dump-outputs: all of them up to DUMP_SAMPLE, else
    DUMP_SAMPLE draws with a fixed seed, sorted and without repeats (the same for the same grid)."""
    import numpy as np
    if n_glob <= DUMP_SAMPLE:
        return np.arange(n_glob)
    return np.unique(np.random.default_rng(0).integers(0, n_glob, DUMP_SAMPLE))


def gather_dump_sample(x_loc, row_start, n_glob, dist=None):
    """The solution at dump_positions(n_glob), from each rank's slab x_loc (global rows row_start..);
    collective at N > 1, where ranks hold consecutive slabs in rank order."""
    import numpy as np
    idx = dump_positions(n_glob)
    mine = idx[(idx >= row_start) & (idx < row_start + len(x_loc))] - row_start
    x = np.asarray(x_loc, dtype=np.float64)[mine]
    if dist is not None:
        parts = [None] * dist.get_world_size()
        dist.all_gather_object(parts, x)
        x = np.concatenate(parts)
    return x


def dump_outputs(outdir, drv, driver, dist, rank, row_start, n_loc, n_glob):
    """What the last timed solve hands its caller, as float64 .npy files under `outdir` (rank 0):
    solution.npy (at dump_positions), iterations.npy and final_rel_res_norm.npy (shape (1,)).
    Collective at N > 1."""
    import numpy as np
    L = driver.api()
    pv, it, rr = C.POINTER(C.c_double)(), C.c_int(), C.c_double()
    driver._check(L.HYPREDRV_LinearSystemGetSolutionValues(drv._h, C.byref(pv)), "GetSolutionValues")
    driver._check(L.HYPREDRV_LinearSolverGetNumIter(drv._h, C.byref(it)), "GetNumIter")
    driver._check(L.HYPREDRV_LinearSolverGetFinalRelativeResidualNorm(drv._h, C.byref(rr)), "GetFinalRelRes")
    x = gather_dump_sample(np.ctypeslib.as_array(pv, shape=(n_loc,)), row_start, n_glob, dist)
    if rank == 0:
        os.makedirs(outdir, exist_ok=True)
        np.save(os.path.join(outdir, "solution.npy"), x)
        np.save(os.path.join(outdir, "iterations.npy"), np.array([it.value], dtype=np.float64))
        np.save(os.path.join(outdir, "final_rel_res_norm.npy"), np.array([rr.value], dtype=np.float64))

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="lap7_256", choices=sorted(CONFIGS),
                    help="BASELINE.json configuration (default: the 256^3 headline)")
    ap.add_argument("--n", type=int, default=0, help="development override: cube edge instead of the config's")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed solve returned (solution, "
                         "iterations, final relative residual norm) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    args.cfg = CONFIGS[args.config]
    if args.n:                                    # development override of the cube edge (both arms)
        args.cfg = dict(args.cfg, edge=(args.n, args.n, args.n))
    if args.impl == "reference":
        return reference_arm(args)
    return ours(args)


if __name__ == "__main__":
    sys.exit(main())
