"""Scalar vs systems AMG on clamped Q1 linear elasticity (tests/systems_cases.py).

Assembles the 3-D elasticity problem with m^3 free nodes (3 m^3 rows; default m = 96, about
2.65 M rows and 215 M non-zeros) and solves it with AMG-preconditioned PCG twice through the
device C-ABI: scalar AMG with the default settings, and the `elasticity_3d` preset settings
(num_functions = 3, strong_th = 0.8, interleaved labels).  For each run it reports the setup time
(median of 3 after a warm-up), the solve time, iterations, operator complexity and levels, with the
card name and power limit read in the same run, as JSON in <out>/bench_systems.json.

    python bench_systems.py [--m 96] [--tol 1e-8] [--out bench_systems_out]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def host_mem_gb() -> float:
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) / 2 ** 20
    except OSError:
        pass
    return float("nan")


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": plim}
    except Exception as e:                                    # noqa: BLE001
        return {"name": "unknown", "power_limit": "unknown", "error": str(e)}


def run(hdk, dA, db, params, reps, tol):
    setups = []
    M = None
    for k in range(reps + 1):                                 # k = 0: warm-up
        if M is not None:
            M.free()
        hdk.sync()
        t0 = time.perf_counter()
        M = hdk.DAmg(dA, params)
        hdk.sync()
        if k:
            setups.append(time.perf_counter() - t0)
    n = db.n
    dx = hdk.DVec(n)
    dx.fill(0.0)
    hdk.pcg(dA, db, dx, M, max_iter=500, rel_tol=tol)         # warm-up solve
    dx.fill(0.0)
    res = hdk.pcg(dA, db, dx, M, max_iter=500, rel_tol=tol)
    out = dict(setup_s=statistics.median(setups), setup_all_s=setups, solve_ms=res["solve_ms"], iters=res["iters"],
               converged=res["converged"], rel_res=res["rel_res_norm"], op_complexity=M.operator_complexity(),
               levels=M.nlev, sizes=M.sizes())
    M.free()
    return out, dx


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--m", type=int, default=96, help="free nodes per direction (3 m^3 rows)")
    ap.add_argument("--tol", type=float, default=1e-8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="bench_systems_out", help="directory of bench_systems.json")
    a = ap.parse_args()
    rows, nnz = 3 * a.m ** 3, 81 * 3 * a.m ** 3
    need_gb = nnz * 40 / 2 ** 30                               # assembly temporaries: padded blocks, columns, CSR
    have_gb = host_mem_gb()
    if have_gb == have_gb and need_gb > 0.8 * have_gb:
        sys.exit(f"bench_systems: m={a.m} needs about {need_gb:.0f} GB of host memory, {have_gb:.0f} GB available")

    import systems_cases as SC
    from hypredrive_b200 import hdk
    if hdk.device_count() <= 0:
        sys.exit("bench_systems: no CUDA device visible")
    hdk.init(0)
    t0 = time.perf_counter()
    A, b = SC.elasticity(a.m, 3)
    t_asm = time.perf_counter() - t0
    dA = hdk.DCsr.from_csr(A.indptr, A.indices, A.data)
    db = hdk.DVec(A.shape[0], b)
    res = {"case": f"Q1 elasticity, clamped face, {a.m}^3 free nodes", "rows": A.shape[0], "nnz": int(A.nnz),
           "assembly_s": t_asm, "tol": a.tol, "card": card()}
    scalar, xs = run(hdk, dA, db, hdk.amg_params(), a.reps, a.tol)
    systems, xv = run(hdk, dA, db, hdk.amg_params(num_functions=3, strong_th=0.8), a.reps, a.tol)
    for r, x in ((scalar, xs), (systems, xv)):
        r["true_rel_res"] = float(np.linalg.norm(b - A @ x.get()) / np.linalg.norm(b))
    res["scalar"], res["systems"] = scalar, systems
    res["card_after"] = card()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_systems.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: (v if k not in ("scalar", "systems") else {kk: vv for kk, vv in v.items() if kk != "sizes"})
                      for k, v in res.items()}))


if __name__ == "__main__":
    main()
