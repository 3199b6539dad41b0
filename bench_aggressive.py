"""AMG-PCG with and without aggressive coarsening (agg_num_levels 0 and 1) on the 7-point Poisson and
the 27-point anisotropic (c = 1, 1, 0.01) problems, assembled on the device (hdk_csr_stencil).

For every problem and setting it reports the setup time (median of --reps after a warm-up), the PCG
solve time and iterations (tolerance 1e-6, as bench.py), the time of one V-cycle (mean over 20 after a
warm-up), the operator complexity and the levels, with the card name and power limit read in the same
run, as JSON in <out>/bench_aggressive.json.

    python bench_aggressive.py [--edge 256] [--reps 3] [--out bench_aggressive_out]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bench_systems import card      # noqa: E402

PROBLEMS = {"lap7": (7, (1.0, 1.0, 1.0)), "lap27_aniso": (27, (1.0, 1.0, 0.01))}


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
    dz = hdk.DVec(n)
    M.apply(db, dz)
    hdk.sync()
    t0 = time.perf_counter()
    for _ in range(20):
        M.apply(db, dz)
    hdk.sync()
    vcycle_ms = (time.perf_counter() - t0) / 20 * 1e3
    out = dict(setup_s=statistics.median(setups), setup_all_s=setups, solve_ms=res["solve_ms"], iters=res["iters"],
               converged=res["converged"], rel_res=res["rel_res_norm"], vcycle_ms=vcycle_ms,
               op_complexity=M.operator_complexity(), levels=M.nlev, sizes=M.sizes())
    M.free()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--edge", type=int, default=256, help="grid points per direction")
    ap.add_argument("--tol", type=float, default=1e-6)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="bench_aggressive_out", help="directory of bench_aggressive.json")
    a = ap.parse_args()
    from hypredrive_b200 import hdk
    if hdk.device_count() <= 0:
        sys.exit("bench_aggressive: no CUDA device visible")
    hdk.init(0)
    e = a.edge
    res = {"edge": e, "rows": e ** 3, "tol": a.tol, "card": card(), "problems": {}}
    for name, (kind, c) in PROBLEMS.items():
        dA, db = hdk.DCsr.stencil(kind, e, e, e, c)
        entry = {"nnz": dA.info()["global_nnz"]}
        for lev in (0, 1):
            entry[f"agg_num_levels={lev}"] = run(hdk, dA, db, hdk.amg_params(agg_num_levels=lev), a.reps, a.tol)
        res["problems"][name] = entry
        del dA, db
    res["card_after"] = card()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_aggressive.json"), "w") as f:
        json.dump(res, f, indent=1)
    brief = {k: v for k, v in res.items() if k != "problems"}
    brief["problems"] = {p: {k: ({kk: vv for kk, vv in v.items() if kk != "sizes"} if isinstance(v, dict) else v)
                             for k, v in d.items()} for p, d in res["problems"].items()}
    print(json.dumps(brief))


if __name__ == "__main__":
    main()
