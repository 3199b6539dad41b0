"""AMG-PCG with l1-Jacobi (relax 18) and Chebyshev (relax 16) smoothing, down and up.

Problems: the 7-point Poisson and the 27-point anisotropic (c = 1, 1, 0.01) problems, assembled on the
device (hdk_csr_stencil), and clamped Q1 elasticity with num_functions = 3 (bench_systems.py's builder,
tests/systems_cases.py).  Settings: l1-Jacobi (the baseline), Chebyshev order 2 with 10 CG-Lanczos steps,
order 3, order 2 with Gershgorin bounds, and on the 7-point problem also order 2 with one level of
aggressive coarsening.  For every problem and setting: the setup time (median of --reps after a
warm-up), the PCG iterations and solve time (tolerance --tol), the time of one V-cycle (mean over 20
after a warm-up); per problem, the fine-level Chebyshev sweep (hdk_time_kernel 9) and the l1-Jacobi
sweep (id 1), timed in the same run, in TB/s of algorithmic bytes.  The card name and power limit are
read in the same run; everything goes as JSON to <out>/bench_chebyshev.json.

    python bench_chebyshev.py [--edge 256] [--m 64] [--reps 3] [--out bench_chebyshev_out]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from bench_aggressive import run    # noqa: E402
from bench_systems import card      # noqa: E402

CHEB = dict(relax_down=16, relax_up=16)
SETTINGS = {
    "l1_jacobi": {},
    "cheby2_cg10": dict(CHEB, cheby_order=2, cheby_eig_est=10),
    "cheby3_cg10": dict(CHEB, cheby_order=3, cheby_eig_est=10),
    "cheby2_gershgorin": dict(CHEB, cheby_order=2, cheby_eig_est=0),
}


def sweeps(hdk, dA, reps=50):
    """fine-level sweeps timed in the same run: id 9 (Chebyshev order 2) and id 1 (l1-Jacobi)"""
    M = hdk.DAmg(dA, hdk.amg_params(**SETTINGS["cheby2_cg10"]))
    out = {}
    for name, kid, m in (("cheby2", 9, M), ("l1_jacobi", 1, None), ("cheby2_again", 9, M)):
        ms, by = hdk.time_kernel(dA, m, kid, reps)
        out[name] = dict(ms=ms, bytes=by, tbs=by / (ms * 1e-3) / 1e12)
    M.free()
    out["cheby_over_jacobi_tbs"] = min(out["cheby2"]["tbs"], out["cheby2_again"]["tbs"]) / out["l1_jacobi"]["tbs"]
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--edge", type=int, default=256, help="grid points per direction of the stencil problems")
    ap.add_argument("--m", type=int, default=64, help="free nodes per direction of the elasticity problem (3 m^3 rows)")
    ap.add_argument("--tol", type=float, default=1e-6)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="bench_chebyshev_out", help="directory of bench_chebyshev.json")
    a = ap.parse_args()
    from hypredrive_b200 import hdk
    if hdk.device_count() <= 0:
        sys.exit("bench_chebyshev: no CUDA device visible")
    hdk.init(0)
    e = a.edge
    res = {"edge": e, "tol": a.tol, "card": card(), "problems": {}}
    problems = {"lap7": (7, (1.0, 1.0, 1.0)), "lap27_aniso": (27, (1.0, 1.0, 0.01)), "elasticity": None}
    for name, spec in problems.items():
        if spec is None:
            import systems_cases as SC
            A, b = SC.elasticity(a.m, 3)
            dA = hdk.DCsr.from_csr(A.indptr, A.indices, A.data)
            db = hdk.DVec(A.shape[0], b)
            extra = dict(num_functions=3, strong_th=0.8)
            entry = {"rows": A.shape[0], "nnz": int(A.nnz), "num_functions": 3}
            del A, b
        else:
            dA, db = hdk.DCsr.stencil(spec[0], e, e, e, spec[1])
            extra = {}
            entry = {"rows": e ** 3, "nnz": dA.info()["global_nnz"]}
        for s, kw in SETTINGS.items():
            entry[s] = run(hdk, dA, db, hdk.amg_params(**kw, **extra), a.reps, a.tol)
        if name == "lap7":
            entry["cheby2_cg10_agg1"] = run(hdk, dA, db, hdk.amg_params(**SETTINGS["cheby2_cg10"], agg_num_levels=1),
                                            a.reps, a.tol)
        entry["fine_sweep"] = sweeps(hdk, dA)
        res["problems"][name] = entry
        del dA, db
    res["card_after"] = card()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_chebyshev.json"), "w") as f:
        json.dump(res, f, indent=1)
    brief = {k: v for k, v in res.items() if k != "problems"}
    brief["problems"] = {p: {k: ({kk: vv for kk, vv in v.items() if kk not in ("sizes", "setup_all_s")} if isinstance(v, dict) else v)
                             for k, v in d.items()} for p, d in res["problems"].items()}
    print(json.dumps(brief))


if __name__ == "__main__":
    main()
