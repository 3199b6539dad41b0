"""Child process of test_gpu_aggressive.test_forced_paths_run_the_aggressive_kernels.  The path switch
HDK_AGG_THREAD is read once per process, so the parent sets it in this process's environment.  For
every amg_paths case named on the command line the device hierarchy with aggressive coarsening is
compared with the restatement's bit for bit under torch.profiler (with and without a row limit); the
names of the setup kernels that ran are printed as one line `KERNELS <name>|<name>|...`.  Exits
non-zero on the first mismatch."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import amg_paths as AP                      # noqa: E402
from hypredrive_b200 import hdk            # noqa: E402
from test_gpu_aggressive import compare_aggressive_hierarchy, device_storage   # noqa: E402


def main():
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.init()
    hdk.init()
    hdk.tune("amg_keep_debug", 1)
    names = set()
    for name in sys.argv[1:]:
        make, params, _, _ = AP.CASES[name]
        A = device_storage(make())
        for agg in (dict(num_levels=2), dict(num_levels=1, num_paths=2, max_nnz_row=4)):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                try:
                    H, dA, M = compare_aggressive_hierarchy(A, agg, params)
                    r = np.random.default_rng(1).standard_normal(A.shape[0])
                    dr, dz = hdk.DVec(A.shape[0], r), hdk.DVec(A.shape[0])
                    M.apply(dr, dz)
                    z = H.precond(r)
                    assert np.allclose(dz.get(), z, rtol=1e-11, atol=1e-13 * np.abs(z).max()), "V-cycle"
                except AssertionError as e:
                    print(f"AGGPATH MISMATCH case={name} agg={agg}: {e}", flush=True)
                    sys.exit(1)
                hdk.sync()
            names |= {e.key for e in prof.key_averages() if e.key.startswith(("void hdk::k_", "hdk::k_"))}
            print(f"AGGPATH ok case={name} agg={agg} levels={H.nlev}", flush=True)
    print("KERNELS " + "|".join(sorted(n.split("(")[0] for n in names)), flush=True)


if __name__ == "__main__":
    main()
