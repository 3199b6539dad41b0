"""Child process of test_gpu_systems.test_forced_paths_run_the_systems_kernels.  The interpolation
path switches (HDK_INTERP_THREAD_AVG, HDK_INTERP_SINGLE) are read once per process, so the parent
sets them in this process's environment.  For every systems case named on the command line the
device hierarchy is compared with the oracle's bit for bit under torch.profiler; the names of the
setup kernels that ran are printed as one line `KERNELS <name>|<name>|...`.  Exits non-zero on the
first mismatch."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import systems_cases as SC                 # noqa: E402
from hypredrive_b200 import hdk            # noqa: E402
from test_gpu_systems import compare_systems_hierarchy, device_storage   # noqa: E402


def main():
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.init()
    hdk.init()
    hdk.tune("amg_keep_debug", 1)
    names = set()
    for name in sys.argv[1:]:
        A_in, _, nf, dof, th = SC.cases()[name]
        A = device_storage(A_in)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            try:
                H, dA, M = compare_systems_hierarchy(A, nf, dof, dict(strong_th=th))
                r = np.random.default_rng(1).standard_normal(A.shape[0])
                dr, dz = hdk.DVec(A.shape[0], r), hdk.DVec(A.shape[0])
                M.apply(dr, dz)
                z = H.precond(r)
                assert np.allclose(dz.get(), z, rtol=1e-11, atol=1e-13 * np.abs(z).max()), "V-cycle"
            except AssertionError as e:
                print(f"SYSPATH MISMATCH case={name}: {e}", flush=True)
                sys.exit(1)
            hdk.sync()
        names |= {e.key for e in prof.key_averages() if e.key.startswith(("void hdk::k_", "hdk::k_"))}
        print(f"SYSPATH ok case={name} levels={H.nlev}", flush=True)
    print("KERNELS " + "|".join(sorted(n.split("(")[0] for n in names)), flush=True)


if __name__ == "__main__":
    main()
