"""Child process of test_gpu_chebyshev.test_chebyshev_kernels_run_on_sliced_ell_and_stream.  One 128^3
7-point hierarchy with order-3 Chebyshev down and up runs a V-cycle under torch.profiler: the fine level
(sliced-ELL) and the coarse levels (stream kernel) take the START / STEP / FIN passes.  The V-cycle is
compared with the restatement, and the names of the SpMV kernels that ran are printed as one line
`KERNELS <name>|<name>|...`."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from hypredrive_b200 import hdk             # noqa: E402
from test_gpu_chebyshev import compare_cheby_hierarchy, device_storage   # noqa: E402
from oracle import oracle as O             # noqa: E402


def main():
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.init()
    hdk.init()
    A = device_storage(O.gen("lap7", 128, 128, 128)[0])
    kw = dict(relax_down=16, relax_up=16)
    H, dA, M = compare_cheby_hierarchy(A, kw, dict(order=3, eig_est=10))
    r = np.random.default_rng(1).standard_normal(A.shape[0])
    dr, dz = hdk.DVec(A.shape[0], r), hdk.DVec(A.shape[0])
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        M.apply(dr, dz)
        hdk.sync()
    z = H.precond(r)
    if not np.allclose(dz.get(), z, rtol=1e-11, atol=1e-11 * np.abs(z).max()):
        print("CHEBPATH MISMATCH V-cycle", flush=True)
        sys.exit(1)
    names = {e.key for e in prof.key_averages() if "k_spmv" in e.key}
    print("KERNELS " + "|".join(sorted(n.split("(")[0] for n in names)), flush=True)


if __name__ == "__main__":
    main()
