"""Child process of test_gpu_unstructured.test_forced_setup_paths_match_oracle.  The path switches
HDK_INTERP_THREAD_AVG, HDK_INTERP_SINGLE and HDK_RAP_SINGLE are read once per process, so the
parent sets them in this process's environment.  For every case named on the command line and
every truncation setting of amg_paths.FORCED_SETTINGS the device hierarchy is compared
with the oracle's bit for bit; prints one line per run and the paths the forced switches reach,
exits non-zero on the first mismatch."""
import os
import sys

import numpy as np
import scipy.sparse as sp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import amg_paths as AP                       # noqa: E402
from hypredrive_b200 import hdk              # noqa: E402
from test_gpu_kernels import _compare_hierarchy  # noqa: E402


def main():
    hdk.init()
    hdk.tune("amg_keep_debug", 1)
    knob = AP.knobs(os.environ)
    for name in sys.argv[1:]:
        mk = AP.CASES[name][0]
        A0 = mk()
        rp, cj, va = hdk.DCsr.from_scipy(A0).diag_arrays()
        A = sp.csr_matrix((va.copy(), cj.copy(), rp.copy()), shape=A0.shape)
        for kw in AP.FORCED_SETTINGS:
            try:
                H, dA, M = _compare_hierarchy(hdk, A, kw)
                n = A.shape[0]
                r = np.random.default_rng(1).standard_normal(n)
                dr, dz = hdk.DVec(n, r), hdk.DVec(n)
                M.apply(dr, dz)
                z = H.precond(r)
                assert np.allclose(dz.get(), z, rtol=1e-11, atol=1e-13 * np.abs(z).max()), "V-cycle"
            except AssertionError as e:
                print(f"FORCED MISMATCH case={name} {kw}: {e}", flush=True)
                sys.exit(1)
            print(f"FORCED ok case={name} {kw} levels={H.nlev} paths={sorted(AP.paths(H, kw, A, knob))}", flush=True)


if __name__ == "__main__":
    main()
