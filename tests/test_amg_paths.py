"""CPU tests of the code-path census (tests/amg_paths.py) used by tests/test_gpu_unstructured.py:
the census against a per-row set construction, the mirrored thresholds against the library's
source, and the unstructured cases against the list of paths they must reach."""
import os
import re

import numpy as np
import pytest

import amg_paths as AP
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_census_matches_per_row_sets():
    A = AP.heavy_tailed(1500, 3)
    H = O.Hierarchy(A, O.default_params(True))
    assert H.nlev >= 2
    for l in range(H.nlev - 1):
        S, cf = H.S(l), H.cf(l, raw=True)
        chat, nf, ins = AP.row_census(S, cf)
        for i in range(S.shape[0]):
            if cf[i] != -1:
                assert chat[i] == 0 and nf[i] == 0
                continue
            strong = S.indices[S.indptr[i]:S.indptr[i + 1]]
            c_hat, f_nb = set(), 0
            for j in strong:
                if cf[j] > 0:
                    c_hat.add(j)
                elif cf[j] == -1:
                    f_nb += 1
                    c_hat.update(k for k in S.indices[S.indptr[j]:S.indptr[j + 1]] if cf[k] > 0)
            assert (chat[i], nf[i], ins[i]) == (len(c_hat), f_nb, len(c_hat) + f_nb), (l, i)
        # the oracle's untruncated P has |C-hat_i| entries in every F row
        P = O.Hierarchy(A, O.default_params(True, max_nnz_row=0)).P(l) if l == 0 else None
        if P is not None:
            lens = np.diff(P.indptr)
            assert np.array_equal(lens[cf == -1], chat[cf == -1])


def test_thresholds_mirror_the_library():
    src = open(os.path.join(ROOT, "hypredrive_b200", "csrc", "hdk_amg_setup.cu")).read()
    spmv = open(os.path.join(ROOT, "hypredrive_b200", "csrc", "hdk_spmv.cu")).read()

    def const(text, name):
        return int(re.search(rf"constexpr int\s+{name}\s*=\s*(\d+)", text).group(1))

    assert const(src, "IS_CAP") == AP.IS_CAP and const(src, "IS_F") == AP.IS_F
    assert const(src, "IW_LIST") == AP.IW_LIST and const(src, "IW_CAP") * 3 // 4 == AP.IW_INS
    assert const(src, "RW_LIMIT") == AP.RW_LIMIT and 256 * 5 // 8 == AP.RAP_256
    assert const(src, "GJ_ONE_CTA") == AP.GE_ONE_CTA
    assert const(spmv, "S_MAXR") == AP.S_MAXR
    assert re.search(r'getenv\("HDK_INTERP_THREAD_AVG"\); slow_avg = e \? atof\(e\) : 10\.0', src)
    assert "(double)Lc.n * Lc.n < 2.0e8" in src
    assert "(double)n * n < 2.0e8" in open(os.path.join(ROOT, "oracle", "amg_setup.c")).read()
    for b in AP.RAP_BANDS:
        assert re.search(rf"lo, \d+, {b if b != AP.RW_LIMIT else 'RW_LIMIT'}\);", src), b


@pytest.mark.parametrize("name", list(AP.CASES))
def test_case_reaches_its_paths(name):
    mk, prm, _, want = AP.CASES[name]
    A = mk()
    assert 2000 <= A.shape[0] <= 40000
    H = O.Hierarchy(A, O.default_params(True, **prm))
    got = AP.paths(H, prm, A)
    assert want <= got, sorted(want - got)
    assert AP.counts(H) == AP.COUNTS[name]


def test_max_coarse_size_boundary():
    """max_coarse_size equal to a level's size ends the hierarchy at that level; one less adds a level."""
    at, below = AP.COUNTS["coarse_size_at"]["rows"], AP.COUNTS["coarse_size_below"]["rows"]
    assert at[-1] == AP.CASES["coarse_size_at"][1]["max_coarse_size"] and below[:-1] == at and below[-1] < at[-1]


@pytest.mark.parametrize("config", list(AP.FORCED))
def test_forced_configuration_reaches_its_paths(config):
    env, want = AP.FORCED[config]
    got = set()
    for name in AP.FORCED_CASES:
        A = AP.CASES[name][0]()
        for kw in AP.FORCED_SETTINGS:
            got |= AP.paths(O.Hierarchy(A, O.default_params(True, **kw)), kw, A, AP.knobs(env))
    assert want <= got, sorted(want - got)


def test_cases_cover_every_path():
    """Each case's and forced configuration's claims are checked above; together they name every
    decision of the device setup and SpMV."""
    covered = set().union(*(c[3] for c in AP.CASES.values()), *(f[1] for f in AP.FORCED.values()))
    assert AP.REQUIRED <= covered, sorted(AP.REQUIRED - covered)
