"""C callers of the HYPREDRV_* API, built by __graft_entry__.build() from tests/callers/ against
include/ + libHYPREDRV.so only, as an application links it:
  * laplacian.c -- the 7-point problem of hypredrive's C_laplacian example on a Cartesian process
    grid (MPI_Cart_* of the include/mpi.h shim), assembled through the HYPRE_IJ interface and
    solved five times.  `laplacian -n 10 10 10`: the STATISTICS table the library prints must have
    the layout of the reference's golden output (examples/refOutput/laplacian.txt, transcribed into
    tests/golden/laplacian_layout.json) with the same initial residual norm; the iteration count is
    the GPU-default chain's (PMIS + l1-Jacobi), checked against the oracle; also as two ranks
    (`-P 1 1 2`, communicator from the launcher environment).  The banner lines before the table
    are the program's own (its command line, and the process grid as the Cartesian communicator
    reports it).
  * csr_ingest.c -- unit test of the CSR ingest path: error bits through the error-module entry
    points, HYPRE_Int overflow, empty rows, ownership of CSR input and of a caller's IJ objects
    across matrix replacements, known answers, offset indptr slabs."""
import json
import os
import re
import subprocess

import numpy as np

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFBIN = os.path.join(ROOT, "build", "callers")


def _need(name):
    p = os.path.join(REFBIN, name)
    if not os.path.exists(p):
        pytest.fail(f"{p} missing: run __graft_entry__.build()")
    return p


def test_laplacian_example_runs_against_this_library(gpu):
    from oracle import oracle as O
    exe = _need("laplacian")
    r = subprocess.run([exe, "-n", "10", "10", "10"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    fx = json.load(open(os.path.join(ROOT, "tests", "golden", "laplacian_layout.json")))
    out = r.stdout.splitlines()
    for line in fx["setup_lines"]:
        assert line in out, line
    i = out.index("STATISTICS SUMMARY:")
    assert out[i:i + 6] == fx["table_header"]                         # banner, rules and both header rows
    rows = [l for l in out[i + 6:] if l.startswith("|")]
    assert len(rows) == len(fx["table_rows"]) == 5
    # the GPU-default chain's iteration count (the golden row holds the CPU-default chain: 5)
    A, b = O.gen("lap7", 10, 10, 10)
    H = O.Hierarchy(A, O.default_params(True))
    _, info = O.pcg(A, b, M=H, rel_tol=1e-6)
    for k, (row, gold) in enumerate(zip(rows, fx["table_rows"])):
        cells, gcells = [c.strip() for c in row.split("|")[1:-1]], [c.strip() for c in gold.split("|")[1:-1]]
        assert len(row) == len(gold) and [m.start() for m in re.finditer(r"\|", row)] == [m.start() for m in re.finditer(r"\|", gold)]
        assert cells[0] == gcells[0] == str(k)
        assert (cells[1] == "") == (gcells[1] == "")                    # LS build time only on the first entry
        assert cells[4] == fx["initial_res_norm"]                       # r0 = 10: the reference's own right-hand side
        assert float(cells[5]) < 1e-6 and int(cells[6]) == info["iters"]


def test_csr_ingest_unit_test(gpu):
    exe = _need("csr_ingest")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


def test_laplacian_example_as_two_ranks(gpu, tmp_path):
    """The same example as TWO processes (`-P 1 1 2`: a 1 x 1 x 2 Cartesian communicator of the
    `include/mpi.h` shim): the communicator comes from the launcher environment
    (`hdk_comm_init_from_env`, rank 0 publishes the NCCL id in a file), the hierarchy is set up
    row-distributed, and the printed iteration count / residual are the oracle's for the whole grid."""
    from oracle import oracle as O
    exe = _need("laplacian")
    shared = gpu.device_count() < 2
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1", MASTER_PORT="29777",
                   HDK_NCCL_ID_FILE=str(tmp_path / "nccl_id"), NCCL_SOCKET_IFNAME="lo", NCCL_IB_DISABLE="1")
        if shared:      # both ranks on the one GPU: NCCL needs distinct host ids, no peer-memory halo between them
            env.update(NCCL_HOSTID=f"hdk-ref-rank{r}", HDK_HALO_IPC="0")
        procs.append(subprocess.Popen([exe, "-n", "10", "10", "20", "-P", "1", "1", "2"], stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True, env=env, cwd=ROOT))
    outs = []
    for p in procs:
        try:
            out, _ = p.communicate(timeout=300)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise
        outs.append(out)
    assert all(p.returncode == 0 for p in procs), outs[0][-2000:] + outs[1][-2000:]
    out = outs[0].splitlines()
    assert "Processor topology:   1 x 1 x 2" in out
    rows = [l for l in out[out.index("STATISTICS SUMMARY:") + 6:] if l.startswith("|")]
    assert len(rows) == 5 and not any(l.startswith("|") for l in outs[1].splitlines())   # rank 0 prints the table
    A, b = O.gen("lap7", 10, 10, 20)
    _, info = O.pcg(A, b, M=O.Hierarchy(A, O.default_params(True)), rel_tol=1e-6)
    for row in rows:
        cells = [c.strip() for c in row.split("|")[1:-1]]
        assert int(cells[6]) == info["iters"]
        assert cells[4] == "%.2e" % np.linalg.norm(b) and cells[5] == "%.2e" % info["rel_res_norm"]
