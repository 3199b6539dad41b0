"""CPU tests of Chebyshev smoothing (relax 16) in the CPU restatement (tests/cheby_oracle.c, built on the
parity oracle) and in the host option layer.  The coefficients are checked against a numpy statement
of the polynomial, the Gershgorin bounds against a plain statement over the CSR arrays, the CG-Lanczos
estimate against scipy's eigsh, one sweep against a dense evaluation of the polynomial, and the
V-cycle for symmetry."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla
from numpy.polynomial import Chebyshev, Polynomial

import amg_paths as AP
import cheby_oracle as CO
from hypredrive_b200 import driver, hdk
from oracle import oracle as O

INVALID_VAL = 0x200


def cases():
    return {
        "lap7": lambda: O.gen("lap7", 12, 11, 10)[0],
        "lap27_aniso": lambda: O.gen("lap27", 12, 10, 9, c=(1.0, 1.0, 0.01))[0],
        "fe_dirichlet": lambda: AP.fe_dirichlet(40, 35, 5),
    }


def _params(**kw):
    return O.default_params(True, **kw)


# ---- coefficients ------------------------------------------------------------------------------
def numpy_coefs(max_eig, min_eig, fraction, order):
    lower, upper = CO.interval(max_eig, min_eig, fraction)
    theta, delta = (upper + lower) / 2, (upper - lower) / 2
    Tk = Chebyshev.basis(order).convert(kind=Polynomial)
    p = Tk(Polynomial([theta / delta, -1.0 / delta])) / Tk(theta / delta)
    one_minus = (Polynomial([1.0]) - p).coef
    return one_minus[1:order + 1], lower, upper, theta, delta


EIGS = [(2.0, 0.1), (1.9, 0.0), (7.5, 1.2), (1.0, -0.4), (-0.5, -3.0), (12.0, 12.0)]


@pytest.mark.parametrize("order", [1, 2, 3, 4])
@pytest.mark.parametrize("eig", EIGS, ids=[f"{a}_{b}" for a, b in EIGS])
@pytest.mark.parametrize("fraction", [0.3, 1.0 / 30.0, 0.9])
def test_coefficients_match_numpy_polynomial(order, eig, fraction):
    ref, *_ = numpy_coefs(*eig, fraction, order)
    got = CO.coefs(*eig, fraction, order)
    assert np.allclose(got, ref, rtol=1e-12, atol=1e-12 * np.max(np.abs(ref))), (got, ref)


@pytest.mark.parametrize("order", [1, 2, 3, 4])
@pytest.mark.parametrize("eig", EIGS[:5], ids=[f"{a}_{b}" for a, b in EIGS[:5]])
def test_residual_polynomial_bounded_on_the_interval(order, eig):
    c = CO.coefs(*eig, 0.3, order)
    _, lower, upper, theta, delta = numpy_coefs(*eig, 0.3, order)
    t = np.linspace(lower, upper, 2001)
    s = np.polynomial.polynomial.polyval(t, c)
    bound = 1.0 / abs(Chebyshev.basis(order)(theta / delta))
    assert np.max(np.abs(1.0 - t * s)) <= bound * (1 + 1e-9)


def test_order_one_and_two_closed_forms():
    lower, upper = CO.interval(2.0, 0.1, 0.3)
    theta, delta = (upper + lower) / 2.0, (upper - lower) / 2.0
    assert CO.coefs(2.0, 0.1, 0.3, 1)[0] == 1.0 / theta
    den = delta * delta - 2.0 * (theta * theta)
    c = CO.coefs(2.0, 0.1, 0.3, 2)
    assert c[0] == -4.0 * theta / den and c[1] == 2.0 / den


def test_degenerate_interval_is_rejected():
    with pytest.raises(ValueError):
        CO.coefs(0.0, 0.0, 0.3, 2)
    with pytest.raises(ValueError):
        CO.coefs(np.inf, 0.0, 0.3, 2)


# ---- eigenvalue bounds ---------------------------------------------------------------------------
def gershgorin_plain(A, scale):
    A = sp.csr_matrix(A)
    hi, lo, ds = -np.inf, np.inf, np.zeros(A.shape[0])
    for i in range(A.shape[0]):
        d, R = 0.0, 0.0
        for k in range(A.indptr[i], A.indptr[i + 1]):
            if A.indices[k] == i:
                d = d + float(A.data[k])
            else:
                R = R + abs(float(A.data[k]))
        ad = abs(d)
        ds[i] = 1.0 / np.sqrt(ad) if scale else 1.0
        hi = max(hi, (ad + R) / ad if scale else ad + R)
        lo = min(lo, (ad - R) / ad if scale else ad - R)
    return ds, (hi, lo)


@pytest.mark.parametrize("scale", [0, 1])
@pytest.mark.parametrize("name", list(cases()))
def test_gershgorin_bounds_exact(name, scale):
    A = cases()[name]()
    ds, eig = CO.gershgorin(A, scale)
    ds_ref, eig_ref = gershgorin_plain(A, scale)
    assert np.array_equal(ds, ds_ref)
    assert eig == eig_ref


def test_zero_diagonal_is_rejected():
    A = sp.csr_matrix(np.array([[0.0, 1.0], [1.0, 2.0]]))
    with pytest.raises(ValueError):
        CO.gershgorin(A, 1)
    CO.gershgorin(A, 0)


@pytest.mark.parametrize("name", list(cases()))
def test_cg_lanczos_max_eig_against_eigsh(name):
    A = sp.csr_matrix(cases()[name]())
    d = np.abs(A.diagonal())
    B = sp.diags(1 / np.sqrt(d)) @ A @ sp.diags(1 / np.sqrt(d))
    true = spla.eigsh(B, k=1, which="LA", return_eigenvectors=False, tol=1e-14)[0]
    (mx, mn), m = CO.cg_eig(A, 10, 1)
    assert m == 10
    assert mx <= true * (1 + 1e-12) and mx >= 0.9 * true, (mx, true)
    assert 0.0 < mn <= mx


# ---- sweep, V-cycle ------------------------------------------------------------------------------
@pytest.mark.parametrize("order", [1, 2, 3, 4])
@pytest.mark.parametrize("scale", [0, 1])
def test_sweep_matches_dense_polynomial(order, scale):
    A = sp.csr_matrix(O.gen("lap27", 8, 7, 6, c=(1.0, 1.0, 0.1))[0])
    H = CO.Hierarchy(O.Hierarchy(A, _params(relax_down=16, relax_up=16)), order=order, scale=scale)
    c = H.cheby(0)
    rng = np.random.default_rng(3)
    f, u = rng.standard_normal(A.shape[0]), rng.standard_normal(A.shape[0])
    ds = c["ds"]
    B = np.diag(ds) @ A.toarray() @ np.diag(ds)
    S = sum(ci * np.linalg.matrix_power(B, i) for i, ci in enumerate(c["coefs"]))
    ref = u + ds * (S @ (ds * (f - A @ u)))
    got = H.sweep(0, f, u)
    assert np.linalg.norm(got - ref) <= 1e-12 * np.linalg.norm(ref)


@pytest.mark.parametrize("eig_est", [0, 10])
@pytest.mark.parametrize("name", list(cases()))
def test_chebyshev_vcycle_is_symmetric(name, eig_est):
    A = cases()[name]()
    H = CO.Hierarchy(O.Hierarchy(A, _params(relax_down=16, relax_up=16)), eig_est=eig_est)
    rng = np.random.default_rng(7)
    x, y = rng.standard_normal(A.shape[0]), rng.standard_normal(A.shape[0])
    Mx, My = H.precond(x), H.precond(y)
    assert abs(x @ My - Mx @ y) <= 1e-12 * np.linalg.norm(x) * np.linalg.norm(My)


def test_levels_without_type_16_carry_no_data_and_pcg_converges():
    A, b = O.gen("lap7", 14, 14, 14)
    base = O.Hierarchy(A, _params(relax_down=16, relax_up=18))
    H = CO.Hierarchy(base, order=3)
    assert H.cheby(0) is not None and H.cheby(base.nlev - 1) is None
    x, info = CO.pcg(A, b, M=H, rel_tol=1e-8)
    assert info["converged"] and np.linalg.norm(b - A @ x) <= 1e-7 * np.linalg.norm(b)
    # the Chebyshev data does not change the hierarchy: with type 18 everywhere the V-cycle is the oracle's
    Hj = CO.Hierarchy(O.Hierarchy(A, _params()))
    assert np.array_equal(Hj.precond(b), O.Hierarchy(A, _params()).precond(b))


def test_injected_bounds_replace_the_estimate():
    A = cases()["lap7"]()
    base = O.Hierarchy(A, _params(relax_down=16, relax_up=16))
    H = CO.Hierarchy(base, eigs=[(1.5, 0.25)] + [None] * (base.nlev - 1))
    assert H.cheby(0)["eig"] == (1.5, 0.25)
    assert np.array_equal(H.cheby(0)["coefs"], CO.coefs(1.5, 0.25, 0.3, 2))


# ---- host options ------------------------------------------------------------------------------
def _host_params(text, capfd=None):
    driver.initialize()
    L = driver.api()
    h = C.c_void_p()
    assert L.HYPREDRV_Create(1, C.byref(h)) == 0
    assert L.HYPREDRV_SetLibraryMode(h) == 0
    argv = (C.c_char_p * 1)(text.encode())
    code = L.HYPREDRV_InputArgsParse(1, argv, h)
    L.HYPREDRV_ErrorCodeClear()
    assert code == 0, hex(code)
    p = hdk.AmgParams()
    code = L.HYPREDRV_PreconGetDeviceParams(h, C.byref(p))
    msg = ""
    if code and capfd is not None:
        capfd.readouterr()
        L.HYPREDRV_ErrorCodeDescribe(code)
        msg = capfd.readouterr().err
    L.HYPREDRV_ErrorCodeClear()
    L.HYPREDRV_Destroy(C.byref(h))
    return code, p, msg


def _cheby_yaml(body, types=("down_type: chebyshev", "up_type: chebyshev")):
    lines = "".join(f"        {kv}\n" for kv in body)
    t = "".join(f"      {kv}\n" for kv in types)
    return f"solver: pcg\npreconditioner:\n  amg:\n    relaxation:\n{t}      chebyshev:\n{lines}"


def test_chebyshev_keys_reach_the_device_parameters():
    code, p, _ = _host_params(_cheby_yaml(["order: 3", "fraction: 0.2", "eig_est: 0", "variant: 0", "scale: 0"]))
    assert code == 0
    assert (p.relax_down, p.relax_up, p.cheby_order, p.cheby_eig_est, p.cheby_variant, p.cheby_scale) == (16, 16, 3, 0, 0, 0)
    assert p.cheby_fraction == 0.2
    code, p, _ = _host_params("solver: pcg\npreconditioner:\n  amg:\n    max_iter: 1\n")
    assert code == 0
    assert (p.cheby_order, p.cheby_fraction, p.cheby_eig_est, p.cheby_variant, p.cheby_scale) == (2, 0.3, 10, 0, 1)


@pytest.mark.parametrize("keys", [["order: 0"], ["order: 5"], ["fraction: 0"], ["fraction: 1.5"], ["eig_est: -1"],
                                  ["variant: 1"], ["variant: 2"], ["scale: 2"]],
                         ids=["order_lo", "order_hi", "fraction_lo", "fraction_hi", "eig_est", "variant1", "variant2", "scale"])
def test_rejected_chebyshev_options(keys, capfd):
    code, _, msg = _host_params(_cheby_yaml(keys), capfd)
    assert code & INVALID_VAL and "amg:relaxation:chebyshev" in msg


def test_coarse_type_chebyshev_enables_the_checks(capfd):
    code, p, msg = _host_params(_cheby_yaml(["order: 9"], types=("coarse_type: chebyshev",)), capfd)
    assert code & INVALID_VAL and "order" in msg


@pytest.mark.parametrize("keys", [["order: 9"], ["variant: 1", "fraction: 3"]], ids=["order", "variant_fraction"])
def test_chebyshev_keys_without_type_16_are_still_accepted(keys):
    code, p, _ = _host_params(_cheby_yaml(keys, types=("down_type: l1-jacobi",)))
    assert code == 0 and p.relax_down == 18 and p.relax_up == 18


# ---- device build --------------------------------------------------------------------------------
def test_chebyshev_kernel_register_budget():
    """Every Chebyshev variant of the sliced-ELL kernel keeps the occupancy of the fused-dot variants
    (<= 40 registers, 6 CTAs of 256 threads per SM) without spills, and the stream / warp-per-row
    variants stay within the budget of their kernel (64 with 4 CTAs per SM, 32)."""
    import os
    import re
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    lib = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "hypredrive_b200", "lib", "libHYPREDRV.so")
    out = subprocess.run([cuobjdump, "--dump-resource-usage", lib], capture_output=True, text=True).stdout
    found = re.findall(r"Function _ZN3hdk(\d+)(k_spmv_\w+?)ILi(1[0-3])E(\S*)E\w*:\s*\n\s*REG:(\d+) STACK:(\d+)", out)
    kinds = {}
    for _, kern, mode, _, reg, stack in found:
        kinds.setdefault(kern, set()).add(int(mode))
        limit = {"k_spmv_sell": 40, "k_spmv_tma": 64, "k_spmv_vector": 32}[kern]
        assert int(reg) <= limit, (kern, mode, reg)
        assert int(stack) <= 8, (kern, mode, stack)
    assert kinds == {k: {10, 11, 12, 13} for k in ("k_spmv_sell", "k_spmv_tma", "k_spmv_vector")}, kinds
    assert len([f for f in found if f[1] == "k_spmv_sell"]) == 4 * 6
