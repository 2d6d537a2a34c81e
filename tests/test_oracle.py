"""CPU tests pinning the ORACLE (oracle/) against the reference.

Three anchors (task section 3): the reference's own known-answer vectors restated from
pyamg/relaxation/tests/test_relaxation.py; golden fixtures produced by running the real reference
(tests/golden/make_golden.py); and digests of what the reference's compiled relaxation.h
returned on seeded inputs (tests/golden/reference/).  The oracle restates the reference's arithmetic in the same order,
so agreement is expected to rounding of identical operations (bit-exact in practice).
"""
import hashlib
import json
import os

import numpy as np
import pytest
import scipy.sparse as sp

import oracle
from conftest import GOLDEN_ALL as GOLDEN, GOLDEN_DIR, relerr

TIGHT = 1e-14   # oracle vs reference: same operations, same order


from kats import poisson1d, run_kats, gs_convergence_case, dense_gs_gold, block_jacobi_gold


# ---------------------------------------------------------------- reference KATs (tests/kats.py)
def test_kats_from_reference_tests():
    """pyamg/relaxation/tests/test_relaxation.py:148-197, :299-346, :364-411."""
    for case, got, exp in run_kats(oracle):
        assert np.allclose(got, exp, rtol=1e-14, atol=1e-15), case


def test_kat_gs_forward_backward_convergence():
    """test_relaxation.py:348-362."""
    r1, r2 = gs_convergence_case(oracle)
    assert r1 < 0.01 and r2 < 0.01 and abs(r1 - r2) < 1e-7


def test_kat_gauss_seidel_vs_triangular_solve():
    """test_relaxation.py:251-297: GS == (D+L)^-1 / (D+U)^-1 dense gold, all sweeps."""
    rng = np.random.default_rng(20260922)
    A = poisson1d(10).toarray()
    A += 0.1 * np.diag(rng.random(10))
    As = sp.csr_array(A)
    for sweep in ("forward", "backward", "symmetric"):
        x = rng.random(10)
        b = rng.random(10)
        g = dense_gs_gold(A, x, b, sweep)
        oracle.gauss_seidel(As, x, b, sweep=sweep)
        assert np.allclose(x, g, rtol=1e-13, atol=1e-14)


def test_kat_bsr_equals_csr():
    """test_relaxation.py:199-249: point Jacobi on BSR == on CSR for every block size dividing N."""
    rng = np.random.default_rng(7919)
    N = 12
    A = poisson1d(N).toarray() + np.diag(rng.random(N))
    for bs in (1, 2, 3, 4, 6, 12):
        x0 = rng.random(N)
        b = rng.random(N)
        xc = x0.copy()
        oracle.jacobi(sp.csr_array(A), xc, b, omega=0.8)
        xb = x0.copy()
        oracle.jacobi(sp.bsr_array(A, blocksize=(bs, bs)), xb, b, omega=0.8)
        assert np.allclose(xc, xb, rtol=1e-14, atol=1e-15)


def test_kat_block_jacobi_python_gold():
    """test_relaxation.py:1517-1777 style: block Jacobi against a dense Python gold incl. omega=1.1."""
    rng = np.random.default_rng(104729)
    N, bs = 12, 3
    A = poisson1d(N).toarray() + 0.3 * rng.random((N, N))
    nb = N // bs
    Dinv = np.zeros((nb, bs, bs))
    for i in range(nb):
        Dinv[i] = np.linalg.pinv(A[i * bs:(i + 1) * bs, i * bs:(i + 1) * bs])
    for omega in (1.0, 1.1):
        x = rng.random(N)
        b = rng.random(N)
        g = block_jacobi_gold(A, x, b, Dinv, bs, omega)
        oracle.block_jacobi(sp.bsr_array(A, blocksize=(bs, bs)), x, b, Dinv=Dinv, blocksize=bs, omega=omega)
        assert np.allclose(x, g, rtol=1e-12, atol=1e-13)


def test_make_system_contract():
    """test_relaxation.py:48-111: the validation contract of make_system."""
    A = poisson1d(4)
    with pytest.raises(ValueError):
        oracle.jacobi(A, [0, 0, 0, 0], np.zeros(4))
    with pytest.raises(ValueError):
        oracle.jacobi(A, np.zeros(5), np.zeros(4))
    with pytest.raises(TypeError):
        oracle.jacobi(A, np.zeros(4, dtype=np.float32), np.zeros(4))
    with pytest.raises(ValueError):
        oracle.jacobi(A, np.zeros(8)[::2], np.zeros(4))
    with pytest.raises(ValueError):
        oracle.jacobi(sp.csr_array(np.ones((3, 4))), np.zeros(3), np.zeros(3))


def test_zero_diagonal_and_duplicate_quirks():
    """SURVEY.md hazard 3: zero diagonal leaves the row alone; last diagonal duplicate wins."""
    indptr = np.array([0, 2, 4, 5], dtype=np.int32)
    indices = np.array([1, 2, 0, 1, 2], dtype=np.int32)           # row 0 has no diagonal
    data = np.array([1.0, 2.0, 3.0, 4.0, 5.0])
    A = sp.csr_array((data, indices, indptr), shape=(3, 3))
    x = np.array([1.0, 2.0, 3.0])
    oracle.gauss_seidel(A, x, np.ones(3))
    assert x[0] == 1.0
    indptr = np.array([0, 3], dtype=np.int32)
    A = sp.csr_array((np.array([2.0, 4.0, 8.0]), np.array([0, 0, 0], dtype=np.int32), indptr), shape=(1, 1))
    x = np.array([1.0])
    oracle.jacobi(A, x, np.array([16.0]))
    assert x[0] == 2.0     # diag = 8 (last), the earlier duplicates are dropped entirely


# ---------------------------------------------------------------- golden fixtures (real reference)
@pytest.mark.parametrize("name", GOLDEN)
def test_oracle_vcycle_matches_reference(name, load_golden):
    ml, ex = load_golden(name)
    cyc = oracle.Cycle(oracle.hierarchy_spec(ml), coarse_pinv=ml.coarse_solver.P)
    res = []
    x = cyc.solve(ex["b"], tol=0, maxiter=len(ex["residuals"]) - 1, residuals=res)
    assert relerr(x, ex["x_ref"]) < TIGHT
    # residual norms: b - A x cancels ~4 digits by the last cycle, so iterates equal to 2e-16 give norms equal to 1e-11
    assert np.allclose(res, ex["residuals"], rtol=1e-10, atol=0)
    assert relerr(cyc.solve(ex["b"], tol=0, maxiter=2, cycle="W"), ex["x_ref_W"]) < TIGHT
    assert relerr(cyc.solve(ex["b"], tol=0, maxiter=2, cycle="F"), ex["x_ref_F"]) < TIGHT
    res = []
    assert relerr(cyc.solve(ex["b"], tol=0, maxiter=3, cycle="AMLI", residuals=res), ex["x_ref_AMLI"]) < TIGHT
    assert np.allclose(res, ex["residuals_AMLI"], rtol=1e-12, atol=0)
    res = []
    x, info = cyc.solve(ex["b"], x0=ex["x0"], tol=1e-6, maxiter=50, residuals=res, return_info=True)
    assert info == int(ex["info_tol"][0])
    assert len(res) == len(ex["residuals_tol"])
    assert relerr(x, ex["x_ref_tol"]) < TIGHT


@pytest.mark.parametrize("name", GOLDEN)
def test_oracle_kernels_match_reference(name, load_golden):
    ml, ex = load_golden(name)
    lvl = ml.levels[0]
    A, x, b = lvl.A, ex["k_x"], ex["k_b"]
    assert relerr(oracle.matvec(A, x), ex["k_Ax"]) < TIGHT
    assert relerr(oracle.matvec(lvl.R, x), ex["k_Rx"]) < TIGHT
    assert relerr(oracle.matvec(lvl.P, ex["k_xc"]), ex["k_Pxc"]) < TIGHT
    spec = oracle.hierarchy_spec(ml)[0]
    for which, key in (("pre", "k_presmoother"), ("post", "k_postsmoother")):
        y = x.copy()
        oracle._smooth(spec[which], A, y, b, "oracle")
        assert relerr(y, ex[key]) < TIGHT
    Ac = A.tocsr()
    y = x.copy(); oracle.jacobi(Ac, y, b, omega=0.7)
    assert relerr(y, ex["k_jacobi_w07"]) < TIGHT
    y = x.copy(); oracle.gauss_seidel(Ac, y, b, sweep="symmetric")
    assert relerr(y, ex["k_gs_symmetric"]) < TIGHT
    y = x.copy(); oracle.gauss_seidel(Ac, y, b, iterations=2, sweep="backward")
    assert relerr(y, ex["k_gs_backward2"]) < TIGHT
    y = x.copy(); oracle.sor(Ac, y, b, omega=1.3)
    assert relerr(y, ex["k_sor_13"]) < TIGHT


# ---------------------------------------------------------------- compiled reference cross-check
COMPILED_KERNELS = os.path.join(GOLDEN_DIR, "reference", "compiled_kernels.json")


def kernel_digests(ml, kernels):
    """Per level, the SHA-256 of what one application of every kernel a cycle uses there returns on seeded vectors:
    pre- and post-smoother, A x, R x, P x_c and a coarsest-level relaxation.  Only native kernels and SciPy's sparse
    matvecs take part (no BLAS), so the digests do not depend on the host CPU."""
    out = []
    for k, d in enumerate(oracle.hierarchy_spec(ml)):
        rng = np.random.default_rng(1000 + k)
        A = d["A"]
        x, b = rng.random(A.shape[0]), rng.random(A.shape[0])
        h = hashlib.sha256()
        for which in ("pre", "post", "coarse_relax"):
            if which in d:
                y = x.copy()
                oracle._smooth(d[which], A, y, b, kernels)
                h.update(y.tobytes())
        h.update(oracle.matvec(A, x, kernels).tobytes())
        if "P" in d:
            h.update(oracle.matvec(d["R"], x, kernels).tobytes())
            h.update(oracle.matvec(d["P"], rng.random(d["P"].shape[1]), kernels).tobytes())
        out.append(h.hexdigest())
    return out


@pytest.mark.parametrize("name", GOLDEN)
def test_oracle_equals_compiled_reference(name, load_golden):
    """The C restatement and the reference's own relaxation.h (+ SciPy matvec) agree bit for bit: the oracle's
    kernels against digests of what oracle/_ref/libamg_ref.so returned on the same inputs
    (tests/golden/reference/, written by make_golden.py --reference-checks)."""
    ml, _ = load_golden(name)
    with open(COMPILED_KERNELS) as f:
        want = json.load(f)[name]
    got = kernel_digests(ml, "oracle")
    assert got == want, [k for k, (g, w) in enumerate(zip(got, want)) if g != w]


@pytest.mark.parametrize("name", GOLDEN)
def test_oracle_pcg_matches_reference(name, load_golden):
    """ml.solve(accel='cg') = pyamg.krylov.cg preconditioned by one cycle (multilevel.py:479-508,
    krylov/_cg.py:97-196): V-cycle from x0 = 0 with tol 1e-10, and W-cycle from x0 with tol 1e-3."""
    ml, ex = load_golden(name)
    if "x_ref_cg" not in ex:
        pytest.skip("no CG golden for this hierarchy (nonsymmetric operator)")
    cyc = oracle.Cycle(oracle.hierarchy_spec(ml), coarse_pinv=ml.coarse_solver.P)
    res = []
    x, info = cyc.solve(ex["b"], tol=1e-10, maxiter=10, accel="cg", residuals=res, return_info=True)
    assert info == int(ex["info_cg"][0]) and len(res) == len(ex["residuals_cg"])
    assert relerr(x, ex["x_ref_cg"]) < TIGHT
    assert np.allclose(res, ex["residuals_cg"], rtol=1e-10)
    res = []
    x, info = cyc.solve(ex["b"], x0=ex["x0"], tol=1e-3, maxiter=30, accel="cg", cycle="W", residuals=res,
                        return_info=True)
    assert info == int(ex["info_cgW"][0]) and len(res) == len(ex["residuals_cgW"])
    assert relerr(x, ex["x_ref_cgW"]) < TIGHT


KRYLOV_RUNS = {"gmres": dict(tol=1e-10, maxiter=12, accel="gmres"),
               "gmresW": dict(tol=1e-3, maxiter=25, accel="gmres", cycle="W"),
               "fgmres": dict(tol=1e-10, maxiter=12, accel="fgmres"),
               "fgmresF": dict(tol=1e-4, maxiter=25, accel="fgmres", cycle="F"),
               "fgmresAMLI": dict(tol=1e-8, maxiter=5, accel="fgmres", cycle="AMLI"),
               "bicgstab": dict(tol=1e-10, maxiter=8, accel="bicgstab"),
               "bicgstabW": dict(tol=1e-4, maxiter=20, accel="bicgstab", cycle="W")}


@pytest.mark.parametrize("name", GOLDEN)
def test_oracle_gmres_and_fgmres_match_reference(name, load_golden):
    """ml.solve(accel='gmres' | 'fgmres') of the real reference (Householder GMRES, left-preconditioned; flexible
    GMRES, right-preconditioned; krylov/_gmres_householder.py, _fgmres.py) vs oracle/krylov.py: same iteration
    counts, info flags, residual histories and iterates (tests/golden/krylov/, made by make_golden.py --krylov)."""
    import os
    from conftest import GOLDEN_DIR
    ml, ex = load_golden(name)
    kg = np.load(os.path.join(GOLDEN_DIR, "krylov", name + ".npz"))
    cyc = oracle.Cycle(oracle.hierarchy_spec(ml), coarse_pinv=ml.coarse_solver.P)
    for tag, kw in KRYLOV_RUNS.items():
        kw = dict(kw)
        if tag in ("gmresW", "fgmresF", "bicgstabW"):
            kw["x0"] = ex["x0"]
        res = []
        x, info = cyc.solve(ex["b"], residuals=res, return_info=True, **kw)
        assert info == int(kg["info_" + tag][0]), tag
        assert len(res) == len(kg["residuals_" + tag]), tag
        assert np.allclose(res, kg["residuals_" + tag], rtol=1e-6, atol=1e-13 * res[0]), tag
        assert relerr(x, kg["x_ref_" + tag]) < 1e-9, tag
