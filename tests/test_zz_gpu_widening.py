"""SURVEY.md 8(f)-2 widening: polynomial (chebyshev / richardson), indexed / CF / FC Jacobi, AIR hierarchies and
block Gauss-Seidel on the engine, against the real reference's goldens (cfg7-10) and the oracle.

This file sorts LAST on purpose: the kernels below were written after round 1's GPU budget was spent and have so
far only run on tests/emu (the engine's kernel sources on host fibers: `AMGB_TEST_EMU=1 pytest -m gpu`); under
`pytest -x` a failure here cannot hide the results of the B200-validated suites.

Tolerance as everywhere: ||x_gpu - x_ref|| / ||x_ref|| < 1e-12 in fp64 (1e-11 for the Krylov-accelerated runs).
"""
import os

import numpy as np
import pytest
import scipy.sparse as sp

import oracle
import pyamg_b200
from pyamg_b200.relaxation import relaxation as gpu_relax
from pyamg_b200.relaxation import smoothing
from conftest import GOLDEN_ALL, GOLDEN_WIDENING, golden_path, relerr, summation_order_sensitivity
import test_gpu_parity as T

# first hardware run of these kernels: a hang must not take the whole GPU tier down with it (pytest-timeout)
pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]
TOL = 1e-12


# ------------------------------------------------------------------ the parity suite of the BASELINE goldens, re-run
@pytest.mark.parametrize("name", GOLDEN_WIDENING)
def test_vcycle_matches_reference_golden(name, load_golden):
    T.test_vcycle_matches_reference_golden(name, load_golden)


@pytest.mark.parametrize("name", GOLDEN_WIDENING)
def test_w_and_f_cycles_match_reference_golden(name, load_golden):
    T.test_w_and_f_cycles_match_reference_golden(name, load_golden)


@pytest.mark.parametrize("name", GOLDEN_WIDENING)
def test_tolerance_stop_and_x0_match_reference_golden(name, load_golden):
    T.test_tolerance_stop_and_x0_match_reference_golden(name, load_golden)


@pytest.mark.parametrize("name", GOLDEN_WIDENING)
def test_vcycle_matches_oracle_on_fresh_rhs(name, load_golden):
    T.test_vcycle_matches_oracle_on_fresh_rhs(name, load_golden)


@pytest.mark.parametrize("env", [{"AMGB_NO_TILES": "1"}, {"AMGB_NO_PERMUTE": "1"}, {"AMGB_NO_GRAPH": "1"},
                                 {"AMGB_TILE_MIN_NNZ": "0"}, {"AMGB_TILE_MIN_NNZ": "0", "AMGB_TILE_G": "4"},
                                 {"AMGB_TAIL_NNZ": "600000"}, {"AMGB_NO_PDL": "1"}, {"AMGB_NO_CF_LAYOUT": "1"}])
@pytest.mark.parametrize("name", GOLDEN_WIDENING)
def test_every_kernel_path_matches_reference_golden(name, env, monkeypatch):
    T.test_every_kernel_path_matches_reference_golden(name, env, monkeypatch)


@pytest.mark.parametrize("name", GOLDEN_WIDENING)
def test_relaxation_kernels_and_matvecs_match_reference_golden(name, load_golden):
    T.test_relaxation_kernels_match_reference_golden(name, load_golden)
    T.test_matvecs_match_scipy_golden(name, load_golden)


@pytest.mark.parametrize("name", GOLDEN_WIDENING)
def test_gpu_resident_pcg_matches_reference_golden(name, load_golden):
    T.test_gpu_resident_pcg_matches_reference_golden(name, load_golden)


# ------------------------------------------------------------------ the smoother routines themselves vs the oracle
def _system(n=23, seed=5, bs=1):
    rng = np.random.default_rng(seed)
    A = sp.random(n * bs, n * bs, density=0.2, random_state=np.random.RandomState(seed), format="csr")
    A = (A + A.T + sp.eye(n * bs) * (4.0 + n * bs * 0.2)).tocsr()
    A.sort_indices()
    return A, rng.standard_normal(n * bs), rng.standard_normal(n * bs)


def test_polynomial_matches_oracle():
    A, x0, b = _system()
    for coef, its in (([0.3], 1), ([0.01, -0.2, 0.7], 2), ([1e-3, 2e-2, -0.1, 0.4], 1)):
        xg, xo = x0.copy(), x0.copy()
        gpu_relax.polynomial(A, xg, b, coef, iterations=its)
        oracle.polynomial(A, xo, b, coef, iterations=its)
        assert relerr(xg, xo) < TOL
    xg, xo = np.zeros_like(b), np.zeros_like(b)                      # the x = 0 shortcut of the reference (:646-649)
    gpu_relax.polynomial(A, xg, b, [0.05, 0.5])
    oracle.polynomial(A, xo, b, [0.05, 0.5])
    assert relerr(xg, xo) < TOL


def test_jacobi_indexed_and_cf_fc_jacobi_match_oracle():
    A, x0, b = _system(n=31, seed=8)
    n = A.shape[0]
    rng = np.random.default_rng(3)
    split = rng.random(n) < 0.4
    C, F = np.where(split)[0], np.where(~split)[0]
    for idx in (np.arange(n), C, F[::-1].copy(), np.array([2, 0]), np.array([5, 5, 7])):
        xg, xo = x0.copy(), x0.copy()
        gpu_relax.jacobi_indexed(A, xg, b, idx, iterations=2, omega=0.7)
        oracle.jacobi_indexed(A, xo, b, idx, iterations=2, omega=0.7)
        assert relerr(xg, xo) < TOL
    for fn_g, fn_o in ((gpu_relax.cf_jacobi, oracle.cf_jacobi), (gpu_relax.fc_jacobi, oracle.fc_jacobi)):
        for kw in ({}, {"iterations": 2, "f_iterations": 2, "c_iterations": 1, "omega": 0.6},
                   {"f_iterations": 0, "c_iterations": 3, "omega": 1.1}):
            xg, xo = x0.copy(), x0.copy()
            fn_g(A, xg, b, C, F, **kw)
            fn_o(A, xo, b, C, F, **kw)
            assert relerr(xg, xo) < TOL
    # the reference's doctest system (relaxation.py:1110-1118): rows outside the list are untouched
    A4 = sp.csr_array(np.array([[4.0, -1, 0, 0], [-1, 4, -1, 0], [0, -1, 4, -1], [0, 0, -1, 4]]))
    x, b4 = np.zeros(4), np.array([0.0, 1.0, 2.0, 3.0])
    gpu_relax.jacobi_indexed(A4, x, b4, [2, 3])
    assert np.array_equal(x[:2], [0.0, 0.0]) and relerr(x[2:], [0.5, 0.75]) < TOL


@pytest.mark.parametrize("bs", [1, 2, 3, 4])
def test_block_gauss_seidel_matches_oracle_and_compiled_reference(bs):
    from pyamg_b200.util import get_block_diag
    A, x0, b = _system(n=17, seed=20 + bs, bs=bs)
    Ab = A.tobsr(blocksize=(bs, bs))
    Dinv = get_block_diag(Ab, blocksize=bs, inv_flag=True)
    for sweep, its in (("forward", 1), ("backward", 2), ("symmetric", 2)):
        xg, xo = x0.copy(), x0.copy()
        gpu_relax.block_gauss_seidel(Ab, xg, b, iterations=its, sweep=sweep, blocksize=bs, Dinv=Dinv)
        oracle.block_gauss_seidel(Ab, xo, b, iterations=its, sweep=sweep, blocksize=bs, Dinv=Dinv,
                                  kernels="ref" if oracle.have_ref() else "oracle")
        assert relerr(xg, xo) < TOL
    with pytest.raises(ValueError):
        gpu_relax.block_gauss_seidel(Ab, x0.copy(), b, sweep="diagonal", blocksize=bs, Dinv=Dinv)


def test_smoother_factory_builds_what_the_engine_runs():
    """change_smoothers with the widened registry on hierarchies set up here (no reference needed): chebyshev +
    richardson on SA, cf/fc Jacobi on RS (needs lvl.splitting), block Gauss-Seidel default on elasticity."""
    from pyamg_b200.aggregation import smoothed_aggregation_solver
    from pyamg_b200.classical import ruge_stuben_solver
    from pyamg_b200.gallery import poisson, linear_elasticity
    cases = []
    np.random.seed(7)
    cases.append(smoothed_aggregation_solver(poisson((30, 30)), presmoother=("chebyshev", {"degree": 4}),
                                             postsmoother=("richardson", {"omega": 0.9, "iterations": 2})))
    cases.append(ruge_stuben_solver(poisson((10, 10, 10)), presmoother=("cf_jacobi", {"omega": 0.7}),
                                    postsmoother=("fc_jacobi", {"omega": 0.7, "f_iterations": 2})))
    A, B = linear_elasticity((10, 10))
    cases.append(smoothed_aggregation_solver(A, B=B, presmoother=("block_gauss_seidel", {"sweep": "symmetric"}),
                                             postsmoother=("block_gauss_seidel", {"sweep": "symmetric"})))
    for ml in cases:
        n = ml.levels[0].A.shape[0]
        b = np.random.default_rng(n).random(n)
        cyc = oracle.Cycle(oracle.hierarchy_spec(ml), coarse_pinv=ml.coarse_solver.dense_operator(ml.levels[-1].A))
        res = []
        x = ml.solve(b, tol=0, maxiter=3, residuals=res)
        assert relerr(x, cyc.solve(b, tol=0, maxiter=3)) < TOL
        assert res[-1] < res[0]
        assert relerr(ml.solve(b, tol=0, maxiter=2, cycle="W"), cyc.solve(b, tol=0, maxiter=2, cycle="W")) < TOL
    assert cases[0].levels[0].presmoother.__name__ == "chebyshev"
    assert cases[0].symmetric_smoothing is False and cases[1].symmetric_smoothing is False
    assert cases[2].symmetric_smoothing is True


# ------------------------------------------------------------------ AMLI cycles (multilevel.py:631-657)
@pytest.mark.parametrize("env", [{}, {"AMGB_NO_GRAPH": "1"}])
@pytest.mark.parametrize("name", GOLDEN_ALL)
def test_amli_cycle_matches_reference_golden(name, env, monkeypatch):
    """cycle='AMLI' (multilevel.py:631-657): goldens from the real reference; the oracle restatement is
    bit-identical to them on the CPU (tests/test_oracle.py)."""
    from pyamg_b200.hierarchy_io import load_hierarchy
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ml, ex = load_hierarchy(golden_path(name))
    # AMLI's step sizes are ratios of inner products of nearly collinear corrections: on the elasticity hierarchy
    # the REFERENCE's own iterate moves by 3e-9 when its SpMVs merely sum each row backwards (1e-16 for a V-cycle)
    tol = max(1e-11, 20 * summation_order_sensitivity(ml, ex["b"], tol=0, maxiter=3, cycle="AMLI"))
    res = []
    for _ in range(2):          # second call replays the captured graph
        x = ml.solve(ex["b"], tol=0, maxiter=3, cycle="AMLI", residuals=res)
        assert relerr(x, ex["x_ref_AMLI"]) < tol
        assert np.allclose(res, ex["residuals_AMLI"], rtol=max(1e-8, 100 * tol))
    # V-cycles afterwards are unaffected by the AMLI buffers / graph
    assert relerr(ml.solve(ex["b"], tol=0, maxiter=len(ex["residuals"]) - 1), ex["x_ref"]) < 1e-12


# ------------------------------------------------------------------ GPU-resident GMRES / FGMRES (SURVEY 8(f)-1)
@pytest.mark.parametrize("name", GOLDEN_ALL)
def test_gpu_resident_gmres_and_fgmres_match_reference_golden(name, load_golden):
    """solve(accel='gmres' | 'fgmres') with every long vector in HBM (amgb_solve_gmres) against the real
    reference's ml.solve(accel=...) (pyamg.krylov.gmres = Householder GMRES, left-preconditioned; fgmres,
    right-preconditioned; V, W, F and AMLI cycles as preconditioner): same iteration count, info flag, residual
    history and iterate.  Goldens: tests/golden/krylov/ (make_golden.py --krylov); the oracle restatement
    (oracle/krylov.py) is pinned to the same files on the CPU."""
    import os
    import warnings
    from conftest import GOLDEN_DIR
    from test_oracle import KRYLOV_RUNS
    ml, ex = load_golden(name)
    kg = np.load(os.path.join(GOLDEN_DIR, "krylov", name + ".npz"))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for tag, kw in KRYLOV_RUNS.items():
            kw = dict(kw)
            if tag in ("gmresW", "fgmresF", "bicgstabW"):
                kw["x0"] = ex["x0"]
            res = []
            x, info = ml.solve(ex["b"], residuals=res, return_info=True, **kw)
            assert info == int(kg["info_" + tag][0]), tag
            assert len(res) == len(kg["residuals_" + tag]), tag
            assert np.allclose(res, kg["residuals_" + tag], rtol=1e-5, atol=1e-12 * res[0]), tag
            # yardstick: how far the REFERENCE algorithm's own iterate moves under a rounding-level change (every
            # SpMV summing its rows backwards); 1e-15..1e-12 except with the AMLI cycle on elasticity (1e-9)
            bound = max(1e-9, 20 * summation_order_sensitivity(ml, ex["b"], **kw))
            assert relerr(x, kg["x_ref_" + tag]) < bound, tag
    # misuse mirrors the reference: AMLI needs fgmres (multilevel.py:487-490)
    with pytest.raises(ValueError):
        ml.solve(ex["b"], accel="gmres", cycle="AMLI")


# ------------------------------------------------------------------ Galerkin product on the GPU (SURVEY 8(f)-3)
def _bitwise_equal(C, D):
    C, D = sp.csr_array(C), sp.csr_array(D)
    return (C.shape == D.shape and np.array_equal(C.indptr, D.indptr) and np.array_equal(C.indices, D.indices)
            and np.array_equal(C.data.view(np.int64), D.data.view(np.int64)))


def test_spgemm_equals_scipy_csr_matmat_bit_for_bit():
    """amgb_host_csr_matmat vs SciPy's csr_matmat (what `R @ A @ P` runs, classical.py:201): identical indptr,
    identical column ORDER inside every row (reverse first appearance), identical value bits (same summation order,
    no FMA), exact zeros dropped; unsorted operands, empty rows / columns, rectangular shapes, all three row bins."""
    from pyamg_b200 import _engine as E
    for (m, k, n, d, seed) in [(30, 40, 25, 0.1, 1), (50, 50, 50, 0.3, 2), (7, 3, 9, 0.9, 3), (200, 150, 180, 0.05, 4),
                               (12, 60, 100, 0.9, 5)]:
        A = sp.csr_array(sp.random(m, k, density=d, random_state=np.random.RandomState(seed), format="csr"))
        B = sp.csr_array(sp.random(k, n, density=d, random_state=np.random.RandomState(seed + 50), format="csr"))
        A.data = np.round(A.data * 8) / 8 - 0.5            # exact cancellations: csr_matmat drops the zeros
        B.data = np.round(B.data * 8) / 8 - 0.5
        assert _bitwise_equal(A @ B, E.csr_matmat(A, B))
        C = A @ B                                          # a SciPy product has unsorted column indices
        assert _bitwise_equal(C.T.tocsr() @ C, E.csr_matmat(C.T.tocsr(), C))
        assert _bitwise_equal(C @ sp.csr_array((n, 4)), E.csr_matmat(C, sp.csr_array((n, 4))))   # empty operand
    with pytest.raises(ValueError):
        E.csr_matmat(sp.eye(3, format="csr"), sp.eye(4, format="csr"))
    dense = sp.csr_array(np.ones((2, 100))), sp.csr_array(np.ones((100, 100)))
    with pytest.raises(NotImplementedError):               # 10 000 products in one row: outside the supported bins
        E.csr_matmat(*dense)


@pytest.mark.parametrize("name", ["cfg1_rs_gs_poisson2d", "cfg3_rs_mcgs_poisson3d", "cfg9_air_fcjacobi_advection2d"])
def test_galerkin_product_reproduces_the_reference_hierarchy(name, load_golden):
    """(R A) P on the GPU == the coarse operators the REAL reference stored in the golden hierarchies, bit for bit
    (classical RS, and AIR where R != P^T)."""
    from pyamg_b200.util import galerkin
    ml, _ = load_golden(name)
    for lvl, nxt in zip(ml.levels[:-1], ml.levels[1:]):
        assert _bitwise_equal(galerkin(lvl.R, lvl.A, lvl.P, where="gpu"), nxt.A)


def test_host_setup_with_gpu_galerkin_builds_the_same_hierarchy(monkeypatch):
    from pyamg_b200.classical import ruge_stuben_solver
    from pyamg_b200.gallery import poisson
    A = poisson((14, 14, 14))
    ref = ruge_stuben_solver(A)
    monkeypatch.setenv("AMGB_GPU_RAP", "1")
    gpu = ruge_stuben_solver(A)
    assert len(ref.levels) == len(gpu.levels)
    for a, b in zip(ref.levels, gpu.levels):
        assert _bitwise_equal(a.A, b.A)


# ------------------------------------------------------------------ spectral-radius estimates on the GPU (8(f)-4)
def test_gpu_arnoldi_matches_the_host_estimator():
    """amgb_arnoldi_* (restarted modified-Gram-Schmidt Arnoldi with the basis resident in HBM) vs the host
    estimator of pyamg_b200.util (same algorithm as the reference's approximate_spectral_radius,
    pyamg/util/linalg.py:255-383): rho(A) and rho(D^-1 A) equal to rounding, incl. an exhausted Krylov space."""
    from pyamg_b200.gallery import poisson, stencil_grid, diffusion_stencil_2d
    from pyamg_b200.util import approximate_spectral_radius, get_diagonal
    for A in (poisson((20, 20)), stencil_grid(diffusion_stencil_2d(0.001, np.pi / 6, "FE"), (24, 24)), poisson((7,)),
              poisson((6, 6, 6))):
        A = sp.csr_array(A)
        D = get_diagonal(A, inv=True)
        for scale in (None, D):
            rh = approximate_spectral_radius(A, row_scale=scale, where="host")
            rg = approximate_spectral_radius(A, row_scale=scale, where="gpu")
            assert abs(rh - rg) <= 1e-8 * rh
    assert approximate_spectral_radius(poisson((20, 20)), where="gpu") == pytest.approx(7.955, rel=2e-2)   # lambda_max of the 20 x 20 5-point Laplacian; the estimator stops at 1 % (tol)


def test_sa_setup_with_gpu_spectral_radius_builds_the_same_hierarchy(monkeypatch):
    """Jacobi's omega and the prolongation smoother's rho from the device estimate.  The estimator stops as soon as
    the dominant Ritz pair is converged to 1 % (the reference's tol), where the value still responds to rounding at
    first order: host and device agree to ~1e-10, not to machine precision."""
    from pyamg_b200.aggregation import smoothed_aggregation_solver
    from pyamg_b200.gallery import poisson
    sm = ("jacobi", {"omega": 4.0 / 3.0})
    ref = smoothed_aggregation_solver(poisson((24, 24)), presmoother=sm, postsmoother=sm)
    monkeypatch.setenv("AMGB_GPU_RHO", "1")
    gpu = smoothed_aggregation_solver(poisson((24, 24)), presmoother=sm, postsmoother=sm)
    assert len(ref.levels) == len(gpu.levels)
    for a, b in zip(ref.levels[:-1], gpu.levels[:-1]):
        assert a.presmoother.keywords["omega"] == pytest.approx(b.presmoother.keywords["omega"], rel=1e-8)
        assert abs(a.P - b.P).max() <= 1e-8 * abs(a.P).max()


# ------------------------------------------------------------------ misuse of the new entry points fails loudly
def test_new_entry_points_reject_bad_arguments():
    import ctypes
    from pyamg_b200 import _engine as E
    L = E.lib()
    A = sp.csr_array(np.array([[4.0, -1.0], [-1.0, 4.0]]))
    keep = []
    M = E.as_matrix(A, keep)
    x, b = np.zeros(2), np.ones(2)
    S = gpu_relax._descriptor()
    S.kind = 99                                                    # unknown smoother kind
    assert L.amgb_host_relax(M, S, E.f64p(x), E.f64p(b)) == E.ENOTIMPL
    S.kind, S.n_coefficients = E.SM_POLYNOMIAL, 0                  # polynomial without coefficients
    assert L.amgb_host_relax(M, S, E.f64p(x), E.f64p(b)) == E.EINVAL
    S = gpu_relax._descriptor()
    idx = np.array([0, 5], dtype=np.int32)                          # row index outside the matrix
    S.kind, S.indices, S.n_indices = E.SM_JACOBI_INDEXED, E.i32p(idx), 2
    assert L.amgb_host_relax(M, S, E.f64p(x), E.f64p(b)) == E.EINVAL
    S = gpu_relax._descriptor()
    S.kind, S.blocksize = E.SM_BLOCK_GAUSS_SEIDEL, 2                # block Gauss-Seidel without Dinv
    assert L.amgb_host_relax(M, S, E.f64p(x), E.f64p(b)) == E.EINVAL
    assert L.amgb_host_relax(None, S, E.f64p(x), E.f64p(b)) == E.EINVAL
    # Arnoldi: run before any start vector, combination outside the basis
    h = ctypes.c_void_p()
    E.check(L.amgb_arnoldi_create(0, M, None, 5, ctypes.byref(h)))
    H = np.zeros(3 * 2)
    m = ctypes.c_int32(0)
    assert L.amgb_arnoldi_run(h, None, 1e-12, E.f64p(H), ctypes.byref(m)) == E.ESTATE
    coef = np.ones(4)
    assert L.amgb_arnoldi_combine(h, E.f64p(coef), 4) == E.EINVAL
    L.amgb_arnoldi_destroy(h)
    # GMRES on a one-unknown system is the caller's closed form; the Python mirror handles it on the host
    lvl = pyamg_b200.MultilevelSolver.Level()
    lvl.A = sp.csr_array(np.array([[2.0]]))
    ml1 = pyamg_b200.MultilevelSolver([lvl])
    assert ml1.solve(np.array([4.0]), maxiter=1, tol=0)[0] == pytest.approx(2.0)
    # cycle / accelerator combinations the reference rejects (multilevel.py:487-490)
    from pyamg_b200.classical import ruge_stuben_solver
    from pyamg_b200.gallery import poisson
    ml = ruge_stuben_solver(poisson((8, 8)))
    with pytest.raises(ValueError):
        ml.solve(np.ones(64), cycle="AMLI", accel="gmres")
    with pytest.raises(TypeError):
        ml.solve(np.ones(64), cycle="Z", accel="fgmres")


def test_krylov_module_keeps_the_preconditioned_solve_resident(load_golden):
    """pyamg.krylov-style calls `gmres(A, b, M=ml.aspreconditioner())`: with a pyamg_b200 preconditioner they run
    resident and equal ml.solve(accel=...); other operators / preconditioners are refused loudly."""
    import os
    import warnings
    from conftest import GOLDEN_DIR
    from pyamg_b200 import krylov
    ml, ex = load_golden("cfg3_rs_mcgs_poisson3d")
    kg = np.load(os.path.join(GOLDEN_DIR, "krylov", "cfg3_rs_mcgs_poisson3d.npz"))
    A = ml.levels[0].A
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        res = []
        x, info = krylov.gmres(A, ex["b"], tol=1e-10, maxiter=12, M=ml.aspreconditioner("V"), residuals=res)
        assert info == int(kg["info_gmres"][0]) and len(res) == len(kg["residuals_gmres"])
        assert relerr(x, kg["x_ref_gmres"]) < 1e-9
        x, info = krylov.fgmres(A.copy(), ex["b"], x0=ex["x0"], tol=1e-4, maxiter=25, M=ml.aspreconditioner("F"))
        assert relerr(x, kg["x_ref_fgmresF"]) < 1e-9
        x, info = krylov.cg(A, ex["b"], tol=1e-10, maxiter=10, M=ml.aspreconditioner())
        assert relerr(x, ex["x_ref_cg"]) < 1e-11
        x, info = krylov.bicgstab(A, ex["b"], tol=1e-10, maxiter=8, M=ml.aspreconditioner())
        assert info == int(kg["info_bicgstab"][0]) and relerr(x, kg["x_ref_bicgstab"]) < 1e-9
    with pytest.raises(NotImplementedError):
        krylov.gmres(A, ex["b"], M=None)
    with pytest.raises(NotImplementedError):
        krylov.gmres(2.0 * A, ex["b"], M=ml.aspreconditioner())
    with pytest.raises(NotImplementedError):
        krylov.cg(A, ex["b"], M=ml.aspreconditioner(), callback=lambda xk: None)


# ------------------------------------------------------------------ relaxation as the coarsest-level solver
@pytest.mark.parametrize("coarse", [("jacobi", {"iterations": 5, "omega": 0.8, "withrho": False}),
                                    ("sor", {"omega": 1.2, "iterations": 3, "sweep": "backward"}),
                                    ("chebyshev", {"degree": 2, "iterations": 2}),
                                    "gauss_seidel"])
def test_relaxation_coarse_solvers_match_oracle(coarse):
    """coarse_solver=<relaxation method> (multilevel.py:764-781: x = 0, then `iterations` sweeps, default 10)."""
    from pyamg_b200.classical import ruge_stuben_solver
    from pyamg_b200.gallery import poisson
    np.random.seed(3)
    ml = ruge_stuben_solver(poisson((24, 24)), max_coarse=40, coarse_solver=coarse)
    assert ml.levels[-1].A.shape[0] > 10
    b = np.random.default_rng(4).random(ml.levels[0].A.shape[0])
    cyc = oracle.Cycle(oracle.hierarchy_spec(ml))
    for cycle in ("V", "W"):
        assert relerr(ml.solve(b, tol=0, maxiter=3, cycle=cycle), cyc.solve(b, tol=0, maxiter=3, cycle=cycle)) < TOL
    with pytest.raises(NotImplementedError):
        pyamg_b200.coarse_grid_solver("cg")


def test_block_relaxation_coarse_solver_on_elasticity():
    from pyamg_b200.aggregation import smoothed_aggregation_solver
    from pyamg_b200.gallery import linear_elasticity
    A, B = linear_elasticity((12, 12))
    ml = smoothed_aggregation_solver(A, B=B, max_coarse=30, max_levels=2,
                                     coarse_solver=("block_gauss_seidel", {"sweep": "symmetric", "iterations": 6}))
    b = np.random.default_rng(5).random(A.shape[0])
    cyc = oracle.Cycle(oracle.hierarchy_spec(ml))
    assert relerr(ml.solve(b, tol=0, maxiter=3), cyc.solve(b, tol=0, maxiter=3)) < TOL


# ------------------------------------------------------------------ the device-pointer entry points (C ABI group 3)
class _DevMem:
    """Device arrays for the amgb_dev_* calls: torch CUDA tensors on a GPU, NumPy arrays on the kernel emulator."""

    def __init__(self):
        import os
        self.emu = os.environ.get("AMGB_TEST_EMU") == "1"
        if not self.emu:
            import torch
            self.torch = torch

    def up(self, a):
        a = np.ascontiguousarray(a)
        if self.emu:
            return a.copy()
        return self.torch.from_numpy(a.copy()).cuda()

    def ptr(self, d):
        import ctypes
        return ctypes.c_void_p(d.ctypes.data if self.emu else d.data_ptr())

    def get(self, d):
        if self.emu:
            return d.copy()
        self.torch.cuda.synchronize()
        return d.cpu().numpy()


def test_device_pointer_entry_points():
    """SURVEY.md 8(b): csr_spmv, csr_residual(+norm), csr_spmv_add, fused Jacobi(+residual), GS wave, dense matvec,
    fill, gather, norm2 / dot, axpby, block Jacobi -- each against NumPy / the oracle on device-resident arrays."""
    from pyamg_b200 import _engine as E
    from pyamg_b200.util import get_block_diag
    L, D = E.lib(), _DevMem()
    A, x0, b = _system(n=40, seed=31)
    n = A.shape[0]
    Ap, Aj, Ax = (D.up(A.indptr.astype(np.int32)), D.up(A.indices.astype(np.int32)), D.up(A.data))
    dx, db = D.up(x0), D.up(b)
    dy, dr = D.up(np.zeros(n)), D.up(np.zeros(n))
    P = D.ptr
    for lanes in (0, 4, 32):
        E.check(L.amgb_dev_csr_spmv(n, P(Ap), P(Aj), P(Ax), P(dx), P(dy), lanes, None))
        assert relerr(D.get(dy), A @ x0) < TOL
        parts, nrm = D.up(np.zeros(int(L.amgb_dev_partials_len(n, lanes)))), D.up(np.zeros(1))
        E.check(L.amgb_dev_csr_residual(n, P(Ap), P(Aj), P(Ax), P(dx), P(db), P(dr), P(parts), P(nrm), lanes, None))
        r = b - A @ x0
        assert relerr(D.get(dr), r) < TOL and D.get(nrm)[0] == pytest.approx(r @ r, rel=1e-13)
        dacc = D.up(b)
        E.check(L.amgb_dev_csr_spmv_add(n, P(Ap), P(Aj), P(Ax), P(dx), P(dacc), lanes, None))
        assert relerr(D.get(dacc), b + A @ x0) < TOL
        xo = x0.copy()
        oracle.jacobi(A, xo, b, omega=0.7)
        E.check(L.amgb_dev_csr_jacobi(n, P(Ap), P(Aj), P(Ax), P(dx), P(db), P(dy), P(dr), 0.7, lanes, None))
        assert relerr(D.get(dy), xo) < TOL and relerr(D.get(dr), r) < TOL      # r: residual of the INPUT iterate
    # one Gauss-Seidel "wave" over an independent set (rows 0, 1, ... with no mutual coupling are not guaranteed here:
    # use a single row list of one row at a time == the sequential sweep)
    xg, xo = D.up(x0), x0.copy()
    oracle.gauss_seidel(A, xo, b, sweep="forward")
    for i in range(n):
        E.check(L.amgb_dev_csr_gs_wave(1, i, None, P(Ap), P(Aj), P(Ax), P(xg), P(db), 1.0, 4, None))
    assert relerr(D.get(xg), xo) < TOL
    rows = D.up(np.array([5, 3], dtype=np.int32))                              # explicit (independent) row list
    xg, xo = D.up(x0), x0.copy()
    Aloc = A.tolil(); Aloc[5, 3] = 0; Aloc[3, 5] = 0; Aloc = sp.csr_array(Aloc.tocsr()); Aloc.eliminate_zeros()
    Bp, Bj, Bx = D.up(Aloc.indptr.astype(np.int32)), D.up(Aloc.indices.astype(np.int32)), D.up(Aloc.data)
    oracle.gauss_seidel_indexed(Aloc, xo, b, np.array([5, 3], dtype=np.int32))
    E.check(L.amgb_dev_csr_gs_wave(2, 0, P(rows), P(Bp), P(Bj), P(Bx), P(xg), P(db), 1.0, 8, None))
    assert relerr(D.get(xg), xo) < TOL
    # dense matvec, fill, gather
    M = np.random.default_rng(2).standard_normal((7, n))
    dM, d7 = D.up(M), D.up(np.zeros(7))
    E.check(L.amgb_dev_dense_matvec(7, n, P(dM), P(dx), P(d7), None))
    assert relerr(D.get(d7), M @ x0) < TOL
    E.check(L.amgb_dev_fill(P(dy), n, 2.5, None))
    assert np.array_equal(D.get(dy), np.full(n, 2.5))
    idx = np.random.default_rng(3).permutation(n).astype(np.int32)
    didx = D.up(idx)
    E.check(L.amgb_dev_gather(P(dx), P(didx), P(dy), n, None))
    assert np.array_equal(D.get(dy), x0[idx])
    # norm2 / dot, axpby
    scratch, out = D.up(np.zeros(int(L.amgb_dev_reduce_len()))), D.up(np.zeros(1))
    E.check(L.amgb_dev_dot(P(dx), P(db), n, P(scratch), P(out), None))
    assert D.get(out)[0] == pytest.approx(x0 @ b, rel=1e-13)
    E.check(L.amgb_dev_dot(P(dx), P(dx), n, P(scratch), P(out), None))
    assert D.get(out)[0] == pytest.approx(x0 @ x0, rel=1e-13)
    dz = D.up(b)
    E.check(L.amgb_dev_axpby(0.3, P(dx), -1.5, P(dz), n, None))
    assert relerr(D.get(dz), 0.3 * x0 - 1.5 * b) < TOL
    # block Jacobi on the point expansion of a BSR(3,3) operator
    Ab3, xb, bb = _system(n=12, seed=33, bs=3)
    Ab = Ab3.tobsr(blocksize=(3, 3))
    Dinv = get_block_diag(Ab, blocksize=3, inv_flag=True)
    Ac = sp.csr_array(Ab.tocsr())
    keep = []
    Mx = E.as_matrix(Ab, keep)                    # the engine's expansion keeps the BSR storage order: rebuild it here
    exp_ptr, exp_j, exp_x = [0], [], []
    for I in range(Ab.shape[0] // 3):
        for rr in range(3):
            for jj in range(Ab.indptr[I], Ab.indptr[I + 1]):
                for cc in range(3):
                    exp_j.append(Ab.indices[jj] * 3 + cc)
                    exp_x.append(Ab.data[jj, rr, cc])
            exp_ptr.append(len(exp_j))
    Ep, Ej, Ex = D.up(np.array(exp_ptr, np.int32)), D.up(np.array(exp_j, np.int32)), D.up(np.array(exp_x))
    dxb, dbb, dyb, dD = D.up(xb), D.up(bb), D.up(np.zeros_like(xb)), D.up(Dinv.reshape(-1))
    xo = xb.copy()
    oracle.block_jacobi(Ab, xo, bb, Dinv=Dinv, blocksize=3, omega=0.9)
    E.check(L.amgb_dev_block_jacobi(Ab.shape[0] // 3, 3, P(Ep), P(Ej), P(Ex), P(dxb), P(dbb), P(dD), P(dyb), 0.9, 4, None))
    assert relerr(D.get(dyb), xo) < TOL
    assert L.amgb_dev_block_jacobi(4, 3, P(Ep), P(Ej), P(Ex), P(dxb), P(dbb), P(dD), P(dxb), 0.9, 4, None) == E.EINVAL


# ------------------------------------------------------------------ randomised hierarchies
_FUZZ_ENVS = ({}, {"AMGB_TILE_MIN_NNZ": "0"}, {"AMGB_TILE_MIN_NNZ": "0", "AMGB_TILE_CFG": "0"},
              {"AMGB_NO_PERMUTE": "1", "AMGB_TILE_MIN_NNZ": "0", "AMGB_TILE_G": "8"})
_FUZZ_KEYS = ("AMGB_TILE_MIN_NNZ", "AMGB_TILE_CFG", "AMGB_NO_PERMUTE", "AMGB_TILE_G", "AMGB_TILE_FLAT", "AMGB_RESIDENT",
              "AMGB_RESIDENT_MAX_ROWS", "AMGB_TILE_PDL")


@pytest.mark.parametrize("case", range(6))
def test_random_two_level_hierarchies_with_long_rows_and_quirks(case, monkeypatch):
    random_hierarchy_check(case, monkeypatch, _FUZZ_ENVS)


def random_hierarchy_check(case, monkeypatch, envs):
    """Seeded random operators built to hit the corners of the tile builder and the kernels: rows longer than a tile
    (230-700 entries; geometries T = 224 and 512), empty-ish and short rows, a zero diagonal, unsorted column indices,
    random P (R = P^T), random pre/post smoothers incl. the wave-major and C|F layouts -- two V-cycles against the
    oracle through the lanes-per-row kernels, the TMA tile kernels on every operator, a second tile geometry and
    the un-permuted layout."""
    from pyamg_b200.relaxation.smoothing import change_smoothers
    rng = np.random.default_rng(1000 + case)
    n, nc = int(rng.integers(300, 1200)), int(rng.integers(20, 90))
    A = sp.random(n, n, density=float(rng.choice([0.02, 0.1, 0.4])),
                  random_state=np.random.RandomState(int(rng.integers(1 << 30))), format="lil")
    for i in rng.choice(n, size=max(1, n // 40), replace=False):
        cols = rng.choice(n, size=min(n, int(rng.integers(230, 700))), replace=False)
        A[i, cols] = rng.standard_normal(len(cols))
    A = sp.csr_array(A.tocsr())
    A = (A + A.T).tocsr()
    A = (A + sp.diags_array(np.asarray(np.abs(A).sum(axis=1)).ravel() + 1.0)).tocsr()
    if case % 2:
        A = A.tolil()
        A[3, 3] = 0.0
        A = sp.csr_array(A.tocsr())
        A.eliminate_zeros()
    A = sp.csr_array(A)
    A.sort_indices()
    for i in range(0, n, 7):                                       # unsorted indices, as RS coarse levels have
        s, e = A.indptr[i], A.indptr[i + 1]
        perm = rng.permutation(e - s)
        A.indices[s:e], A.data[s:e] = A.indices[s:e][perm], A.data[s:e][perm]
    P = sp.random(n, nc, density=min(1.0, 3.0 / nc), random_state=np.random.RandomState(int(rng.integers(1 << 30))),
                  format="csr")
    P = sp.csr_array(P + sp.csr_array((np.ones(n), (np.arange(n), np.arange(n) % nc)), shape=(n, nc)))

    def i32(M):
        M = sp.csr_array(M)
        M.indptr, M.indices = M.indptr.astype(np.int32), M.indices.astype(np.int32)
        return M
    R = i32(P.T.tocsr())
    A, P = i32(A), i32(P)
    Ac = i32(R @ A @ P)
    l0, l1 = pyamg_b200.MultilevelSolver.Level(), pyamg_b200.MultilevelSolver.Level()
    l0.A, l0.P, l0.R, l1.A = A, P, R, Ac
    l0.splitting = rng.random(n) < 0.5
    ml = pyamg_b200.MultilevelSolver([l0, l1])
    choices = [("jacobi", {"omega": 0.6, "withrho": False, "iterations": int(rng.integers(1, 4))}),
               ("gauss_seidel", {"sweep": str(rng.choice(["forward", "backward", "symmetric"]))}),
               ("gauss_seidel_indexed", {"sweep": "symmetric"}), ("sor", {"omega": 1.3, "sweep": "forward"}),
               ("cf_jacobi", {"omega": 0.5, "f_iterations": 2}), ("fc_jacobi", {"omega": 0.5}), None]
    change_smoothers(ml, choices[int(rng.integers(len(choices)))], choices[int(rng.integers(len(choices)))])
    b = rng.standard_normal(n)
    xo = oracle.Cycle(oracle.hierarchy_spec(ml), coarse_pinv=ml.coarse_solver.dense_operator(Ac)).solve(b, tol=0, maxiter=2)
    for env in envs:
        for k in _FUZZ_KEYS:
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        ml._invalidate()
        assert relerr(ml.solve(b, tol=0, maxiter=2), xo) < 1e-12, env


# ------------------------------------------------------------------ adoption of real reference solvers
# The hierarchies are the ones the REAL reference built (tests/golden/make_golden.py --reference-checks writes each
# with pyamg_b200.hierarchy_io.save_hierarchy, i.e. through the same reading of its smoothers and coarse solver that
# from_pyamg does, next to the reference's own ml.solve results on them).
ADOPT_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
ADOPT_FAMILIES = ["rs_default", "rs_cljp_direct_jacobi", "sa_default", "sa_elasticity_default", "sa_energy_chebyshev",
                  "rootnode", "pairwise", "adaptive_sa", "air", "sa_sor_none_lu", "rs_coarse_gauss_seidel",
                  "sa_richardson_splu", "sa_schwarz", "sa_strength_schwarz"]
VARIANT_FAMILIES = ["rs", "sa_elasticity", "air", "rootnode"]


def variant_runs(x0):
    """The ml.solve arguments of test_adopted_hierarchies_all_solve_variants_match_the_reference, in order."""
    return (dict(accel="cg", tol=1e-8, maxiter=8), dict(accel="gmres", tol=1e-8, maxiter=8),
            dict(accel="fgmres", tol=1e-8, maxiter=8, cycle="W"), dict(accel="bicgstab", tol=1e-8, maxiter=8),
            dict(accel="fgmres", cycle="AMLI", tol=1e-6, maxiter=4), dict(tol=1e-6, maxiter=30, x0=x0),
            dict(cycle="AMLI", tol=0, maxiter=2), dict(cycle="F", tol=0, maxiter=2, cycles_per_level=2))


@pytest.mark.parametrize("family", ADOPT_FAMILIES)
def test_from_pyamg_adopts_every_solver_family(family):
    """MultilevelSolver.from_pyamg on hierarchies the REAL reference built: three V-cycles and two W-cycles equal the
    reference's own ml.solve to 1e-12 -- classical RS (RS / CLJP splittings, direct interpolation), SA with default
    block Gauss-Seidel (scalar and elasticity), energy-minimising SA + Chebyshev, root-node, pairwise, adaptive SA,
    AIR, SOR on BSR coarse levels (omega ignored there, as in the reference), None smoothers, lu / splu / relaxation
    coarse solvers."""
    from pyamg_b200.hierarchy_io import load_hierarchy
    ref, ex = load_hierarchy(os.path.join(ADOPT_DIR, f"adopt_{family}.npz"))
    gpu = pyamg_b200.MultilevelSolver.from_pyamg(ref)
    assert relerr(gpu.solve(ex["b"], tol=0, maxiter=3), ex["x_V3"]) < TOL
    assert relerr(gpu.solve(ex["b"], tol=0, maxiter=2, cycle="W"), ex["x_W2"]) < TOL


@pytest.mark.parametrize("family", VARIANT_FAMILIES)
def test_adopted_hierarchies_all_solve_variants_match_the_reference(family):
    """On hierarchies adopted from the real reference: CG / GMRES / FGMRES / BiCGStab acceleration, FGMRES + AMLI,
    tolerance stop from x0, AMLI and F(cycles_per_level=2) cycles -- same iterates, iteration counts and info flags
    as the reference's own ml.solve."""
    from pyamg_b200.hierarchy_io import load_hierarchy
    ref, ex = load_hierarchy(os.path.join(ADOPT_DIR, f"variants_{family}.npz"))
    gpu = pyamg_b200.MultilevelSolver.from_pyamg(ref)
    for k, kw in enumerate(variant_runs(ex["x0"])):
        if family == "air" and kw.get("accel") == "cg":
            continue                                  # nonsymmetric operator
        rg = []
        xg, ig = gpu.solve(ex["b"], residuals=rg, return_info=True, **kw)
        assert (int(ex["info"][k]), int(ex["nres"][k])) == (ig, len(rg)), kw
        assert relerr(xg, ex[f"x_{k}"]) < 1e-9, kw


# ------------------------------------------------------------------ CF / FC block Jacobi (AIR on block systems)
@pytest.mark.parametrize("bs", [2, 3])
def test_cf_fc_block_jacobi_match_oracle_and_compiled_reference(bs):
    """relaxation.cf_block_jacobi / fc_block_jacobi (relaxation.py:1271-1412 -> block_jacobi_indexed,
    relaxation.h:1113-1172): listed block rows relaxed from a snapshot, C then F or F then C."""
    from pyamg_b200.util import get_block_diag
    rng = np.random.default_rng(40 + bs)
    nb = 15
    n = nb * bs
    A = sp.random(n, n, density=0.3, random_state=np.random.RandomState(bs), format="csr")
    A = (A + A.T + sp.eye(n) * 8).tobsr(blocksize=(bs, bs))
    Dinv = get_block_diag(A, blocksize=bs, inv_flag=True)
    split = rng.random(nb) < 0.5
    C, F = np.where(split)[0], np.where(~split)[0]
    x0, b = rng.standard_normal(n), rng.standard_normal(n)
    kern = "ref" if oracle.have_ref() else "oracle"
    for fg, fo in ((gpu_relax.cf_block_jacobi, oracle.cf_block_jacobi), (gpu_relax.fc_block_jacobi, oracle.fc_block_jacobi)):
        for kw in ({}, {"iterations": 2, "f_iterations": 2, "c_iterations": 0, "omega": 0.7}):
            xg, xo = x0.copy(), x0.copy()
            fg(A, xg, b, C, F, Dinv=Dinv, blocksize=bs, **kw)
            fo(A, xo, b, C, F, Dinv=Dinv, blocksize=bs, kernels=kern, **kw)
            assert relerr(xg, xo) < TOL


def test_block_cf_jacobi_in_a_cycle_and_through_hierarchy_io(tmp_path):
    """A two-level block hierarchy with fc_block_jacobi (what air_solver installs on BSR operators): engine vs oracle,
    also after a save / load round trip of the descriptor (Cpts, Fpts, Dinv, blocksize)."""
    from pyamg_b200.hierarchy_io import save_hierarchy, load_hierarchy
    from pyamg_b200.relaxation.smoothing import change_smoothers
    rng = np.random.default_rng(77)
    bs, nb, ncb = 2, 30, 9
    n, nc = nb * bs, ncb * bs
    A = sp.random(n, n, density=0.15, random_state=np.random.RandomState(5), format="csr")
    A = sp.bsr_array((A + A.T + sp.eye(n) * 6).tobsr(blocksize=(bs, bs)))
    P = sp.bsr_array(sp.kron(sp.csr_array((np.ones(nb), (np.arange(nb), np.arange(nb) % ncb)), shape=(nb, ncb)),
                             np.eye(bs)).tobsr(blocksize=(bs, bs)))
    R = sp.bsr_array(P.T.tobsr(blocksize=(bs, bs)))
    def i32(M):
        M.indptr, M.indices = M.indptr.astype(np.int32), M.indices.astype(np.int32)
        return M
    l0, l1 = pyamg_b200.MultilevelSolver.Level(), pyamg_b200.MultilevelSolver.Level()
    l0.A, l0.P, l0.R = i32(A), i32(P), i32(R)
    l1.A = i32(sp.bsr_array((R @ A @ P).tobsr(blocksize=(bs, bs))))
    l0.splitting = rng.random(nb) < 0.4
    ml = pyamg_b200.MultilevelSolver([l0, l1])
    change_smoothers(ml, ("cf_block_jacobi", {"omega": 0.8}), ("fc_block_jacobi", {"omega": 0.8, "f_iterations": 2}))
    b = rng.standard_normal(n)
    xo = oracle.Cycle(oracle.hierarchy_spec(ml), coarse_pinv=ml.coarse_solver.dense_operator(l1.A)).solve(b, tol=0, maxiter=3)
    assert relerr(ml.solve(b, tol=0, maxiter=3), xo) < TOL
    p = str(tmp_path / "h.npz")
    save_hierarchy(p, ml)
    ml2, _ = load_hierarchy(p)
    assert ml2.levels[0].postsmoother.__name__ == "fc_block_jacobi"
    assert relerr(ml2.solve(b, tol=0, maxiter=3), xo) < TOL


# ------------------------------------------------------------------ normal-equation smoothers (Kaczmarz family)
def test_normal_equation_smoothers_match_oracle_and_compiled_reference():
    """relaxation.jacobi_ne / gauss_seidel_ne / gauss_seidel_nr (relaxation.py:734-999 -> relaxation.h:579-713): the
    row / column projections run as conflict waves (rows of a wave share no column), which reproduces the sequential
    sweep; forward, backward, symmetric, several iterations, omega != 1."""
    rng = np.random.default_rng(0)
    n = 60
    A = sp.random(n, n, density=0.15, random_state=np.random.RandomState(1), format="csr")
    A = sp.csr_array(A + sp.eye(n) * 3)
    A.indptr, A.indices = A.indptr.astype(np.int32), A.indices.astype(np.int32)
    x0, b = rng.standard_normal(n), rng.standard_normal(n)
    kern = "ref" if oracle.have_ref() else "oracle"
    for name, kw in (("jacobi_ne", dict(iterations=2, omega=0.3)),
                     ("gauss_seidel_ne", dict(sweep="symmetric", iterations=2, omega=0.9)),
                     ("gauss_seidel_ne", dict(sweep="backward")),
                     ("gauss_seidel_nr", dict(sweep="forward", iterations=2, omega=1.1)),
                     ("gauss_seidel_nr", dict(sweep="symmetric")),
                     ("gauss_seidel_nr", dict(sweep="backward", iterations=3))):
        xo, xg = x0.copy(), x0.copy()
        getattr(oracle, name)(sp.csc_array(A) if name.endswith("nr") else A.copy(), xo, b, kernels=kern, **kw)
        getattr(gpu_relax, name)(A.copy(), xg, b, **kw)
        assert relerr(xg, xo) < TOL, (name, kw)
    with pytest.raises(ValueError):
        gpu_relax.gauss_seidel_ne(A, x0.copy(), b, sweep="diagonal")


def test_normal_equation_smoothers_from_the_factory():
    from pyamg_b200.classical import ruge_stuben_solver
    from pyamg_b200.gallery import poisson
    np.random.seed(11)
    ml = ruge_stuben_solver(poisson((18, 18)), presmoother=("gauss_seidel_nr", {"sweep": "symmetric"}),
                            postsmoother=("jacobi_ne", {"omega": 1.0, "iterations": 2}))
    b = np.random.default_rng(12).random(ml.levels[0].A.shape[0])
    cyc = oracle.Cycle(oracle.hierarchy_spec(ml), coarse_pinv=ml.coarse_solver.dense_operator(ml.levels[-1].A))
    assert relerr(ml.solve(b, tol=0, maxiter=3), cyc.solve(b, tol=0, maxiter=3)) < TOL
    assert ml.levels[0].presmoother.__name__ == "gauss_seidel_nr"


# ------------------------------------------------------------------ overlapping multiplicative Schwarz
def _cover(n, rng, max_m):
    """A random overlapping cover of range(n): subdomains of 1..max_m distinct rows, every row in at least one."""
    subs = [rng.choice(n, size=int(rng.integers(1, max_m + 1)), replace=False) for _ in range(n // 3)]
    missing = np.setdiff1d(np.arange(n), np.concatenate(subs))
    subs += [missing[k:k + 3] for k in range(0, len(missing), 3)]
    ptr = np.zeros(len(subs) + 1, dtype=np.int32)
    ptr[1:] = np.cumsum([len(u) for u in subs])
    return np.concatenate(subs).astype(np.int32), ptr


def test_schwarz_matches_oracle_and_compiled_reference():
    """relaxation.schwarz (relaxation.py:157-262 -> overlapping_schwarz_csr, relaxation.h:818-880): subdomains that
    touch (a row of one is a row or a column neighbour of the other) keep their sequential order, the others share a
    wave -- bit for bit the sequential sweep.  Default subdomains (sparsity patterns), random overlapping covers with
    subdomains of 1 row and of more rows than a warp has lanes, the three sweeps, several iterations."""
    from pyamg_b200.gallery import poisson
    rng = np.random.default_rng(3)
    kern = "ref" if oracle.have_ref() else "oracle"
    cases = []
    for A in (poisson((9, 8), format="csr"), poisson((4, 5, 3), format="csr"),
              sp.random(70, 70, density=0.08, random_state=np.random.RandomState(5), format="csr") + 4 * sp.eye(70)):
        A = sp.csr_array(A)
        A.sort_indices()
        A.indptr, A.indices = A.indptr.astype(np.int32), A.indices.astype(np.int32)
        cases.append((A, None, None))
        cases.append((A, *_cover(A.shape[0], rng, 6)))
    cases.append((cases[-1][0], *_cover(70, rng, 45)))
    for A, sub, ptr in cases:
        n = A.shape[0]
        x0, b = rng.standard_normal(n), rng.standard_normal(n)
        for kw in (dict(), dict(sweep="backward", iterations=2), dict(sweep="symmetric", iterations=2)):
            xo, xg = x0.copy(), x0.copy()
            oracle.schwarz(A.copy(), xo, b, subdomain=sub, subdomain_ptr=ptr, kernels=kern, **kw)
            gpu_relax.schwarz(A.copy(), xg, b, subdomain=sub, subdomain_ptr=ptr, **kw)
            assert relerr(xg, xo) < TOL, (n, kw)            # (bit-equal without FMA contraction: the emulator)
    with pytest.raises(ValueError):
        gpu_relax.schwarz(A, x0.copy(), b, sweep="diagonal")
    with pytest.raises(NotImplementedError):          # a row twice in one subdomain: two lanes would update it at once
        gpu_relax.schwarz(A.copy(), x0.copy(), b, subdomain=np.array([0, 1, 0], dtype=np.int32),
                          subdomain_ptr=np.array([0, 3], dtype=np.int32))


def test_schwarz_smoothers_from_the_factory():
    """('schwarz', ...) and ('strength_based_schwarz', ...) through the setup registry (smoothing.py:509-548) on an SA
    hierarchy whose coarse levels are BSR."""
    from pyamg_b200.aggregation import smoothed_aggregation_solver
    from pyamg_b200.gallery import poisson
    np.random.seed(13)
    ml = smoothed_aggregation_solver(poisson((16, 16), format="csr"), max_coarse=15,
                                     presmoother=("schwarz", {"sweep": "forward", "iterations": 2}),
                                     postsmoother=("strength_based_schwarz", {"sweep": "symmetric"}))
    assert len(ml.levels) >= 3 and ml.levels[0].presmoother.__name__ == "schwarz"
    b = np.random.default_rng(14).random(ml.levels[0].A.shape[0])
    cyc = oracle.Cycle(oracle.hierarchy_spec(ml), coarse_pinv=ml.coarse_solver.dense_operator(ml.levels[-1].A))
    for cycle in ("V", "W"):
        assert relerr(ml.solve(b, tol=0, maxiter=3, cycle=cycle), cyc.solve(b, tol=0, maxiter=3, cycle=cycle)) < TOL
    res = []
    ml.solve(b, tol=1e-8, residuals=res)
    assert res[-1] < 1e-8 * np.linalg.norm(b) and len(res) < 20


@pytest.mark.gpu
def test_device_mis_colouring_equals_the_sequential_reference():
    """SURVEY 8(f)-4: pyamg.graph.vertex_coloring(G, 'MIS') (amg_core/graph.h:218-235) computed on the device as a
    wavefront of first-fit decisions equals the sequential routine vertex by vertex -- host restatement on every
    level of a Ruge-Stuben hierarchy and on random graphs, the REAL reference where it is importable."""
    import scipy.sparse as sp
    from pyamg_b200.classical import ruge_stuben_solver
    from pyamg_b200.gallery import poisson
    from pyamg_b200.graph import vertex_coloring
    graphs = [sp.csr_array(lvl.A) for lvl in ruge_stuben_solver(poisson((14, 14, 14))).levels]
    graphs += [sp.csr_array(poisson((40, 40)))]
    for seed in (1, 2):
        R = sp.random(700, 700, 0.02, random_state=seed)
        graphs.append((R + R.T).tocsr())
    for G in graphs:
        host = vertex_coloring(G, "MIS", where="host")
        dev = vertex_coloring(G, "MIS", where="gpu")
        assert np.array_equal(host, dev)
        G2 = G.tocsr()
        rows = np.repeat(np.arange(G2.shape[0]), np.diff(G2.indptr))
        off = rows != G2.indices
        assert not np.any(dev[rows[off]] == dev[G2.indices[off]])
    try:
        from pyamg.graph import vertex_coloring as reference_coloring
    except ImportError:
        return
    for G in graphs:
        assert np.array_equal(reference_coloring(G, "MIS"), vertex_coloring(G, "MIS", where="gpu"))
