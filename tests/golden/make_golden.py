"""Generate the golden fixtures under tests/golden/ by running the REAL reference.

Run in the build container only (the GPU box has no /root/reference):

    # 1. build the reference in a scratch dir (SURVEY.md 8(c) recipe; nothing is copied here)
    D=/tmp/pyamg_ref; mkdir -p $D; cp -r /root/reference/pyamg $D/pyamg; cd $D/pyamg/amg_core
    for h in air evolution_strength graph krylov linalg relaxation ruge_stuben smoothed_aggregation; do
      g++ -O2 -std=c++11 -ftemplate-depth=2048 -shared -fPIC -fvisibility=hidden \
          $(python3 -m pybind11 --includes) ${h}_bind.cpp \
          -o ${h}$(python3 -c "import sysconfig;print(sysconfig.get_config_var('EXT_SUFFIX'))") & done; wait
    mkdir $D/pyamg-0.0.0.dist-info
    printf 'Metadata-Version: 2.1\nName: pyamg\nVersion: 0.0.0+oracle\n' > $D/pyamg-0.0.0.dist-info/METADATA
    # 2. generate
    cd /root/repo && PYTHONPATH=/tmp/pyamg_ref python tests/golden/make_golden.py
    # 3. the goldens of the tests that compare with the reference directly (tests/golden/reference/; they also
    #    need oracle/_ref/libamg_ref.so, which build() compiles where the reference sources are present)
    PYTHONPATH=<the reference build of step 1> python tests/golden/make_golden.py --reference-checks

Every fixture is one .npz written by pyamg_b200.hierarchy_io.save_hierarchy: the hierarchy the
reference built (operators, smoother closures' parameters, cached coarse pinv) plus, as extra
arrays, the rhs ``b``, the reference's ``x_ref = ml.solve(b, tol=0, maxiter=N)``, its residual
history, W/F/AMLI-cycle results, and single-sweep outputs of the reference's own relaxation routines and
SciPy matvecs on level 0 (``k_*``).  Configs are the five BASELINE.json families at sizes the CPU
suite runs in seconds.  rhs seed = 20260922 (SURVEY.md 8(d)).
"""
import os
import sys

import numpy as np

import pyamg
from pyamg.gallery import poisson, stencil_grid, linear_elasticity
from pyamg.gallery.diffusion import diffusion_stencil_2d
from pyamg.graph import vertex_coloring
from pyamg.relaxation import relaxation as ref_relax
from functools import partial, update_wrapper

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from pyamg_b200.hierarchy_io import save_hierarchy  # noqa: E402

SEED = 20260922
NCYC = 6


def install_multicolor_gs(ml, sweep="symmetric"):
    """SURVEY.md 8(d) config 3: replace every level's smoothers by gauss_seidel_indexed over the
    MIS-colour-sorted row list (the reference's only expression of multi-colour GS)."""
    for lvl in ml.levels[:-1]:
        c = vertex_coloring(lvl.A, "MIS")
        order = np.argsort(c, kind="stable").astype(np.int32)
        for which in ("presmoother", "postsmoother"):
            sm = partial(ref_relax.gauss_seidel_indexed, indices=order, iterations=1, sweep=sweep)
            update_wrapper(sm, ref_relax.gauss_seidel_indexed)
            setattr(lvl, which, sm)


def kernel_goldens(ml, rng):
    """Single-sweep outputs of the reference's native kernels on level 0."""
    lvl = ml.levels[0]
    A = lvl.A
    n = A.shape[0]
    x = rng.random(n)
    b = rng.random(n)
    out = {"k_x": x, "k_b": b, "k_Ax": A @ x, "k_Rx": lvl.R @ x,
           "k_Pxc": lvl.P @ rng.random(lvl.P.shape[1])}
    out["k_xc"] = None
    xc = rng.random(lvl.P.shape[1])
    out["k_xc"] = xc
    out["k_Pxc"] = lvl.P @ xc
    for which in ("presmoother", "postsmoother"):
        y = x.copy()
        getattr(lvl, which)(A, y, b)
        out["k_" + which] = y
    Acsr = A.tocsr()
    y = x.copy()
    ref_relax.jacobi(Acsr, y, b, iterations=1, omega=0.7)
    out["k_jacobi_w07"] = y
    y = x.copy()
    ref_relax.gauss_seidel(Acsr, y, b, iterations=1, sweep="symmetric")
    out["k_gs_symmetric"] = y
    y = x.copy()
    ref_relax.gauss_seidel(Acsr, y, b, iterations=2, sweep="backward")
    out["k_gs_backward2"] = y
    y = x.copy()
    ref_relax.sor(Acsr, y, b, omega=1.3, iterations=1, sweep="forward")
    out["k_sor_13"] = y
    return out


ONLY = None               # --only <name>: write just this configuration's files
KRYLOV_ONLY = False       # --krylov: rebuild the same hierarchies, write only the GMRES / FGMRES goldens


def emit_krylov(name, ml, b, x0):
    """Supplementary goldens tests/golden/krylov/<name>.npz: ml.solve(accel='gmres' | 'fgmres') of the real
    reference (pyamg.krylov.gmres = Householder GMRES, left-preconditioned; pyamg.krylov.fgmres, right-
    preconditioned) with the cycle as preconditioner."""
    import warnings
    out = {}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for tag, kw in (("gmres", dict(tol=1e-10, maxiter=12, accel="gmres")),
                        ("gmresW", dict(x0=x0, tol=1e-3, maxiter=25, accel="gmres", cycle="W")),
                        ("fgmres", dict(tol=1e-10, maxiter=12, accel="fgmres")),
                        ("fgmresF", dict(x0=x0, tol=1e-4, maxiter=25, accel="fgmres", cycle="F")),
                        ("fgmresAMLI", dict(tol=1e-8, maxiter=5, accel="fgmres", cycle="AMLI")),
                        ("bicgstab", dict(tol=1e-10, maxiter=8, accel="bicgstab")),
                        ("bicgstabW", dict(x0=x0, tol=1e-4, maxiter=20, accel="bicgstab", cycle="W"))):
            res = []
            x, info = ml.solve(b, residuals=res, return_info=True, **kw)
            out["x_ref_" + tag] = x
            out["residuals_" + tag] = np.array(res)
            out["info_" + tag] = np.array([info])
    os.makedirs(os.path.join(HERE, "krylov"), exist_ok=True)
    np.savez_compressed(os.path.join(HERE, "krylov", name + ".npz"), **out)
    print(f"krylov/{name}: " + ", ".join(f"{t}: {len(out['residuals_' + t]) - 1} its info={int(out['info_' + t][0])}"
                                       for t in ("gmres", "gmresW", "fgmres", "fgmresF", "fgmresAMLI", "bicgstab", "bicgstabW")))


def emit(name, ml, extra_kw=None, ncyc=NCYC, cg_anyway=True):
    if ONLY is not None and name != ONLY:
        return
    rng = np.random.default_rng(SEED)
    n = ml.levels[0].A.shape[0]
    b = rng.random(n)
    extra = {"b": b}
    res = []
    extra["x_ref"] = ml.solve(b, tol=0, maxiter=ncyc, residuals=res)   # also caches coarse pinv
    extra["residuals"] = np.array(res)
    if KRYLOV_ONLY:
        stored = np.load(os.path.join(HERE, name + ".npz"))
        assert np.array_equal(stored["X_x_ref"], extra["x_ref"]), "rebuilt hierarchy differs from the stored golden"
        rng2 = np.random.default_rng(SEED)
        rng2.random(n)
        emit_krylov(name, ml, b, stored["X_x0"])
        return
    extra["x_ref_W"] = ml.solve(b, tol=0, maxiter=2, cycle="W")
    extra["x_ref_F"] = ml.solve(b, tol=0, maxiter=2, cycle="F")
    res = []
    extra["x_ref_AMLI"] = ml.solve(b, tol=0, maxiter=3, cycle="AMLI", residuals=res)
    extra["residuals_AMLI"] = np.array(res)
    x0 = rng.random(n)
    res = []
    xt, info = ml.solve(b, x0=x0, tol=1e-6, maxiter=50, residuals=res, return_info=True)
    extra.update({"x0": x0, "x_ref_tol": xt, "residuals_tol": np.array(res),
                  "info_tol": np.array([info])})
    if ml.symmetric_smoothing or cg_anyway:
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            res = []
            xc, info = ml.solve(b, tol=1e-10, maxiter=10, accel="cg", residuals=res, return_info=True)
            extra.update({"x_ref_cg": xc, "residuals_cg": np.array(res), "info_cg": np.array([info])})
            res = []
            xc, info = ml.solve(b, x0=x0, tol=1e-3, maxiter=30, accel="cg", cycle="W", residuals=res, return_info=True)
            extra.update({"x_ref_cgW": xc, "residuals_cgW": np.array(res), "info_cgW": np.array([info])})
    extra.update(kernel_goldens(ml, rng))
    if extra_kw:
        extra.update(extra_kw)
    path = os.path.join(HERE, name + ".npz")
    save_hierarchy(path, ml, extra=extra)
    sizes = [lv.A.shape[0] for lv in ml.levels]
    print(f"{name}: levels={sizes} fmt={[lv.A.format for lv in ml.levels]} "
          f"res {extra['residuals'][0]:.3e}->{extra['residuals'][-1]:.3e} "
          f"tol-its={len(res) - 1} info={info}  {os.path.getsize(path) / 1024:.0f} KB")


def main():
    # cfg1 family: RS, default symmetric (lexicographic) Gauss-Seidel
    np.random.seed(SEED)
    A = poisson((30, 30), format="csr")
    emit("cfg1_rs_gs_poisson2d", pyamg.ruge_stuben_solver(A))

    # cfg2 family: SA + weighted Jacobi (P, R and coarse A are BSR(1,1))
    np.random.seed(SEED)
    A = poisson((40, 40), format="csr")
    sm = ("jacobi", {"omega": 4.0 / 3.0})
    emit("cfg2_sa_jacobi_poisson2d", pyamg.smoothed_aggregation_solver(A, presmoother=sm, postsmoother=sm))

    # cfg3 family: RS on 3D Poisson with multi-colour GS (gauss_seidel_indexed over MIS colours)
    np.random.seed(SEED)
    A = poisson((12, 12, 12), format="csr")
    ml = pyamg.ruge_stuben_solver(A)
    install_multicolor_gs(ml)
    emit("cfg3_rs_mcgs_poisson3d", ml)

    # cfg4 family: anisotropic diffusion, SA (evolution strength: the symmetric default diverges,
    # SURVEY.md 8(d)-4) + Jacobi, two sweeps pre / one post to exercise the ping-pong parity
    np.random.seed(SEED)
    S = diffusion_stencil_2d(epsilon=0.001, theta=np.pi / 6, type="FE")
    A = stencil_grid(S, (48, 48), format="csr")
    ml = pyamg.smoothed_aggregation_solver(A, strength=("evolution", {}),
                                           presmoother=("jacobi", {"omega": 4.0 / 3.0, "iterations": 2}),
                                           postsmoother=("jacobi", {"omega": 4.0 / 3.0}))
    emit("cfg4_sa_jacobi_aniso2d", ml)

    # cfg5 family: linear elasticity BSR(2,2) -> (3,3), SA with rigid-body modes, block Jacobi
    np.random.seed(SEED)
    A, B = linear_elasticity((14, 14))
    ml = pyamg.smoothed_aggregation_solver(A, B=B, presmoother="block_jacobi", postsmoother="block_jacobi")
    emit("cfg5_sa_bjacobi_elasticity", ml)

    # extra: RS with forward/backward SOR-free GS pair and None post-smoother (descriptor coverage)
    np.random.seed(SEED)
    A = poisson((9, 9, 9), format="csr")
    ml = pyamg.ruge_stuben_solver(A, presmoother=("gauss_seidel", {"sweep": "forward", "iterations": 2}),
                                  postsmoother=None, max_coarse=5)
    emit("cfg6_rs_gsfwd_none_poisson3d", ml)


def main_widening():
    """SURVEY.md 8(f)-2 smoothers: polynomial (chebyshev / richardson), CF / FC Jacobi, AIR's hierarchy
    (R != P^T, no pre-smoother, fc_jacobi post-smoother) and block Gauss-Seidel (the SA default)."""
    from pyamg.gallery import advection_2d

    # cfg7: SA + Chebyshev (degree 3) pre, two Richardson sweeps post -- closures, not partials
    np.random.seed(SEED)
    A = poisson((36, 36), format="csr")
    ml = pyamg.smoothed_aggregation_solver(A, presmoother=("chebyshev", {"degree": 3, "iterations": 1}),
                                           postsmoother=("richardson", {"iterations": 2}))
    emit("cfg7_sa_cheby_richardson_poisson2d", ml)

    # cfg8: RS + CF Jacobi pre / FC Jacobi post (two F sweeps), damped
    np.random.seed(SEED)
    A = poisson((11, 11, 11), format="csr")
    ml = pyamg.ruge_stuben_solver(A, presmoother=("cf_jacobi", {"omega": 0.8, "f_iterations": 2}),
                                  postsmoother=("fc_jacobi", {"omega": 0.8, "c_iterations": 2, "iterations": 2}))
    emit("cfg8_rs_cfjacobi_poisson3d", ml)

    # cfg9: AIR on 2-D upwind advection (nonsymmetric; R = approximate ideal restriction != P^T)
    np.random.seed(SEED)
    A, _rhs = advection_2d((30, 30), theta=np.pi / 5.0)
    ml = pyamg.air_solver(A.tocsr())
    emit("cfg9_air_fcjacobi_advection2d", ml, cg_anyway=False)

    # cfg11: relaxation as the coarsest-level solver (multilevel.py:764-781): 4 symmetric Gauss-Seidel sweeps on a
    # 57-unknown coarsest level instead of the pseudo-inverse
    np.random.seed(SEED)
    A = poisson((30, 30), format="csr")
    ml = pyamg.ruge_stuben_solver(A, max_coarse=60, coarse_solver=("gauss_seidel", {"iterations": 4, "sweep": "symmetric"}))
    emit("cfg11_rs_gs_coarse_relaxation", ml)

    # cfg12: SOR on a smoothed-aggregation hierarchy: level 0 is CSR (in-sweep omega, sor_gauss_seidel), the coarse
    # levels are BSR(1,1) where the reference's gauss_seidel ignores omega (relaxation.py:343-346)
    np.random.seed(SEED)
    A = poisson((28, 28), format="csr")
    ml = pyamg.smoothed_aggregation_solver(A, presmoother=("sor", {"omega": 1.2, "sweep": "forward"}),
                                           postsmoother=("sor", {"omega": 1.2, "sweep": "backward", "iterations": 2}))
    emit("cfg12_sa_sor_poisson2d", ml)

    # cfg13: normal-equation smoothers (closures; parameters in cell variables): Gauss-Seidel NR pre, Gauss-Seidel NE
    # post on a nonsymmetric operator (upwind advection + diffusion)
    np.random.seed(SEED)
    Adv = advection_2d((22, 22), theta=np.pi / 7.0)[0]
    m = int(round(np.sqrt(Adv.shape[0])))
    A = (Adv + 0.3 * poisson((m, m))).tocsr()
    ml = pyamg.ruge_stuben_solver(A, presmoother=("gauss_seidel_nr", {"sweep": "symmetric"}),
                                  postsmoother=("gauss_seidel_ne", {"sweep": "backward", "omega": 0.9, "iterations": 2}))
    emit("cfg13_rs_gsnr_gsne_advdiff2d", ml, cg_anyway=False)

    # cfg14: Jacobi NE (omega / rho(D^-1 A)^2 computed by the reference, read back from the closure) on SA
    np.random.seed(SEED)
    A = poisson((26, 26), format="csr")
    ml = pyamg.smoothed_aggregation_solver(A, presmoother=("jacobi_ne", {"omega": 4.0 / 3.0}),
                                           postsmoother=("jacobi_ne", {"omega": 4.0 / 3.0, "iterations": 2}))
    emit("cfg14_sa_jacobine_poisson2d", ml)

    # cfg15: overlapping Schwarz with the default subdomains (the rows' sparsity patterns); subdomains and block
    # inverses live in the closure's cells
    np.random.seed(SEED)
    A = stencil_grid(diffusion_stencil_2d(epsilon=0.05, theta=np.pi / 5.0, type="FE"), (18, 18), format="csr")
    ml = pyamg.smoothed_aggregation_solver(A, strength=("symmetric", {"theta": 0.1}),
                                           presmoother=("schwarz", {"sweep": "symmetric"}),
                                           postsmoother=("schwarz", {"sweep": "backward", "iterations": 2}),
                                           max_coarse=20)
    emit("cfg15_sa_schwarz_aniso2d", ml)

    # cfg16: strength-based Schwarz (subdomains = rows of the strength matrix, which keep=True leaves on the levels;
    # the reference rebuilds the block inverses on every application).  Pre and post share the subdomains: with
    # NumPy 2 the reference's parameter cache (relaxation.py:1036-1041) cannot compare two different sets.
    np.random.seed(SEED)
    A = A.copy()                                    # cfg15 left its parameter cache on the matrix object
    ml = pyamg.smoothed_aggregation_solver(A, strength=("symmetric", {"theta": 0.1}),
                                           presmoother=("strength_based_schwarz", {"sweep": "forward"}),
                                           postsmoother=("strength_based_schwarz", {"sweep": "backward", "iterations": 2}),
                                           max_coarse=20, keep=True)
    emit("cfg16_sa_strength_schwarz_aniso2d", ml)

    # cfg10: linear elasticity with the reference's DEFAULT SA smoothers (symmetric block Gauss-Seidel)
    np.random.seed(SEED)
    A, B = linear_elasticity((12, 12))
    ml = pyamg.smoothed_aggregation_solver(A, B=B)
    emit("cfg10_sa_bgs_elasticity", ml)


REFERENCE_DIR = os.path.join(HERE, "reference")


def adopt_builders():
    """The reference solvers of test_from_pyamg_adopts_every_solver_family (np.random.seed(1) before each)."""
    from pyamg.gallery import advection_2d
    A2, A3 = poisson((24, 24), format="csr"), poisson((9, 9, 9), format="csr")
    return {
        "rs_default": lambda: pyamg.ruge_stuben_solver(A2),
        "rs_cljp_direct_jacobi": lambda: pyamg.ruge_stuben_solver(
            A2, CF="CLJP", interpolation="direct", presmoother=("jacobi", {"omega": 0.8}), postsmoother=("jacobi", {"omega": 0.8})),
        "sa_default": lambda: pyamg.smoothed_aggregation_solver(A3),
        "sa_elasticity_default": lambda: pyamg.smoothed_aggregation_solver(linear_elasticity((10, 10))[0],
                                                                        B=linear_elasticity((10, 10))[1]),
        "sa_energy_chebyshev": lambda: pyamg.smoothed_aggregation_solver(
            stencil_grid(diffusion_stencil_2d(0.01, np.pi / 4, "FD"), (24, 24), format="csr"), smooth="energy",
            presmoother=("chebyshev", {"degree": 2}), postsmoother=("chebyshev", {"degree": 2})),
        "rootnode": lambda: pyamg.rootnode_solver(A2),
        "pairwise": lambda: pyamg.pairwise_solver(A2),
        "adaptive_sa": lambda: pyamg.aggregation.adaptive_sa_solver(A2, num_candidates=1)[0],
        "air": lambda: pyamg.air_solver(advection_2d((20, 20))[0].tocsr()),
        "sa_sor_none_lu": lambda: pyamg.smoothed_aggregation_solver(A2, presmoother=("sor", {"omega": 1.2}),
                                                                   postsmoother=None, coarse_solver="lu"),
        "rs_coarse_gauss_seidel": lambda: pyamg.ruge_stuben_solver(A2, max_coarse=50,
                                                                   coarse_solver=("gauss_seidel", {"iterations": 3})),
        "sa_richardson_splu": lambda: pyamg.smoothed_aggregation_solver(A2, presmoother="richardson",
                                                                       postsmoother="richardson", coarse_solver="splu"),
        "sa_schwarz": lambda: pyamg.smoothed_aggregation_solver(A2.copy(), presmoother="schwarz", postsmoother="schwarz"),
        "sa_strength_schwarz": lambda: pyamg.smoothed_aggregation_solver(
            A2.copy(), strength=("symmetric", {"theta": 0.3}), keep=True, presmoother="strength_based_schwarz",
            postsmoother=("strength_based_schwarz", {"sweep": "forward"})),
    }


def variant_builders():
    """The reference solvers of test_adopted_hierarchies_all_solve_variants_match_the_reference."""
    from pyamg.gallery import advection_2d
    A2 = poisson((20, 20), format="csr")
    return {"rs": lambda: pyamg.ruge_stuben_solver(A2),
            "sa_elasticity": lambda: pyamg.smoothed_aggregation_solver(linear_elasticity((8, 8))[0],
                                                                       B=linear_elasticity((8, 8))[1]),
            "air": lambda: pyamg.air_solver(advection_2d((16, 16))[0].tocsr()),
            "rootnode": lambda: pyamg.rootnode_solver(A2)}


def main_reference_checks():
    """Goldens of the tests that compare with the reference directly, under tests/golden/reference/:
    adopt_<family>.npz / variants_<family>.npz (hierarchies the reference built + its ml.solve results),
    mis_colouring.npz (its 'MIS' colours) and compiled_kernels.json (digests of its compiled relaxation.h kernels,
    which needs oracle/_ref/libamg_ref.so)."""
    import json
    import warnings
    import scipy.sparse as sp
    sys.path.insert(0, os.path.dirname(HERE))
    import oracle
    from pyamg_b200.hierarchy_io import load_hierarchy
    from test_oracle import kernel_digests
    from test_setup import mis_graphs
    from test_zz_gpu_widening import ADOPT_FAMILIES, VARIANT_FAMILIES, variant_runs
    os.makedirs(REFERENCE_DIR, exist_ok=True)

    def load_golden(name):
        return load_hierarchy(os.path.join(HERE, name + ".npz"))

    builders = adopt_builders()
    assert sorted(builders) == sorted(ADOPT_FAMILIES)
    for family in ADOPT_FAMILIES:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            np.random.seed(1)
            ml = builders[family]()
            b = np.random.default_rng(2).random(ml.levels[0].A.shape[0])
            extra = {"b": b, "x_V3": ml.solve(b, tol=0, maxiter=3), "x_W2": ml.solve(b, tol=0, maxiter=2, cycle="W")}
        save_hierarchy(os.path.join(REFERENCE_DIR, f"adopt_{family}.npz"), ml, extra=extra)

    builders = variant_builders()
    assert sorted(builders) == sorted(VARIANT_FAMILIES)
    for family in VARIANT_FAMILIES:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            np.random.seed(1)
            ml = builders[family]()
            n = ml.levels[0].A.shape[0]
            b, x0 = np.random.default_rng(2).random(n), np.random.default_rng(3).random(n)
            extra = {"b": b, "x0": x0}
            runs = variant_runs(x0)
            info, nres = np.full(len(runs), -99), np.zeros(len(runs), dtype=int)
            for k, kw in enumerate(runs):
                if family == "air" and kw.get("accel") == "cg":
                    continue                                  # nonsymmetric operator
                res = []
                extra[f"x_{k}"], info[k] = ml.solve(b, residuals=res, return_info=True, **kw)
                nres[k] = len(res)
            extra.update(info=info, nres=nres)
        save_hierarchy(os.path.join(REFERENCE_DIR, f"variants_{family}.npz"), ml, extra=extra)

    # 'MIS' colours of every level of the reference's RS hierarchies on poisson((30, 30)) and poisson((12, 12, 12)),
    # which are the cfg1 and cfg3 goldens' levels, and of a random symmetric graph
    R = sp.random(300, 300, 0.03, random_state=1)
    R = (R + R.T).tocsr()
    R.sort_indices()
    z = {"random_indptr": R.indptr.astype(np.int32), "random_indices": R.indices.astype(np.int16)}
    ref_graphs = []
    for A in (poisson((30, 30), format="csr"), poisson((12, 12, 12), format="csr")):
        ref_graphs += [lvl.A for lvl in pyamg.ruge_stuben_solver(A, max_coarse=10).levels]
    ref_graphs.append(R)
    graphs = mis_graphs(load_golden, z)
    assert len(graphs) == len(ref_graphs)
    for k, (G, Gr) in enumerate(zip(graphs, ref_graphs)):
        G, Gr = sp.csr_array(G), sp.csr_array(Gr)
        G.sort_indices()
        Gr.sort_indices()
        assert np.array_equal(G.indptr, Gr.indptr) and np.array_equal(G.indices, Gr.indices), k
        z[f"colours_{k}"] = vertex_coloring(Gr, "MIS").astype(np.uint8)
    np.savez_compressed(os.path.join(REFERENCE_DIR, "mis_colouring.npz"), **z)

    assert oracle.have_ref(), "oracle/_ref/libamg_ref.so is needed for compiled_kernels.json"
    from conftest import GOLDEN_ALL
    digests = {name: kernel_digests(load_golden(name)[0], "ref") for name in GOLDEN_ALL}
    with open(os.path.join(REFERENCE_DIR, "compiled_kernels.json"), "w") as f:
        json.dump(digests, f, indent=1)
        f.write("\n")
    for fn in sorted(os.listdir(REFERENCE_DIR)):
        print(f"reference/{fn}: {os.path.getsize(os.path.join(REFERENCE_DIR, fn)) / 1024:.0f} KB")


if __name__ == "__main__":
    if "--reference-checks" in sys.argv:
        main_reference_checks()
        sys.exit(0)
    if "--only" in sys.argv:
        ONLY = sys.argv[sys.argv.index("--only") + 1]
    if "--krylov" in sys.argv:
        KRYLOV_ONLY = True
        main()
        main_widening()
    elif "--widening" in sys.argv:
        main_widening()
    else:
        main()
        main_widening()
