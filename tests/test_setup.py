"""CPU tests of the host-side setup (pyamg_b200.classical / gallery / graph): the hierarchies it
builds coincide with the ones the REAL reference built (golden fixtures), so bench inputs generated
on the GPU box are the BASELINE configs' hierarchies."""
import os

import numpy as np
import pytest

from pyamg_b200.classical import ruge_stuben_solver
from pyamg_b200.gallery import poisson, stencil_grid, diffusion_stencil_2d
from pyamg_b200.graph import vertex_coloring, color_order

CASES = [("cfg1_rs_gs_poisson2d", (30, 30), {}), ("cfg3_rs_mcgs_poisson3d", (12, 12, 12), {}),
         ("cfg6_rs_gsfwd_none_poisson3d", (9, 9, 9), {"max_coarse": 5})]


@pytest.mark.parametrize("name,grid,kw", CASES)
def test_rs_setup_reproduces_reference_hierarchy(name, grid, kw, load_golden):
    ref, _ = load_golden(name)
    ml = ruge_stuben_solver(poisson(grid), presmoother=None, postsmoother=None, **kw)
    assert [lv.A.shape for lv in ml.levels] == [lv.A.shape for lv in ref.levels]
    for a, b in zip(ml.levels, ref.levels):
        assert abs(a.A - b.A).max() < 1e-12
        if hasattr(b, "P"):
            assert a.P.shape == b.P.shape and abs(a.P - b.P).max() < 1e-13
            assert abs(a.R - b.R).max() < 1e-13
    assert ml.operator_complexity() == pytest.approx(ref.operator_complexity(), rel=1e-12)


def test_gallery_matches_reference_operators(load_golden):
    ref, _ = load_golden("cfg4_sa_jacobi_aniso2d")
    A = stencil_grid(diffusion_stencil_2d(epsilon=0.001, theta=np.pi / 6, type="FE"), (48, 48))
    assert abs(A - ref.levels[0].A).max() < 1e-15
    ref, _ = load_golden("cfg2_sa_jacobi_poisson2d")
    assert abs(poisson((40, 40)) - ref.levels[0].A).max() == 0
    P = poisson((2, 3)).toarray()           # pyamg/gallery/laplacian.py docstring example
    assert np.array_equal(P[0], [4, -1, 0, -1, 0, 0]) and np.array_equal(P[4], [0, -1, 0, -1, 4, -1])
    with pytest.raises(ValueError):
        stencil_grid(np.ones((2, 2)), (4, 4))


@pytest.mark.parametrize("method", ["greedy", "smallest_last", "LDF"])
@pytest.mark.parametrize("grid", [(17,), (9, 11), (6, 5, 7)])
def test_greedy_coloring_is_valid_and_red_black_on_stencils(grid, method):
    """pyamg/tests/test_graph.py:41-47 criterion: no edge joins equal colours; all colours used."""
    A = poisson(grid)
    c = vertex_coloring(A, method)
    coo = A.tocoo()
    off = coo.row != coo.col
    assert np.all(c[coo.row[off]] != c[coo.col[off]])
    assert set(c.tolist()) == set(range(c.max() + 1))
    assert c.max() + 1 == 2
    order = color_order(c)
    assert sorted(order.tolist()) == list(range(A.shape[0])) and np.all(np.diff(c[order]) >= 0)


def test_setup_rejects_options_outside_its_scope():
    A = poisson((8, 8))
    with pytest.raises(NotImplementedError):
        ruge_stuben_solver(A, strength="symmetric")
    with pytest.raises(NotImplementedError):
        ruge_stuben_solver(A, CF="PMIS")
    with pytest.raises(NotImplementedError):
        ruge_stuben_solver(A, interpolation="direct")


def test_colorings_are_valid_on_dense_coarse_operators(load_golden):
    """Coarse RS operators (unsorted columns, 20-100 entries per row): every method yields a proper colouring,
    smallest-last never needs more colours than the degeneracy bound allows."""
    ml, _ = load_golden("cfg3_rs_mcgs_poisson3d")
    for lvl in ml.levels[1:-1]:
        coo = lvl.A.tocoo()
        off = coo.row != coo.col
        for method in ("greedy", "smallest_last", "LDF"):
            c = vertex_coloring(lvl.A, method)
            assert np.all(c[coo.row[off]] != c[coo.col[off]]), method
            assert c.max() + 1 <= np.diff(lvl.A.indptr).max()
    with pytest.raises(NotImplementedError):
        vertex_coloring(ml.levels[0].A, "JP")


def test_sa_setup_reproduces_reference_hierarchy(load_golden):
    """Host smoothed-aggregation setup vs the hierarchy the REAL reference built for
    poisson((40,40)) (golden cfg2): identical aggregates / tentative prolongators are implied by identical
    P once the (randomly started, hence unreproducible) spectral-radius estimates of the reference run are
    recovered from its own P and injected; coarse operators then agree to rounding."""
    import scipy.sparse as sp
    from pyamg_b200.aggregation import (smoothed_aggregation_solver, symmetric_strength_pattern,
                                        standard_aggregation, fit_candidates)
    from pyamg_b200.util import get_diagonal
    ref, _ = load_golden("cfg2_sa_jacobi_poisson2d")
    # recover c_k = omega / rho_k of the reference run from P_k = T_k - c_k D^-1 A_k T_k
    rhos, B = [], np.ones(ref.levels[0].A.shape[0])
    import pyamg_b200._host as H
    for k, lv in enumerate(ref.levels[:-1]):
        A = sp.csr_array(lv.A)
        A.indptr, A.indices = A.indptr.astype(np.int32), A.indices.astype(np.int32)
        if k == 0:
            B = B.copy()
            H.lib().amgb_setup_gauss_seidel(A.shape[0], H.ip(A.indptr), H.ip(A.indices), H.dp(A.data), H.dp(B),
                                            H.dp(np.zeros(A.shape[0])), 4, 1)
        AggOp, _ = standard_aggregation(symmetric_strength_pattern(A))
        T, B = fit_candidates(AggOp, B)
        B = B.reshape(-1)
        U = sp.dia_array((get_diagonal(A, inv=True), 0), shape=A.shape) @ A @ T
        Dif = (T - sp.csr_array(lv.P)).tocsr()
        c = Dif.multiply(U).sum() / U.multiply(U).sum()
        rhos.append((4.0 / 3.0) / c)
    sm = ("jacobi", {"omega": 4.0 / 3.0})
    ml = smoothed_aggregation_solver(poisson((40, 40)), presmoother=sm, postsmoother=sm, rho=rhos)
    assert [lv.A.shape for lv in ml.levels] == [lv.A.shape for lv in ref.levels]
    for a, b in zip(ml.levels, ref.levels):
        assert abs(a.A - sp.csr_array(b.A)).max() < 1e-11
        if hasattr(b, "P"):
            assert abs(a.P - sp.csr_array(b.P)).max() < 1e-12
            assert abs(a.R - sp.csr_array(b.R)).max() < 1e-12
    # without injection the seeded estimate is close to the reference's random-start one
    ml2 = smoothed_aggregation_solver(poisson((40, 40)), presmoother=sm, postsmoother=sm)
    assert abs(ml2.levels[0].P - sp.csr_array(ref.levels[0].P)).max() < 5e-3
    w = ml2.levels[0].presmoother.keywords["omega"]
    assert w == pytest.approx(float(ref.levels[0].presmoother.keywords["omega"]), rel=2e-2)
    with pytest.raises(NotImplementedError):
        smoothed_aggregation_solver(poisson((8, 8)), strength="evolution")
    with pytest.raises(NotImplementedError):
        smoothed_aggregation_solver(poisson((8, 8)), symmetry="nonsymmetric")


def test_fit_candidates_known_answers():
    """The worked examples of the reference's fit_candidates docstring (tentative.py:60-114)."""
    import scipy.sparse as sp
    from pyamg_b200.aggregation import fit_candidates
    h = 1.0 / np.sqrt(2.0)
    AggOp = sp.csr_array(np.array([[1, 0], [1, 0], [0, 1], [0, 1]]))
    Q, R = fit_candidates(AggOp, [[1], [1], [1], [1]])
    assert np.allclose(Q.toarray(), [[h, 0], [h, 0], [0, h], [0, h]]) and np.allclose(R, [[2 * h], [2 * h]])
    Q, R = fit_candidates(AggOp, [[1, 0], [1, 1], [1, 2], [1, 3]])
    assert Q.format == "bsr" and Q.blocksize == (1, 2)
    assert np.allclose(Q.toarray(), [[h, -h, 0, 0], [h, h, 0, 0], [0, 0, h, -h], [0, 0, h, h]])
    assert np.allclose(R, [[2 * h, h], [0, h], [2 * h, 5 * h], [0, h]])
    AggOp = sp.csr_array(np.array([[1, 0], [1, 0], [0, 0], [0, 1]]))        # third node not aggregated
    Q, R = fit_candidates(AggOp, [[1], [1], [1], [1]])
    assert np.allclose(Q.toarray(), [[h, 0], [h, 0], [0, 0], [0, 1]]) and np.allclose(R, [[2 * h], [1.0]])
    # a candidate that is linearly dependent on an aggregate is dropped there (column of zeros, zero in R)
    AggOp = sp.csr_array(np.array([[1, 0], [1, 0], [0, 1], [0, 1]]))
    Q, R = fit_candidates(AggOp, [[1, 2], [1, 2], [1, 0], [1, 1]])
    assert np.allclose(Q.toarray()[:2, 1], 0.0) and R[1, 1] == 0.0 and R[3, 1] != 0.0
    assert np.allclose(Q @ R, [[1, 2], [1, 2], [1, 0], [1, 1]])
    with pytest.raises(ValueError):
        fit_candidates(AggOp, np.ones((5, 1)))


def test_vector_sa_setup_reproduces_reference_elasticity_hierarchy(load_golden):
    """BASELINE configs[4] family: gallery.linear_elasticity + smoothed aggregation with the three rigid-body
    modes (BSR(2,2) -> BSR(3,3)), block-Jacobi smoothers, against the hierarchy the REAL reference built
    (golden cfg5).  As in the scalar test the reference run's spectral-radius estimates are recovered from its
    own P and injected."""
    import scipy.sparse as sp
    from pyamg_b200.aggregation import (smoothed_aggregation_solver, symmetric_strength_pattern,
                                        standard_aggregation, fit_candidates, jacobi_prolongation_smoother,
                                        _improve_candidates)
    from pyamg_b200.gallery import linear_elasticity
    from pyamg_b200.util import get_diagonal
    ref, ex = load_golden("cfg5_sa_bjacobi_elasticity")
    A, B = linear_elasticity((14, 14))
    assert A.format == "bsr" and A.blocksize == (2, 2) and B.shape == (392, 3)
    A0 = sp.csr_array(ref.levels[0].A)
    assert abs(A.tocsr() - A0).max() < 1e-14 * abs(A0).max()
    assert np.array_equal(A.indices, ref.levels[0].A.indices) and np.array_equal(A.indptr, ref.levels[0].A.indptr)
    rhos, Ak, Bk = [], A, B
    for k, lv in enumerate(ref.levels[:-1]):
        AggOp, _ = standard_aggregation(symmetric_strength_pattern(Ak))
        if k == 0:
            Bk = _improve_candidates(Ak, Bk, "block_gauss_seidel", {"sweep": "symmetric", "iterations": 4})
        T, Bc = fit_candidates(AggOp, Bk)
        U = (sp.dia_array((get_diagonal(Ak, inv=True), 0), shape=Ak.shape) @ Ak.tocsr() @ T.tocsr()).tocsr()
        Dif = (T.tocsr() - sp.csr_array(lv.P)).tocsr()
        rhos.append((4.0 / 3.0) / (Dif.multiply(U).sum() / U.multiply(U).sum()))
        P = jacobi_prolongation_smoother(Ak, T, rho=rhos[-1])
        Ak, Bk = (P.T @ Ak @ P).tobsr(blocksize=(3, 3)), Bc
    ml = smoothed_aggregation_solver(A, B=B, presmoother="block_jacobi", postsmoother="block_jacobi", rho=rhos)
    assert [(lv.A.shape, lv.A.blocksize) for lv in ml.levels] == [(lv.A.shape, lv.A.blocksize) for lv in ref.levels]
    for a, b in zip(ml.levels, ref.levels):
        assert abs(a.A.tocsr() - sp.csr_array(b.A)).max() < 1e-12 * abs(sp.csr_array(b.A)).max()
        if hasattr(b, "P"):
            assert abs(a.P.tocsr() - sp.csr_array(b.P)).max() < 1e-12
            assert abs(a.R.tocsr() - sp.csr_array(b.R)).max() < 1e-12
            ka, kb = a.presmoother.keywords, b.presmoother.keywords
            assert ka["blocksize"] == kb["blocksize"]
            assert np.allclose(ka["Dinv"], kb["Dinv"], rtol=1e-10, atol=1e-18)
            assert ka["omega"] == pytest.approx(float(kb["omega"]), rel=5e-2)    # its own rho estimate (seeded here)
    # the cycle on the host-built hierarchy converges like the reference's
    import oracle
    spec = oracle.hierarchy_spec(ml)
    res = []
    oracle.Cycle(spec, coarse_pinv=ml.coarse_solver.dense_operator(ml.levels[-1].A)).solve(
        ex["b"], tol=0, maxiter=len(ex["residuals"]) - 1, residuals=res)
    assert res[-1] / res[0] < 2.0 * ex["residuals"][-1] / ex["residuals"][0]
    # default candidates of a block problem: one constant per unknown of a node
    ml3 = smoothed_aggregation_solver(A, max_coarse=20)
    assert ml3.levels[0].B.shape == (392, 2) and ml3.levels[1].A.blocksize == (2, 2)


MIS_COLOURS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "mis_colouring.npz")


def mis_graphs(load_golden, z):
    """Every level of the Ruge-Stuben hierarchies the REAL reference built for poisson((30, 30)) and
    poisson((12, 12, 12)) (golden cfg1 and cfg3), then a random symmetric graph stored beside the colours."""
    import scipy.sparse as sp
    graphs = [lvl.A for name in ("cfg1_rs_gs_poisson2d", "cfg3_rs_mcgs_poisson3d") for lvl in load_golden(name)[0].levels]
    n = len(z["random_indptr"]) - 1
    graphs.append(sp.csr_array((np.ones(len(z["random_indices"])), z["random_indices"], z["random_indptr"]), shape=(n, n)))
    return graphs


def test_mis_colouring_is_the_references(load_golden):
    """pyamg.graph.vertex_coloring(G, 'MIS') (amg_core/graph.h:218-235: repeated lexicographically-first maximal
    independent sets) equals natural-order first fit vertex by vertex -- checked against the colours the REAL
    reference computed (tests/golden/reference/mis_colouring.npz) on every level of two Ruge-Stuben hierarchies and
    a random graph."""
    from pyamg_b200.graph import vertex_coloring
    z = np.load(MIS_COLOURS)
    graphs = mis_graphs(load_golden, z)
    assert len(graphs) == len([k for k in z.files if k.startswith("colours_")])
    for k, G in enumerate(graphs):
        assert np.array_equal(z[f"colours_{k}"], vertex_coloring(G, "MIS")), k
