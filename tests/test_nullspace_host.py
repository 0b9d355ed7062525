"""Singular systems without a GPU: the Neumann generators against the repository's assembly, and the pinned coarsest
solve of tests/nullspace_oracle.py on the coarsest operators of every kind of hierarchy the engine builds."""
import numpy as np
import pytest
import scipy.sparse as sp

import amg_oracle as AO
import nullspace_oracle as NO
import sa_oracle as SO
from learnmultigrid_b200 import formats as F
from learnmultigrid_b200 import problems as P


def assembled(N, coefficient=None):
    from learnmultigrid_b200.mesh.Mesh2D import Mesh2D
    from learnmultigrid_b200.assembly.StiffnessMatrix import StiffnessMatrix
    from learnmultigrid_b200.assembly.LoadVector import LoadVector
    from learnmultigrid_b200.assembly.LoadFunction import LoadFunction
    from learnmultigrid_b200.assembly.Quadrature import Quadrature2D
    from learnmultigrid_b200.assembly.ShapeFunction import FunctionTriangle, GradientTriangle
    mesh, q = Mesh2D(N * N), Quadrature2D(3)
    kw = {} if coefficient is None else {"coefficient": coefficient}
    A = sp.csr_matrix(StiffnessMatrix(mesh).compute_stiffness_2d(GradientTriangle(1), q, format="csr", **kw))
    A.sort_indices()
    b = LoadVector(mesh).compute_rhs_2d(LoadFunction(lambda pts: -1.0), FunctionTriangle(1), q)
    return A, np.asarray(b, dtype=np.float64).reshape(-1, 1)


@pytest.mark.parametrize("N", [4, 8, 16])
@pytest.mark.parametrize("coef", [None, P.variable_coefficient], ids=["constant", "variable"])
def test_neumann_generator_matches_assembly(N, coef):
    A, b = assembled(N, coef)
    G = P.structured_laplacian_2d(N, coef, boundary="neumann")
    assert np.array_equal(G.indptr, A.indptr) and np.array_equal(G.indices, A.indices)
    np.testing.assert_allclose(G.data, A.data, rtol=1e-13, atol=1e-15)
    np.testing.assert_allclose(P.structured_rhs_2d(N, boundary="neumann"), b, rtol=1e-13)
    assert abs(G - G.T).max() <= 1e-15 * abs(G).max()
    assert np.abs(G @ np.ones(G.shape[0])).max() <= 1e-14 * abs(G).sum(axis=1).max()


@pytest.mark.parametrize("coef", [None, P.variable_coefficient], ids=["constant", "variable"])
def test_neumann_interior_rows_equal_dirichlet(coef):
    N = 12
    G = sp.csr_matrix(P.structured_laplacian_2d(N, coef, boundary="neumann"))
    D = sp.csr_matrix(P.structured_laplacian_2d(N, coef))
    assert abs(sp.csr_matrix(P.structured_laplacian_2d(N, coef, boundary="dirichlet")) - D).max() == 0.0
    interior = np.setdiff1d(np.arange(G.shape[0]), P.boundary_nodes_2d(N))
    for i in interior:
        assert np.array_equal(G.indices[G.indptr[i]:G.indptr[i + 1]], D.indices[D.indptr[i]:D.indptr[i + 1]])
        assert np.array_equal(G.data[G.indptr[i]:G.indptr[i + 1]], D.data[D.indptr[i]:D.indptr[i + 1]])
    # row blocks and rectangles as for the Dirichlet generator
    blk = P.structured_laplacian_2d(N, coef, rows=(20, 70), boundary="neumann")
    assert abs(sp.csr_matrix(blk) - G[20:70]).max() == 0.0
    R = sp.csr_matrix(P.structured_laplacian_2d(N, coef, Ny=2 * N, boundary="neumann"))
    assert np.abs(R @ np.ones(R.shape[0])).max() <= 1e-14 * abs(R).max()


def test_irregular_neumann():
    d = P.irregular_p1_2d(16, boundary="neumann")
    e = P.irregular_p1_2d(16)
    A = d["A"]
    assert abs(A - A.T).max() <= 1e-14 * abs(A).max()
    assert np.abs(A @ np.ones(A.shape[0])).max() <= 1e-13 * abs(A).sum(axis=1).max()
    inner = np.setdiff1d(np.arange(A.shape[0]), d["boundary"])
    assert abs(A[inner] - e["A"][inner]).max() == 0.0
    np.testing.assert_array_equal(d["rhs"][inner], e["rhs"][inner])
    assert np.all(d["rhs"][d["boundary"]] != 0.0)
    with pytest.raises(ValueError):
        P.irregular_p1_2d(16, boundary="periodic")


def coarsest_operators():
    """name -> coarsest operator of a Neumann hierarchy (linear, quasi-L2, AMG, SA)"""
    out = {}
    for transfer in ("linear", "quasi"):
        N = 32
        A = sp.csr_matrix(P.structured_laplacian_2d(N, P.variable_coefficient, boundary="neumann"))
        for Q in P.structured_hierarchy_2d(N, 3, transfer=transfer):
            A = sp.csr_matrix(Q.T @ A @ Q)
        out[transfer] = A
    An = P.irregular_p1_2d(32, boundary="neumann")["A"]
    out["amg"] = AO.hierarchy(An, 4)[1][-1]
    out["sa"] = SO.hierarchy(An, 3)[1][-1]
    return out


@pytest.mark.parametrize("name", ["linear", "quasi", "amg", "sa"])
def test_pinned_pseudo_inverse_matches_pinv(name):
    A = coarsest_operators()[name]
    Ad = A.toarray()
    o = NO.pinned(A)
    assert o["singular"], o["null_ratio"]
    want = np.linalg.pinv(Ad, rcond=1e-12, hermitian=True)
    assert np.abs(o["pinv"] - want).max() <= 1e-12 * np.abs(want).max() * max(1.0, np.linalg.cond(Ad + np.outer(
        o["nu"], o["nu"])) * 1e-4)
    s = NO.svd_null_vector(Ad)
    nu = o["nu"] / np.linalg.norm(o["nu"])
    assert min(np.abs(nu - s).max(), np.abs(nu + s).max()) <= 1e-10
    assert o["verify_ratio"] <= 1e-12


def test_decision_rule_and_verification():
    # a Dirichlet coarsest operator is nonsingular: taken unpinned
    A = sp.csr_matrix(P.structured_laplacian_2d(16, P.variable_coefficient))
    A = P.symmetric_dirichlet(A, P.boundary_nodes_2d(16))
    o = NO.pinned(A)
    assert not o["singular"] and o["null_ratio"] > 1e-6
    # two disconnected Neumann squares: singular by the rule, refused by the verification
    o = NO.pinned(NO.two_squares(6))
    assert o["singular"] and o["verify_ratio"] > 1e-2


# recorded: multicolour GS 0.189 (linear) / 0.062 (quasi-L2), damped Jacobi 0.427 (N = 32, variable coefficient)
@pytest.mark.parametrize("smoother,transfer,bound", [("mcgs", "linear", 0.2), ("jacobi", "linear", 0.45),
                                                     ("mcgs", "quasi", 0.07)])
def test_oracle_cycle_converges(smoother, transfer, bound):
    """the convergence factors the GPU tests bound with (tests/test_gpu_nullspace.py)"""
    N = 32
    A = P.structured_laplacian_2d(N, P.variable_coefficient, boundary="neumann")
    Qs = P.structured_hierarchy_2d(N, 3, transfer=transfer)
    b = F.chebyshev_start_vector(np.arange(A.shape[0], dtype=np.int64))
    hist, x = NO.stationary_history(A, Qs, np.ones(A.shape[0]), b, smoother=smoother, cycles=12)
    assert NO.factor(hist) < bound, NO.factor(hist)
    assert hist[-1] < bound ** 11 * hist[0]
    assert abs(x.sum()) <= 1e-12 * np.abs(x).sum()
