"""CPU checks of restarted GMRES: the NumPy oracle (tests/gmres_oracle.py) against SciPy and against the stationary
multigrid iteration, the convection-diffusion generator, and the mg_gmres struct layout."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from gmres_oracle import gmres as oracle_gmres
from learnmultigrid_b200 import problems as P


def _scipy_history(A, b, atol, restart, maxiter):
    hist = []
    kw = {"rtol": 0.0} if "rtol" in spla.gmres.__code__.co_varnames else {"tol": 0.0}
    x, info = spla.gmres(A, b.ravel(), atol=atol, restart=restart, maxiter=maxiter, callback=hist.append,
                         callback_type="pr_norm", **kw)
    return x, np.asarray(hist) * np.linalg.norm(b), info


@pytest.mark.parametrize("restart", [200, 5])
def test_oracle_matches_scipy_on_convection_diffusion(restart):
    """Histories agree to rtol 1e-8 over the steps both take; the last steps before 1e-10 sit near the rounding floor
    of the estimate (a few ulp of ||b||), hence the absolute floor of 1e-14 ||b||."""
    N = 32
    A = P.convection_diffusion_2d(N, 0.02, (1.0, 0.5))
    assert abs(A - A.T).max() > 0
    b = P.structured_rhs_2d(N)
    tol = 1e-10
    x, track, its, res = oracle_gmres(A, b, error=tol, max_iterations=2000, restart=restart)
    xs, hs, info = _scipy_history(A, b, tol, restart, 2000)
    assert info == 0
    assert (its <= restart) == (restart == 200)                 # one cycle, or several restarts
    k = min(len(hs), len(track) - 1)
    assert k > 10
    np.testing.assert_allclose(track[1:k + 1], hs[:k], rtol=1e-8, atol=1e-14 * np.linalg.norm(b))
    assert abs(its - len(hs)) <= 1
    assert res <= tol and np.linalg.norm(b - A @ x) <= tol
    assert np.linalg.norm(b.ravel() - A @ xs) <= tol * 1.0001


def test_oracle_with_multigrid_beats_stationary_iteration():
    from oracle.vcycle import OracleMultigrid
    from learnmultigrid_b200 import formats as F
    N, L = 32, 4
    A = P.convection_diffusion_2d(N, 0.05, (1.0, -0.7))
    b = P.structured_rhs_2d(N)
    Qs = P.structured_hierarchy_2d(N, L, transfer="linear")
    colors = []
    Al = sp.csr_matrix(A)
    for l in range(L - 1):
        c, _ = F.greedy_colors(F.canonical_csr(Al))
        colors.append(c)
        Al = sp.csr_matrix(Qs[l].T @ Al @ Qs[l])
    o = OracleMultigrid(A, b, Qs, smoother="mcgs", colors=colors, hoist_setup=True)
    o.build_hierarchy(L)
    n = A.shape[0]

    def M(v):
        return o.v_cycle(o.matrix, np.zeros((n, 1)), v, 1, L)
    tol = 1e-10
    x = np.zeros((n, 1))
    stat = 0
    while np.linalg.norm(b - A @ x) > tol:
        x = x + M(b - A @ x)
        stat += 1
        assert stat < 500
    xg, track, its, res = oracle_gmres(A, b, precond=M, error=tol, max_iterations=500, restart=stat)
    assert its <= stat
    assert res <= tol and np.linalg.norm(b - A @ xg) <= tol


def test_oracle_restarts_on_true_residual_and_counts_steps():
    A = P.convection_diffusion_2d(16, 0.1, (1.0, 1.0))
    b = np.ones((A.shape[0], 1))
    x, track, its, res = oracle_gmres(A, b, error=1e-12, max_iterations=7, restart=3)
    assert its == 7 and len(track) == 8
    assert res == pytest.approx(np.linalg.norm(b - A @ x), rel=1e-12)
    x0, t0, i0, r0 = oracle_gmres(A, np.zeros_like(b))
    assert i0 == 0 and t0 == [0.0] and r0 == 0.0 and not x0.any()
    with pytest.raises(ValueError):
        oracle_gmres(A, b, restart=0)


def test_convection_diffusion_operator():
    N = 16
    L = P.structured_laplacian_2d(N)
    C = P.convection_diffusion_2d(N, 1.0, (0.0, 0.0))
    for a in ("indptr", "indices", "data"):
        assert np.array_equal(getattr(L, a), getattr(C, a))
    for eps, beta in ((0.01, (1.0, 0.3)), (0.5, (-2.0, 0.0)), (1e-3, (0.0, -1.0))):
        A = sp.csr_matrix(P.convection_diffusion_2d(N, eps, beta))
        assert A.has_canonical_format
        assert (A.diagonal() > 0).all()
        off = A - sp.diags(A.diagonal())
        assert off.data.max() <= 0.0
        interior = np.flatnonzero(np.diff(A.indptr) == 5)
        rs = np.asarray(A.sum(axis=1)).ravel()[interior]
        assert np.abs(rs).max() <= 1e-14 * (eps + abs(beta[0]) + abs(beta[1]))
        Ai = A[interior][:, interior]
        assert abs(Ai - Ai.T).max() > 0                     # nonsymmetric, not only through the Dirichlet rows
    with pytest.raises(ValueError):
        P.convection_diffusion_2d(N, 0.0, (1.0, 0.0))


def test_gmres_struct_size():
    from learnmultigrid_b200 import _lib
    lib = _lib.load()
    assert lib.mg_struct_size(9) == ctypes.sizeof(_lib.mg_gmres)
    assert lib.mg_krylov_partials(1000, 31) >= 31
