"""Chebyshev smoother, host side: coefficient recurrence, the oracle's step, the host twin of the Lanczos estimate."""
import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.linalg import eigsh

from learnmultigrid_b200 import formats as F
from learnmultigrid_b200 import problems as P
from chebyshev_oracle import cheby_smooth, cheby_step


def residual_polynomial(table, lam):
    """error factor of one application on an eigenvector of D^-1 A with eigenvalue lam (scalar recurrence)"""
    e, d = 1.0, 0.0
    for k, (c_d, c_r) in enumerate(table):
        dn = c_r * lam * e if k == 0 else c_d * d + c_r * lam * e
        e, d = e - dn, dn
    return e


@pytest.mark.parametrize("degree", [1, 2, 3, 4, 6])
@pytest.mark.parametrize("lo,hi", [(0.3, 1.1), (0.05, 2.0), (1.0, 1.5)])
def test_coefficients_give_the_chebyshev_residual_polynomial(degree, lo, hi):
    tab = F.chebyshev_coefficients(lo, hi, degree)
    assert tab.shape == (degree, 2) and tab.dtype == np.float64 and tab[0, 0] == 0.0
    theta, delta = (hi + lo) / 2, (hi - lo) / 2
    T = np.polynomial.chebyshev.Chebyshev.basis(degree)
    for lam in np.linspace(0.0, hi, 23):
        want = T((theta - lam) / delta) / T(theta / delta)
        assert abs(residual_polynomial(tab, lam) - want) <= 1e-13


@pytest.mark.parametrize("degree,bounds", [(0, None), (-1, None), (2.5, None), (True, None), (2, [(0.0, 1.0)]),
                                           (2, [(-1.0, 1.0)]), (2, [(1.0, 1.0)]), (2, [(2.0, 1.0)]),
                                           (2, [(0.1, float("inf"))])])
def test_bad_degree_or_bounds_raise(degree, bounds):
    with pytest.raises(ValueError):
        F.chebyshev_check(degree, bounds)
    if bounds is not None and isinstance(degree, int) and degree >= 1:
        with pytest.raises(ValueError):
            F.chebyshev_coefficients(bounds[0][0], bounds[0][1], degree)


def dense_step(A, x, b, d, c_d, c_r, first):
    """the step restated on a dense matrix, row sums over the stored entries in column order, Python floats"""
    n = A.shape[0]
    xo, dn_all = np.empty(n), np.empty(n)
    for i in range(n):
        s = 0.0
        for j in range(n):
            if A[i, j] != 0.0:
                s = s + A[i, j] * x[j]
        t = (1.0 / A[i, i]) * (b[i] - s)
        dn = c_r * t if first else (c_d * d[i]) + (c_r * t)
        xo[i], dn_all[i] = x[i] + dn, dn
    return xo, dn_all


def test_oracle_step_matches_dense_restatement():
    rng = np.random.default_rng(3)
    n = 40
    A = sp.random(n, n, density=0.15, random_state=4, format="csr") + 5.0 * sp.eye(n)
    A = F.canonical_csr(A)
    Ad = A.toarray()
    x, b, d = rng.standard_normal(n), rng.standard_normal(n), rng.standard_normal(n)
    tab = F.chebyshev_coefficients(0.4, 1.3, 3)
    dinv = 1.0 / A.diagonal()
    for k in range(3):
        got = cheby_step(A, x, b, d, dinv, tab[k, 0], tab[k, 1], k == 0)
        want = dense_step(Ad, x, b, d, tab[k, 0], tab[k, 1], k == 0)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
        x, d = got
    # two applications restart at step 0
    x0 = rng.standard_normal(n)
    y = cheby_smooth(A, x0, b, tab, 2)
    xx, dd = x0.copy(), np.zeros(n)
    for _ in range(2):
        for k in range(3):
            xx, dd = dense_step(Ad, xx, b, dd, tab[k, 0], tab[k, 1], k == 0)
    assert np.array_equal(y, xx)


def galerkin_levels(A, Qs):
    out = [sp.csr_matrix(A)]
    for Q in Qs:
        out.append(sp.csr_matrix(Q.T @ out[-1] @ Q))
    return out


def lambda_max(A):
    s = sp.diags(1.0 / np.sqrt(A.diagonal()))
    return float(eigsh(sp.csr_matrix(s @ A @ s), k=1, which="LA", return_eigenvectors=False, tol=1e-12)[0])


@pytest.mark.parametrize("case", ["poisson", "variable", "quasi"])
def test_host_lanczos_estimate_is_a_tight_lower_bound(case):
    N = 64
    coef = P.variable_coefficient if case == "variable" else None
    A = P.symmetric_dirichlet(P.structured_laplacian_2d(N, coef), P.boundary_nodes_2d(N))
    Qs = P.structured_hierarchy_2d(N, 4, transfer="quasi" if case == "quasi" else "linear")
    for Al in galerkin_levels(A, Qs)[:-1]:
        lam = lambda_max(Al)
        est = F.chebyshev_lambda_max_host(Al)
        assert 0.95 * lam <= est <= (1 + 1e-12) * lam, (est, lam)
        assert est == F.chebyshev_lambda_max_host(Al)           # deterministic


def test_start_vector_is_a_function_of_the_global_index():
    idx = np.arange(1000, dtype=np.int64)
    v = F.chebyshev_start_vector(idx)
    assert v.dtype == np.float64 and np.all(v >= -0.5) and np.all(v < 0.5)
    perm = np.random.default_rng(0).permutation(1000)
    assert np.array_equal(F.chebyshev_start_vector(idx[perm]), v[perm])
    big = np.array([2 ** 31 - 1], dtype=np.int64)
    assert np.isfinite(F.chebyshev_start_vector(big)).all()
    torch = pytest.importorskip("torch")
    assert np.array_equal(F.chebyshev_start_vector(torch.from_numpy(idx)).numpy(), v)


def test_lanczos_stops_on_breakdown():
    # D^-1/2 A D^-1/2 = 2 I: the first step spans an invariant space
    A = sp.csr_matrix(2.0 * sp.eye(50))
    assert F.chebyshev_lambda_max_host(A) == pytest.approx(1.0, rel=1e-14)
