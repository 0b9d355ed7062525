"""The classical AMG definition (tests/amg_oracle.py) on the CPU: PMIS invariants, promotion, interpolation rows, the
theta range, stalled coarsening and the convergence of oracle V-cycles with the AMG operators.  The factors measured
here are the bounds tests/test_gpu_amg.py holds the device cycles to."""
import numpy as np
import pytest
import scipy.sparse as sp

import amg_oracle as AO
from learnmultigrid_b200 import formats as F

PROBLEMS = AO.cpu_problems()
NAMES = sorted(PROBLEMS)


@pytest.fixture(scope="module", params=NAMES)
def case(request):
    A = PROBLEMS[request.param]
    return request.param, A, AO.level(A)


def test_pmis_decides_every_point_and_rounds_are_consistent(case):
    name, A, d = case
    S, st0 = d["S"], d["pmis_state"]
    assert np.all(st0 != AO.UNDECIDED)
    assert d["rounds"] == len(d["history"]) > 0
    G = sp.csr_matrix(AO._pattern(S) + AO._pattern(S).T)
    decided = np.zeros(A.shape[0], dtype=bool)
    decided[AO.transpose_counts(S) == 0] = True          # start as F
    assert np.all(st0[AO.transpose_counts(S) == 0] == AO.F_POINT)
    for new_c, new_f in d["history"]:
        # the C points of one round are independent in S u S^T
        sub = G[new_c][:, new_c]
        assert sub.nnz == 0, name
        # every point that mark turns F depends strongly on a C point
        for i in new_f:
            cols = S.indices[S.indptr[i]:S.indptr[i + 1]]
            assert np.any(st0[cols] == AO.C_POINT)
        assert not np.any(decided[new_c]) and not np.any(decided[new_f])
        decided[new_c] = decided[new_f] = True
    assert np.all(decided)


def test_promotion_leaves_no_f_row_without_a_strong_c_point(case):
    _, A, d = case
    S, st = d["S"], d["state"]
    for i in np.flatnonzero(st == AO.F_POINT):
        cols = S.indices[S.indptr[i]:S.indptr[i + 1]]
        if len(cols):
            assert np.any(st[cols] == AO.C_POINT)
    for i in d["promoted"]:
        assert d["pmis_state"][i] == AO.F_POINT and st[i] == AO.C_POINT
    assert np.array_equal(np.flatnonzero(st != d["pmis_state"]), d["promoted"])


def test_interpolation_rows(case):
    _, A, d = case
    Q, st, cmap, S = d["Q"], d["state"], d["cmap"], d["S"]
    A = F.canonical_csr(A)
    assert Q.shape == (A.shape[0], int((st == AO.C_POINT).sum()))
    assert sp.csr_matrix(Q).has_sorted_indices
    lens = np.diff(Q.indptr)
    for i in np.flatnonzero(st == AO.C_POINT):
        assert lens[i] == 1 and Q.indices[Q.indptr[i]] == cmap[i] and Q.data[Q.indptr[i]] == 1.0
    # only F rows with an empty S_i have no entries
    empty = np.flatnonzero(lens == 0)
    assert np.all(st[empty] == AO.F_POINT) and np.all(np.diff(S.indptr)[empty] == 0)
    # partition of unity on the F rows of zero row sum
    rowsum = np.asarray(A.sum(axis=1)).ravel()
    qsum = np.asarray(Q.sum(axis=1)).ravel()
    rows = np.flatnonzero((st == AO.F_POINT) & (rowsum == 0.0) & (lens > 0))
    np.testing.assert_allclose(qsum[rows], 1.0, rtol=0, atol=1e-14)


def test_zero_row_sum_rows_exist_where_expected():
    for name in ("poisson", "irregular"):
        d = AO.level(PROBLEMS[name])
        rowsum = np.asarray(PROBLEMS[name].sum(axis=1)).ravel()
        assert np.sum((d["state"] == AO.F_POINT) & (rowsum == 0.0)) > 100


def test_theta_zero_makes_every_negative_coupling_strong():
    for A in PROBLEMS.values():
        A = F.canonical_csr(A)
        S = AO.strength(A, 0.0)
        N = sp.csr_matrix(A, copy=True)
        N.setdiag(0.0)
        N.data[N.data > 0] = 0.0
        N.eliminate_zeros()
        assert np.array_equal(S.indptr, N.indptr) and np.array_equal(S.indices, N.indices)
        assert np.array_equal(S.data, N.data)


def test_strength_threshold():
    A = F.canonical_csr(sp.csr_matrix(np.array([[4.0, -1.0, -0.2, 0.5], [-1.0, 4.0, -1.0, 0.0],
                                                [-0.3, -1.0, 4.0, -2.0], [0.0, 0.0, 0.0, 1.0]])))
    S = AO.strength(A, 0.25)
    assert list(S.indices[S.indptr[0]:S.indptr[1]]) == [1]               # 0.2 < 0.25 * 1
    assert list(S.indices[S.indptr[2]:S.indptr[3]]) == [1, 3]            # 0.3 < 0.25 * 2 <= 1
    assert np.diff(S.indptr)[3] == 0                                     # no negative off-diagonal entry
    S = AO.strength(A, 0.6)
    assert list(S.indices[S.indptr[2]:S.indptr[3]]) == [3]               # 1 < 0.6 * 2


@pytest.mark.parametrize("theta", [-0.1, 1.0, 1.5, float("nan")])
def test_theta_outside_range_is_rejected(theta):
    with pytest.raises(ValueError):
        AO.strength(PROBLEMS["poisson"], theta)
    from learnmultigrid_b200.amg import check_theta
    with pytest.raises(ValueError):
        check_theta(theta)


def test_stalled_coarsening_is_rejected():
    with pytest.raises(ValueError, match="level 0"):
        AO.hierarchy(sp.identity(50, format="csr"), 2)
    with pytest.raises(ValueError, match="level"):
        AO.hierarchy(PROBLEMS["poisson"], 40)


def test_zero_denominator_names_the_row():
    A = AO.zero_denominator_matrix()
    d_state, _ = AO.promote(AO.strength(A), AO.pmis(AO.strength(A))[0])
    assert list(d_state) == [AO.F_POINT, AO.C_POINT] + [AO.F_POINT] * 4
    with pytest.raises(ValueError, match="row 4"):
        AO.level(A)


def test_weights_host_twin_and_pmis_is_deterministic():
    from learnmultigrid_b200.amg import pmis_weights_host
    S = AO.strength(PROBLEMS["irregular"])
    assert np.array_equal(AO.weights(S), pmis_weights_host(AO.transpose_counts(S)))
    a, b = AO.level(PROBLEMS["irregular"]), AO.level(PROBLEMS["irregular"])
    assert np.array_equal(a["state"], b["state"]) and np.array_equal(a["Q"].data, b["Q"].data)


def test_prefix_property():
    Q3, _, _ = AO.hierarchy(PROBLEMS["variable"], 3)
    Q4, _, _ = AO.hierarchy(PROBLEMS["variable"], 4)
    for a, b in zip(Q3, Q4):
        assert (a != b).nnz == 0


def oracle_factor(name, levels, smoother):
    from oracle.vcycle import OracleMultigrid
    from chebyshev_oracle import ChebyshevOracle
    A = PROBLEMS[name]
    Qs, As, _ = AO.hierarchy(A, levels)
    b = np.random.default_rng(0).standard_normal((A.shape[0], 1))
    if smoother == "cheby":
        tabs = []
        for l in range(levels - 1):
            lam = F.chebyshev_lambda_max_host(As[l])
            tabs.append(F.chebyshev_coefficients(0.3 * lam, 1.1 * lam, 2))
        o = ChebyshevOracle(A, b, Qs, cheby_coefficients=tabs, hoist_setup=True)
    else:
        o = OracleMultigrid(A, b, Qs, smoother=smoother, omega=2.0 / 3.0,
                            colors=[F.greedy_colors(M)[0] for M in As], hoist_setup=True)
    o.solve(levels=levels, smooth_steps=1, error=1e-10 * np.linalg.norm(b), max_iterations=60)
    return AO.convergence_factor(o.track_res), o


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("levels", [3, 4])
@pytest.mark.parametrize("smoother", ["gs", "jacobi", "mcgs", "cheby"])
def test_oracle_vcycles_converge_within_the_measured_bounds(name, levels, smoother):
    rho, o = oracle_factor(name, levels, smoother)
    assert rho < AO.FACTOR_BOUNDS[name][levels][smoother]
    assert rho < 0.8
    assert o.track_res[-1, 0] < o.track_res[1, 0]


def test_algebraic_mg_is_reachable_and_checks_theta_without_a_gpu():
    from learn_multigrid.solvers.Multigrid import AlgebraicMG
    from learnmultigrid_b200.solvers import Multigrid as M
    assert AlgebraicMG is M.AlgebraicMG
    A = PROBLEMS["poisson"]
    for theta in (-0.5, 1.0):
        with pytest.raises(ValueError):
            AlgebraicMG(A, np.ones((A.shape[0], 1)), theta=theta)
    mg = AlgebraicMG(A, np.ones((A.shape[0], 1)), theta=0.5)
    assert mg.theta == 0.5 and mg.l_hierarchy == [] and mg.amg_stats is None
