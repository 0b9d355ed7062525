"""The smoothed aggregation definition (tests/sa_oracle.py) on the CPU: MIS(2) invariants, aggregates, the tentative
prolongator, the smoothed prolongator against its dense formula, theta and omega validation, stalled coarsening, the
prefix property and the convergence of oracle V-cycles with the SA operators.  The factors measured here are the
bounds tests/test_gpu_sa.py holds the device cycles to."""
import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.csgraph import shortest_path

import amg_oracle as AO
import sa_oracle as SO
from learnmultigrid_b200 import formats as F

PROBLEMS = AO.cpu_problems()
NAMES = sorted(PROBLEMS)


@pytest.fixture(scope="module", params=[(name, theta) for name in NAMES for theta in (0.0, 0.25)],
                ids=lambda p: "%s-%g" % p)
def case(request):
    name, theta = request.param
    A = F.canonical_csr(PROBLEMS[name])
    return name, A, SO.level(A, np.ones(A.shape[0]), theta=theta)


def graph_distances(S):
    G, _ = SO.neighbours(S)
    return shortest_path(G, unweighted=True), G


def test_mis2_roots_are_distance_3_apart_and_cover_every_point(case):
    name, A, d = case
    st = d["state"]
    assert np.all(st != SO.UNDECIDED)
    D, G = graph_distances(d["S"])
    isolated = np.diff(G.indptr) == 0
    roots = np.flatnonzero(st == SO.IN)
    assert len(roots) > 0 and not np.any(isolated[roots])
    sub = D[np.ix_(roots, roots)]
    np.fill_diagonal(sub, np.inf)
    assert sub.min() >= 3, name
    assert np.all(D[:, roots][~isolated].min(axis=1) <= 2)
    assert np.all(st[isolated] == SO.OUT)


def test_mis2_round_history_is_consistent(case):
    _, A, d = case
    st = d["state"]
    D, G = graph_distances(d["S"])
    isolated = np.diff(G.indptr) == 0
    assert d["rounds"] == len(d["history"]) > 0
    decided = isolated.copy()
    for new_in, new_out in d["history"]:
        assert not np.any(decided[new_in]) and not np.any(decided[new_out])
        # a point turned OUT has a root of an earlier round within distance 2
        earlier = np.flatnonzero(decided & (st == SO.IN))
        if len(new_out):
            assert len(earlier) and np.all(D[np.ix_(new_out, earlier)].min(axis=1) <= 2)
        decided[new_in] = decided[new_out] = True
        assert np.all(st[new_in] == SO.IN) and np.all(st[new_out] == SO.OUT)
    assert np.all(decided)


def test_aggregates_partition_the_points_around_one_root_each(case):
    _, A, d = case
    agg, nc, st = d["agg"], d["nc"], d["state"]
    G, isolated = SO.neighbours(d["S"])
    assert np.all(agg[isolated] == -1) and np.all(agg[~isolated] >= 0)
    assert set(agg[~isolated]) == set(range(nc))
    roots = np.flatnonzero(st == SO.IN)
    assert np.array_equal(agg[roots], np.arange(nc))               # roots numbered in ascending fine index
    for a in range(nc):
        members = np.flatnonzero(agg == a)
        assert np.sum(st[members] == SO.IN) == 1
        ncomp, _ = sp.csgraph.connected_components(G[members][:, members], directed=False)
        assert ncomp == 1


def test_tentative_prolongator_is_orthonormal_and_reproduces_b(case):
    _, A, d = case
    T, nu = d["T"], d["nu"]
    n = A.shape[0]
    for B in (np.ones(n), np.random.default_rng(3).uniform(0.5, 2.0, n)):
        T2, nu2 = SO.tentative(d["agg"], d["nc"], B)
        TtT = (T2.T @ T2).toarray()
        np.testing.assert_allclose(TtT, np.eye(d["nc"]), rtol=0, atol=4 * np.finfo(float).eps)
        Tnu = T2 @ nu2
        on = d["agg"] >= 0
        np.testing.assert_allclose(Tnu[on], B[on], rtol=4 * np.finfo(float).eps, atol=0)
        assert np.all(Tnu[~on] == 0)
    assert np.array_equal(nu, np.sqrt(np.bincount(d["agg"][d["agg"] >= 0]).astype(np.float64)))


def test_smoothed_prolongator_matches_the_dense_formula(case):
    _, A, d = case
    Ad = A.toarray()
    Dinv = np.diag(1.0 / np.diag(Ad))
    want = (np.eye(A.shape[0]) - d["omega_hat"] * Dinv @ Ad) @ d["T"].toarray()
    np.testing.assert_allclose(d["P"].toarray(), want, rtol=0, atol=1e-14)
    assert sp.csr_matrix(d["P"]).has_sorted_indices and np.all(d["P"].data != 0)
    assert d["omega_hat"] == 4.0 / 3.0 / d["lambda_max"]


def test_strength_threshold():
    A = F.canonical_csr(sp.csr_matrix(np.array([[4.0, -1.0, -0.2, 0.5], [-1.0, 4.0, -1.0, 0.0],
                                                [-0.2, -1.0, 1.0, -0.3], [0.5, 0.0, -0.3, 1.0]])))
    S = SO.strength(A, 0.25)
    # row 0: 1 >= 0.0625 * 16; 0.04 < 0.0625 * 4; 0.25 >= 0.0625 * 4 (positive couplings count too)
    assert list(S.indices[S.indptr[0]:S.indptr[1]]) == [1, 3]
    assert list(S.indices[S.indptr[2]:S.indptr[3]]) == [1, 3]              # 0.09 >= 0.0625 * 1
    S0 = SO.strength(A, 0.0)
    assert S0.nnz == np.count_nonzero(A.toarray() - np.diag(np.diag(A.toarray())))


def test_hash_keys_never_tie():
    """r_i is h(i) / 2^32 for a 32-bit hash h made of bijections, so the key's index component never decides"""
    h = (SO.r_hash(1 << 22) * 4294967296.0).astype(np.uint64)
    assert np.all(h == SO.r_hash(1 << 22) * 4294967296.0)
    assert len(np.unique(h)) == 1 << 22


@pytest.mark.parametrize("theta", [-0.1, 1.0, 1.5, float("nan")])
def test_theta_outside_range_is_rejected(theta):
    with pytest.raises(ValueError):
        SO.strength(PROBLEMS["poisson"], theta)
    from learnmultigrid_b200.sa import SaBuilder        # noqa: F401  (importable without a GPU)
    from learnmultigrid_b200.amg import check_theta
    with pytest.raises(ValueError):
        check_theta(theta)


@pytest.mark.parametrize("omega", [0.0, -1.0, 2.0, 3.0, float("nan")])
def test_omega_outside_range_is_rejected(omega):
    from learnmultigrid_b200.sa import check_omega
    with pytest.raises(ValueError):
        check_omega(omega)
    with pytest.raises(ValueError):
        SO.hierarchy(PROBLEMS["poisson"], 2, omega=omega)


def test_stalled_coarsening_is_rejected():
    with pytest.raises(ValueError, match="level 0"):
        SO.hierarchy(sp.identity(50, format="csr"), 2)                 # every point isolated: no aggregate
    with pytest.raises(ValueError, match="level 2"):
        SO.hierarchy(PROBLEMS["random"], 4)                            # one row left at level 2
    with pytest.raises(ValueError, match="level 1"):
        SO.hierarchy(PROBLEMS["poisson"], 3, theta=0.25)               # every coarse coupling weak


def test_zero_diagonal_is_rejected():
    with pytest.raises(ValueError, match="row 2"):
        SO.hierarchy(SO.zero_diagonal_matrix(), 2, lambdas=[1.0])


def test_isolated_points_stay_unaggregated():
    A = sp.lil_matrix(F.canonical_csr(PROBLEMS["poisson"]))
    A[0, :] = 0.0
    A[:, 0] = 0.0
    A[0, 0] = 3.0
    d = SO.level(F.canonical_csr(sp.csr_matrix(A)), np.ones(A.shape[0]))
    assert d["isolated"] >= 1 and d["agg"][0] == -1 and d["state"][0] == SO.OUT
    assert d["T"].indptr[1] == d["T"].indptr[0] and d["P"].indptr[1] == d["P"].indptr[0]


def test_prefix_property():
    P3, _, _ = SO.hierarchy(PROBLEMS["variable"], 3)
    P4, _, _ = SO.hierarchy(PROBLEMS["variable"], 4)
    for a, b in zip(P3, P4):
        assert (a != b).nnz == 0


def test_coarsening_is_aggressive():
    Ps, As, _ = SO.hierarchy(PROBLEMS["poisson"], 3)
    assert [M.shape[0] for M in As] == [1089, 197, 14]
    assert sum(M.nnz for M in As) / As[0].nnz < 1.5


def oracle_factor(name, levels, smoother):
    from oracle.vcycle import OracleMultigrid
    from chebyshev_oracle import ChebyshevOracle
    A = PROBLEMS[name]
    Ps, As, _ = SO.hierarchy(A, levels)
    b = np.random.default_rng(0).standard_normal((A.shape[0], 1))
    if smoother == "cheby":
        tabs = []
        for l in range(levels - 1):
            lam = F.chebyshev_lambda_max_host(As[l])
            tabs.append(F.chebyshev_coefficients(0.3 * lam, 1.1 * lam, 2))
        o = ChebyshevOracle(A, b, Ps, cheby_coefficients=tabs, hoist_setup=True)
    else:
        o = OracleMultigrid(A, b, Ps, smoother=smoother, omega=2.0 / 3.0,
                            colors=[F.greedy_colors(M)[0] for M in As], hoist_setup=True)
    o.solve(levels=levels, smooth_steps=1, error=1e-10 * np.linalg.norm(b), max_iterations=60)
    return AO.convergence_factor(o.track_res), o


CASES = [(name, levels) for name in NAMES for levels in sorted(SO.FACTOR_BOUNDS_SA[name])]


@pytest.mark.parametrize("name,levels", CASES)
@pytest.mark.parametrize("smoother", ["gs", "jacobi", "mcgs", "cheby"])
def test_oracle_vcycles_converge_within_the_measured_bounds(name, levels, smoother):
    rho, o = oracle_factor(name, levels, smoother)
    assert rho < SO.FACTOR_BOUNDS_SA[name][levels][smoother]
    assert o.track_res[-1, 0] < o.track_res[1, 0]


def test_smoothed_aggregation_mg_is_reachable_and_checks_parameters_without_a_gpu():
    from learn_multigrid.solvers.Multigrid import SmoothedAggregationMG
    from learnmultigrid_b200.solvers import Multigrid as M
    assert SmoothedAggregationMG is M.SmoothedAggregationMG and issubclass(SmoothedAggregationMG, M.AlgebraicMG)
    A = PROBLEMS["poisson"]
    b = np.ones((A.shape[0], 1))
    for kw in (dict(theta=-0.5), dict(theta=1.0), dict(omega=0.0), dict(omega=2.0), dict(omega=float("nan"))):
        with pytest.raises(ValueError):
            SmoothedAggregationMG(A, b, **kw)
    mg = SmoothedAggregationMG(A, b)
    assert mg.theta == 0.0 and mg.omega == 4.0 / 3.0 and mg.l_hierarchy == [] and mg.amg_stats is None
