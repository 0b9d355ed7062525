"""Smoothed aggregation on the device against tests/sa_oracle.py: strength pattern, MIS(2) states and rounds, aggregates,
nu, T, At and every P bit for bit, coarse operators bit for bit against SciPy's P^T A P, the device lambda_max against
its host twin, SmoothedAggregationMG histories against the oracle's cycles for every smoother within the convergence
bounds measured on the CPU, partitioned levels, PCG, the prefix property and the error paths."""
import numpy as np
import pytest
import scipy.sparse as sp

import amg_oracle as AO
import sa_oracle as SO
from helpers import assert_history_close
from learnmultigrid_b200 import formats as F

pytestmark = pytest.mark.gpu

PROBLEMS = AO.cpu_problems()
NAMES = sorted(PROBLEMS)
SMOOTHERS = {"mcgs": dict(smoother="GaussSeidel", gs_order="multicolor"),
             "gs": dict(smoother="GaussSeidel", gs_order="lexicographic"),
             "jacobi": dict(smoother="Jacobi"),
             "cheby": dict(smoother="Chebyshev")}
# the deepest hierarchy each problem coarsens to at theta 0 / 0.25 (coarse couplings turn weak at 0.25)
DEPTH = {0.0: {"poisson": 4, "variable": 4, "irregular": 4, "random": 3},
         0.25: {"poisson": 2, "variable": 2, "irregular": 4, "random": 2}}


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


def same_csr(got, want):
    assert got.shape == want.shape
    assert np.array_equal(got.indptr, want.indptr)
    assert np.array_equal(got.indices, want.indices)
    assert np.array_equal(got.data, want.data)


def check_builder_against_oracle(A, levels, theta=0.0):
    from learnmultigrid_b200.sa import SaBuilder
    b = SaBuilder()
    Ps = b.define_hierarchy(A, levels, theta, keep_intermediates=True)
    lams = [s["lambda_max"] for s in b.stats[:-1]]
    Po, As, info = SO.hierarchy(A, levels, theta, lambdas=lams)
    assert len(Ps) == len(Po) == levels - 1
    for l, d in enumerate(info):
        tr = b.trace[l]
        same_csr(b.download(tr["S"]), d["S"])
        St = sp.csr_matrix(d["S"]).T.tocsr()
        St.sort_indices()
        ST = b.download(tr["ST"])
        assert np.array_equal(ST.indptr, St.indptr) and np.array_equal(ST.indices, St.indices)
        assert np.array_equal(tr["state"].cpu().numpy(), d["state"])
        assert b.stats[l]["mis2_rounds"] == d["rounds"]
        assert b.stats[l]["isolated"] == d["isolated"]
        assert b.stats[l]["aggregates"] == d["nc"]
        assert np.array_equal(tr["agg"].cpu().numpy(), d["agg"])
        assert np.array_equal(tr["nu"].cpu().numpy(), d["nu"])
        same_csr(b.download(tr["T"]), d["T"])
        same_csr(b.download(tr["At"]), d["At"])
        assert b.stats[l]["omega_eff"] == d["omega_hat"]
        same_csr(b.download(Ps[l]), d["P"])
        same_csr(b.download(b.trace[l + 1]["A"]), As[l + 1])          # P^T A P: SciPy's bits
        np.testing.assert_allclose(lams[l], F.chebyshev_lambda_max_host(As[l]), rtol=1e-12)
    return b, info


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("theta", [0.0, 0.25])
def test_builder_is_bit_identical_to_the_oracle(torch_mod, name, theta):
    check_builder_against_oracle(PROBLEMS[name], DEPTH[theta][name], theta)


def test_builder_at_1025sq(torch_mod):
    """1.05M rows: thousands of blocks and several MIS(2) rounds on the fine level"""
    from learnmultigrid_b200 import problems as P
    A = P.structured_laplacian_2d(1024, P.variable_coefficient)
    b, info = check_builder_against_oracle(A, 3)
    assert info[0]["rounds"] >= 4
    gc, oc = b.complexities()
    assert 1.0 < gc < 1.5 and 1.0 < oc < 2.0


def run_solve(name, levels, key, **extra):
    from learnmultigrid_b200.solvers.Multigrid import SmoothedAggregationMG
    A = PROBLEMS[name]
    b = np.random.default_rng(0).standard_normal((A.shape[0], 1))
    mg = SmoothedAggregationMG(A, b)
    mg.solve(levels=levels, smooth_steps=1, error=1e-10 * np.linalg.norm(b), max_iterations=60,
             **SMOOTHERS[key], **extra)
    return mg, A, b


CASES = [(name, levels) for name in NAMES for levels in sorted(SO.FACTOR_BOUNDS_SA[name])]


@pytest.mark.parametrize("name,levels", CASES)
@pytest.mark.parametrize("key", sorted(SMOOTHERS))
def test_solve_matches_oracle_history_within_cpu_bounds(torch_mod, name, levels, key):
    from oracle.vcycle import OracleMultigrid
    from chebyshev_oracle import ChebyshevOracle
    mg, A, b = run_solve(name, levels, key)
    h = mg.get_hierarchy()
    assert len(mg.l_hierarchy) == levels - 1
    Ps = [mg._ab().download(q) for q in mg.l_hierarchy]
    st = mg.amg_stats
    Po, _, _ = SO.hierarchy(A, levels, lambdas=[s["lambda_max"] for s in st["levels"][:-1]])
    for q, qo in zip(Ps, Po):
        same_csr(q, qo)
    if key == "cheby":
        o = ChebyshevOracle(A, b, Ps, cheby_coefficients=h.cheby_coefficients, hoist_setup=True)
    else:
        o = OracleMultigrid(A, b, Ps, smoother=key, omega=2.0 / 3.0, colors=h.colors, hoist_setup=True)
    o.solve(levels=levels, smooth_steps=1, error=1e-10 * np.linalg.norm(b), max_iterations=60)
    assert_history_close(mg.track_res, o.track_res, A, o.solution)
    assert AO.convergence_factor(mg.track_res) < SO.FACTOR_BOUNDS_SA[name][levels][key]
    assert [s["rows"] for s in st["levels"]] == [A.shape[0]] + [q.shape[1] for q in Ps]
    assert st["theta"] == 0.0 and st["omega"] == 4.0 / 3.0
    assert st["grid_complexity"] > 1.0 and st["operator_complexity"] > 1.0


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("key", ["mcgs", "jacobi", "cheby"])
def test_partitioned_solve_is_bit_identical_to_one_gpu(torch_mod, world, key):
    from learnmultigrid_b200.distributed import run_virtual_ranks
    from learnmultigrid_b200.solvers.Multigrid import SmoothedAggregationMG
    A = PROBLEMS["poisson"]
    b = np.random.default_rng(0).standard_normal((A.shape[0], 1))
    kw = dict(levels=4, smooth_steps=1, error=0.0, max_iterations=8, **SMOOTHERS[key])
    mg1 = SmoothedAggregationMG(A, b)
    mg1.solve(**kw)
    P1 = [mg1._ab().download(q) for q in mg1.l_hierarchy]

    def body(fab):
        mg = SmoothedAggregationMG(A, b)
        mg.distribute(fab, n_dist=2, region_bytes=1 << 20, max_sites=256, timeout_s=30.0)
        mg.solve(**kw)
        out = (mg.get_solution().copy(), mg.track_res.copy(), [mg._ab().download(q) for q in mg.l_hierarchy])
        mg.get_hierarchy().close()
        return out

    for sol, hist, qs in run_virtual_ranks(world, body):
        for q, q1 in zip(qs, P1):
            same_csr(q, q1)
        assert np.array_equal(sol, mg1.get_solution())
        np.testing.assert_allclose(hist, mg1.track_res, rtol=1e-12)


@pytest.mark.parametrize("key", ["mcgs", "cheby"])
def test_preconditioner_is_symmetric_and_cg_converges(torch_mod, key):
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.solvers.CG import CG
    from learnmultigrid_b200.solvers.Multigrid import SmoothedAggregationMG
    torch = torch_mod
    N = 256
    A = P.symmetric_dirichlet(P.structured_laplacian_2d(N, P.variable_coefficient), P.boundary_nodes_2d(N))
    b = P.structured_rhs_2d(N)
    mg = SmoothedAggregationMG(A, b)
    M = mg.as_preconditioner(levels=4, smooth_steps=1, **SMOOTHERS[key])
    n = A.shape[0]
    rng = np.random.default_rng(0)
    dev = torch.device("cuda", torch.cuda.current_device())
    u, v = (torch.from_numpy(rng.standard_normal(n)).to(dev) for _ in range(2))
    Mu, Mv = torch.empty_like(u), torch.empty_like(v)
    M(u, Mu)
    M(v, Mv)
    asym = abs(float(torch.dot(u, Mv)) - float(torch.dot(v, Mu)))
    assert asym <= 1e-12 * float(torch.linalg.norm(u)) * float(torch.linalg.norm(Mv))
    cg = CG(A, b)
    cg.solve(max_iterations=200, error=1e-10, preconditioner=M)
    hist = np.asarray(cg.track_res).ravel()
    assert hist[-1] <= 1e-10 and len(hist) < 60


def test_solve_converges_on_a_larger_problem(torch_mod):
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.solvers.Multigrid import SmoothedAggregationMG
    from learn_multigrid.solvers.Multigrid import SmoothedAggregationMG as Alias
    assert Alias is SmoothedAggregationMG
    N = 128
    A = P.structured_laplacian_2d(N, P.variable_coefficient)
    b = P.structured_rhs_2d(N)
    mg = SmoothedAggregationMG(A, b)
    mg.solve(levels=4, smoother="GaussSeidel")
    assert mg.track_res[-1, 0] <= 1e-8 and mg.get_iterations() < 60
    x = mg.get_solution().ravel()
    assert np.linalg.norm(b.ravel() - A @ x) <= 1e-8


def test_prefix_property_and_cache(torch_mod):
    from learnmultigrid_b200.solvers.Multigrid import SmoothedAggregationMG
    A = PROBLEMS["irregular"]
    b = np.ones((A.shape[0], 1))
    m3 = SmoothedAggregationMG(A, b)
    q3 = m3.define_hierarchy(3)
    m4 = SmoothedAggregationMG(A, b)
    q4 = m4.define_hierarchy(4)
    assert len(q3) == 2 and len(q4) == 3
    for a, c in zip(q3, q4):
        same_csr(m3._ab().download(a), m4._ab().download(c))
    again = m4.define_hierarchy(3)                     # a prefix of the cached levels, not a new build
    assert all(x is y for x, y in zip(again, q4[:2]))
    assert [s["rows"] for s in m4.amg_stats["levels"]] == [A.shape[0], q4[0].shape[1], q4[1].shape[1]]
    stats, lh = m4.amg_stats, list(m4.l_hierarchy)
    B = PROBLEMS["variable"]
    x = m4.v_cycle(B, np.zeros((B.shape[0], 1)), np.ones((B.shape[0], 1)), "Jacobi", 1, 0.0, 3)
    assert x.shape == (B.shape[0], 1) and np.all(np.isfinite(x))
    assert m4.amg_stats is stats and all(a is c for a, c in zip(m4.l_hierarchy, lh))
    assert m4._amg_cache["other"][0] is B and m4._amg_cache["own"][0] is m4.matrix


def test_unassigned_point_is_an_error_naming_it(torch_mod):
    """states that no MIS(2) can produce: point 3 is OUT with no root within distance 2"""
    from learnmultigrid_b200 import _lib
    from learnmultigrid_b200.sa import SaBuilder, MIS_IN, MIS_OUT
    torch = torch_mod
    b = SaBuilder()
    A = b.upload(sp.diags([-np.ones(7), 2.0 * np.ones(8), -np.ones(7)], [-1, 0, 1]))
    S, ST = b.strength(A)
    state = torch.full((8,), MIS_OUT, dtype=torch.int32, device=b.dev)
    state[0] = MIS_IN
    with pytest.raises(_lib.MgError, match="point 3 is left unassigned"):
        b.aggregate(S, ST, state)
    state[2] = MIS_IN                                  # roots 0 and 2 are both neighbours of 1
    with pytest.raises(_lib.MgError, match="point 1 has two roots"):
        b.aggregate(S, ST, state)


def test_zero_diagonal_and_bad_parameters(torch_mod):
    from learnmultigrid_b200.sa import SaBuilder
    from learnmultigrid_b200.solvers.Multigrid import SmoothedAggregationMG
    with pytest.raises(ValueError, match="level 0.*row 2"):
        SaBuilder().define_hierarchy(SO.zero_diagonal_matrix(), 2)
    with pytest.raises(ValueError):
        SmoothedAggregationMG(PROBLEMS["poisson"], np.ones((1089, 1)), omega=2.0)
    I = sp.identity(300, format="csr")
    with pytest.raises(ValueError, match="level 0"):
        SmoothedAggregationMG(I, np.ones((300, 1))).solve(levels=2, smoother="Jacobi")
    with pytest.raises(ValueError, match="level 2"):
        SmoothedAggregationMG(PROBLEMS["random"], np.ones((600, 1))).define_hierarchy(4)
