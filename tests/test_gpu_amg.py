"""Classical AMG on the device against tests/amg_oracle.py: strength pattern, C/F states, PMIS rounds, promoted points
and every Q bit for bit, coarse operators bit for bit against SciPy's Q^T A Q, AlgebraicMG histories against the
oracle's cycles for every smoother within the convergence bounds measured on the CPU, partitioned levels, PCG and the
prefix property."""
import numpy as np
import pytest
import scipy.sparse as sp

import amg_oracle as AO
from helpers import assert_history_close

pytestmark = pytest.mark.gpu

PROBLEMS = AO.cpu_problems()
NAMES = sorted(PROBLEMS)
SMOOTHERS = {"mcgs": dict(smoother="GaussSeidel", gs_order="multicolor"),
             "gs": dict(smoother="GaussSeidel", gs_order="lexicographic"),
             "jacobi": dict(smoother="Jacobi"),
             "cheby": dict(smoother="Chebyshev")}


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


def download(b, M):
    return b.download(M)


def same_csr(got, want):
    assert got.shape == want.shape
    assert np.array_equal(got.indptr, want.indptr)
    assert np.array_equal(got.indices, want.indices)
    assert np.array_equal(got.data, want.data)


def check_builder_against_oracle(A, levels, theta=0.25):
    from learnmultigrid_b200.amg import AmgBuilder
    b = AmgBuilder()
    Qs = b.define_hierarchy(A, levels, theta, keep_intermediates=True)
    Qo, As, info = AO.hierarchy(A, levels, theta)
    assert len(Qs) == len(Qo) == levels - 1
    for l, d in enumerate(info):
        tr = b.trace[l]
        same_csr(download(b, tr["S"]), d["S"])
        St = sp.csr_matrix(d["S"]).T.tocsr()
        St.sort_indices()
        ST = download(b, tr["ST"])
        assert np.array_equal(ST.indptr, St.indptr) and np.array_equal(ST.indices, St.indices)
        pmis_state = tr["pmis_state"].cpu().numpy()
        state = tr["state"].cpu().numpy()
        assert np.array_equal(pmis_state, d["pmis_state"])
        assert np.array_equal(state, d["state"])
        assert b.stats[l]["pmis_rounds"] == d["rounds"]
        assert b.stats[l]["promoted"] == len(d["promoted"])
        assert np.array_equal(np.flatnonzero(state != pmis_state), d["promoted"])
        assert np.array_equal(tr["cmap"].cpu().numpy(), d["cmap"])
        same_csr(download(b, Qs[l]), d["Q"])
        same_csr(download(b, b.trace[l + 1]["A"]), As[l + 1])          # Q^T A Q: SciPy's bits
        assert b.stats[l]["c_points"] == d["Q"].shape[1]
    return b, info


@pytest.mark.parametrize("name", NAMES)
def test_builder_is_bit_identical_to_the_oracle(torch_mod, name):
    check_builder_against_oracle(PROBLEMS[name], 4)


@pytest.mark.parametrize("theta", [0.0, 0.5])
def test_builder_other_thresholds(torch_mod, theta):
    check_builder_against_oracle(PROBLEMS["variable"], 3, theta)


def test_builder_at_1025sq(torch_mod):
    """1.05M rows: thousands of blocks and several PMIS rounds per level"""
    from learnmultigrid_b200 import problems as P
    A = P.structured_laplacian_2d(1024, P.variable_coefficient)
    b, info = check_builder_against_oracle(A, 3)
    assert all(d["rounds"] >= 4 for d in info)
    gc, oc = b.complexities()
    assert 1.0 < gc < 2.0 and 1.0 < oc < 4.0


def run_solve(name, levels, key, **extra):
    from learnmultigrid_b200.solvers.Multigrid import AlgebraicMG
    A = PROBLEMS[name]
    b = np.random.default_rng(0).standard_normal((A.shape[0], 1))
    mg = AlgebraicMG(A, b)
    mg.solve(levels=levels, smooth_steps=1, error=1e-10 * np.linalg.norm(b), max_iterations=60,
             **SMOOTHERS[key], **extra)
    return mg, A, b


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("levels", [3, 4])
@pytest.mark.parametrize("key", sorted(SMOOTHERS))
def test_solve_matches_oracle_history_within_cpu_bounds(torch_mod, name, levels, key):
    from oracle.vcycle import OracleMultigrid
    from chebyshev_oracle import ChebyshevOracle
    mg, A, b = run_solve(name, levels, key)
    h = mg.get_hierarchy()
    assert len(mg.l_hierarchy) == levels - 1
    Qs = [mg._ab().download(q) for q in mg.l_hierarchy]
    Qo, _, _ = AO.hierarchy(A, levels)
    for q, qo in zip(Qs, Qo):
        same_csr(q, qo)
    if key == "cheby":
        o = ChebyshevOracle(A, b, Qs, cheby_coefficients=h.cheby_coefficients, hoist_setup=True)
    else:
        o = OracleMultigrid(A, b, Qs, smoother=key, omega=2.0 / 3.0, colors=h.colors, hoist_setup=True)
    o.solve(levels=levels, smooth_steps=1, error=1e-10 * np.linalg.norm(b), max_iterations=60)
    assert_history_close(mg.track_res, o.track_res, A, o.solution)
    assert AO.convergence_factor(mg.track_res) < AO.FACTOR_BOUNDS[name][levels][key]
    st = mg.amg_stats
    assert [s["rows"] for s in st["levels"]] == [A.shape[0]] + [q.shape[1] for q in Qs]
    assert st["grid_complexity"] > 1.0 and st["operator_complexity"] > 1.0


def test_solve_converges_without_transfer_operators(torch_mod):
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.solvers.Multigrid import AlgebraicMG
    from learn_multigrid.solvers.Multigrid import AlgebraicMG as Alias
    assert Alias is AlgebraicMG
    N = 128
    A = P.structured_laplacian_2d(N, P.variable_coefficient)
    b = P.structured_rhs_2d(N)
    mg = AlgebraicMG(A, b)
    mg.solve(levels=4, smoother="GaussSeidel")
    assert mg.track_res[-1, 0] <= 1e-8 and mg.get_iterations() < 60
    x = mg.get_solution().ravel()
    assert np.linalg.norm(b.ravel() - A @ x) <= 1e-8


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("key", ["mcgs", "jacobi", "cheby"])
def test_partitioned_solve_is_bit_identical_to_one_gpu(torch_mod, world, key):
    from learnmultigrid_b200.distributed import run_virtual_ranks
    from learnmultigrid_b200.solvers.Multigrid import AlgebraicMG
    A = PROBLEMS["poisson"]
    b = np.random.default_rng(0).standard_normal((A.shape[0], 1))
    kw = dict(levels=4, smooth_steps=1, error=0.0, max_iterations=8, **SMOOTHERS[key])
    mg1 = AlgebraicMG(A, b)
    mg1.solve(**kw)
    Q1 = [mg1._ab().download(q) for q in mg1.l_hierarchy]

    def body(fab):
        mg = AlgebraicMG(A, b)
        mg.distribute(fab, n_dist=2, region_bytes=1 << 20, max_sites=256, timeout_s=30.0)
        mg.solve(**kw)
        out = (mg.get_solution().copy(), mg.track_res.copy(), [mg._ab().download(q) for q in mg.l_hierarchy])
        mg.get_hierarchy().close()
        return out

    for sol, hist, qs in run_virtual_ranks(world, body):
        for q, q1 in zip(qs, Q1):
            same_csr(q, q1)
        assert np.array_equal(sol, mg1.get_solution())
        np.testing.assert_allclose(hist, mg1.track_res, rtol=1e-12)


@pytest.mark.parametrize("key", ["mcgs", "cheby"])
def test_preconditioner_is_symmetric_and_cg_converges(torch_mod, key):
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.solvers.CG import CG
    from learnmultigrid_b200.solvers.Multigrid import AlgebraicMG
    torch = torch_mod
    N = 256
    A = P.symmetric_dirichlet(P.structured_laplacian_2d(N, P.variable_coefficient), P.boundary_nodes_2d(N))
    b = P.structured_rhs_2d(N)
    mg = AlgebraicMG(A, b)
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


def test_prefix_property_and_cache(torch_mod):
    from learnmultigrid_b200.solvers.Multigrid import AlgebraicMG
    A = PROBLEMS["irregular"]
    b = np.ones((A.shape[0], 1))
    m3 = AlgebraicMG(A, b)
    q3 = m3.define_hierarchy(3)
    m4 = AlgebraicMG(A, b)
    q4 = m4.define_hierarchy(4)
    assert len(q3) == 2 and len(q4) == 3
    for a, c in zip(q3, q4):
        same_csr(m3._ab().download(a), m4._ab().download(c))
    again = m4.define_hierarchy(3)                     # a prefix of the cached levels, not a new build
    assert all(x is y for x, y in zip(again, q4[:2]))
    assert [s["rows"] for s in m4.amg_stats["levels"]] == [A.shape[0], q4[0].shape[1], q4[1].shape[1]]
    # a V-cycle for another operator builds and caches its own operators; l_hierarchy and amg_stats stay this matrix's
    stats, lh = m4.amg_stats, list(m4.l_hierarchy)
    B = PROBLEMS["variable"]
    x = m4.v_cycle(B, np.zeros((B.shape[0], 1)), np.ones((B.shape[0], 1)), "Jacobi", 1, 0.0, 3)
    assert x.shape == (B.shape[0], 1) and np.all(np.isfinite(x))
    assert m4.amg_stats is stats and all(a is c for a, c in zip(m4.l_hierarchy, lh))
    assert m4._amg_cache["other"][0] is B and m4._amg_cache["own"][0] is m4.matrix


def test_zero_denominator_is_an_error_naming_the_row(torch_mod):
    from learnmultigrid_b200 import _lib
    from learnmultigrid_b200.amg import AmgBuilder
    b = AmgBuilder()
    A = b.upload(AO.zero_denominator_matrix())
    S, ST = b.strength(A)
    state = b.split(S, ST)
    assert list(state.cpu().numpy()) == [AO.F_POINT, AO.C_POINT] + [AO.F_POINT] * 4
    with pytest.raises(_lib.MgError, match="row 4"):
        b.interpolate(A, S, state)
    with pytest.raises(_lib.MgError, match="row 4"):
        b.define_hierarchy(AO.zero_denominator_matrix(), 2)


def test_invalid_inputs(torch_mod):
    from learnmultigrid_b200.solvers.Multigrid import AlgebraicMG
    with pytest.raises(ValueError):
        AlgebraicMG(PROBLEMS["poisson"], np.ones((1089, 1)), theta=1.0)
    I = sp.identity(300, format="csr")
    with pytest.raises(ValueError, match="level 0"):
        AlgebraicMG(I, np.ones((300, 1))).solve(levels=2, smoother="Jacobi")
    with pytest.raises(ValueError, match="level"):
        AlgebraicMG(PROBLEMS["poisson"], np.ones((1089, 1))).define_hierarchy(40)
