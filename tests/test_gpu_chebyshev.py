"""Chebyshev smoother on the device: the SELL step bit for bit against the oracle on every row path, the V-cycle against
ChebyshevOracle, the Lanczos bounds, the large-level switches, partitioned levels, MG-preconditioned CG and the API."""
import ctypes
import os

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.linalg import eigsh

from oracle.vcycle import pcg_solve
from chebyshev_oracle import ChebyshevOracle, cheby_smooth, cheby_step
from helpers import bilinear_P, poisson2d

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    import torch
    from learnmultigrid_b200 import _lib
    assert torch.cuda.is_available()
    return {"torch": torch, "lib": _lib.load(), "L": _lib, "dev": torch.device("cuda", 0)}


def up(env, a):
    return env["torch"].from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(env["dev"])


def st(env):
    return env["L"].stream_handle(env["torch"])


def rows_matrix(n, per_row, ragged, seed):
    """n x n, per_row entries per row (diagonal included), or 1..per_row entries per row when ragged"""
    from learnmultigrid_b200 import formats as F
    rng = np.random.default_rng(seed)
    cnt = rng.integers(1, per_row + 1, size=n) if ragged else np.full(n, per_row)
    r, c = [], []
    for i in range(n):
        off = rng.choice(np.arange(-3 * per_row, 3 * per_row + 1), size=cnt[i] - 1, replace=False)
        off = off[off != 0][:cnt[i] - 1]
        cols = np.unique(np.concatenate([[i], (i + off) % n]))
        r.extend([i] * len(cols))
        c.extend(cols)
    v = rng.uniform(-1.0, 1.0, size=len(r))
    A = sp.csr_matrix((v, (r, c)), shape=(n, n)) + sp.diags(2.0 * per_row + rng.uniform(0, 1, size=n))
    return F.canonical_csr(A)


def structured(N, transfer_levels=0, quasi=False):
    from learnmultigrid_b200 import formats as F
    from learnmultigrid_b200 import problems as P
    A = P.structured_laplacian_2d(N)
    Qs = P.structured_hierarchy_2d(N, transfer_levels + 1, transfer="quasi" if quasi else "linear") if transfer_levels else []
    for Q in Qs:
        A = F.canonical_csr(sp.csr_matrix(Q.T @ A @ Q))
    return F.canonical_csr(A)


def device_steps(env, S, A, x, b, d, tab):
    """all steps of the table on the device: (x, d) after each, plus the zero-iterate skip"""
    L, lib, torch = env["L"], env["lib"], env["torch"]
    n = A.shape[0]
    dinv = up(env, 1.0 / A.diagonal())
    dx, db, dd = up(env, x), up(env, b), up(env, d)
    xo = torch.empty_like(dx)
    outs = []
    for k in range(len(tab)):
        L.check(lib.mg_sell_chebyshev(ctypes.byref(S.struct), dinv.data_ptr(), dx.data_ptr(), db.data_ptr(),
                                      dd.data_ptr(), xo.data_ptr(), float(tab[k][0]), float(tab[k][1]), int(k == 0),
                                      st(env)), "mg_sell_chebyshev")
        outs.append((xo.clone(), dd.clone()))
        dx, xo = xo, dx
    # the zero-iterate skip against the matrix step on zeros
    z = torch.zeros_like(dx)
    dz, xz = torch.full_like(dx, 7.0), torch.empty_like(dx)
    L.check(lib.mg_sell_chebyshev(ctypes.byref(S.struct), dinv.data_ptr(), z.data_ptr(), db.data_ptr(), dz.data_ptr(),
                                  xz.data_ptr(), 0.0, float(tab[0][1]), 1, st(env)), "mg_sell_chebyshev")
    ds, xs = torch.full_like(dx, 7.0), torch.empty_like(dx)
    L.check(lib.mg_chebyshev_zero_first(n, float(tab[0][1]), dinv.data_ptr(), db.data_ptr(), ds.data_ptr(),
                                        xs.data_ptr(), st(env)), "mg_chebyshev_zero_first")
    assert torch.equal(xz, xs) and torch.equal(dz, ds)
    return outs


def check_steps(env, S, A, seed=0):
    rng = np.random.default_rng(seed)
    n = A.shape[0]
    x, b, d = rng.standard_normal(n), rng.standard_normal(n), rng.standard_normal(n)
    from learnmultigrid_b200 import formats as F
    tab = F.chebyshev_coefficients(0.3, 1.7, 3)
    outs = device_steps(env, S, A, x, b, d, tab)
    dinv = 1.0 / A.diagonal()
    for k in range(len(tab)):
        x, d = cheby_step(A, x, b, d, dinv, tab[k][0], tab[k][1], k == 0)
        assert np.array_equal(outs[k][0].cpu().numpy(), x), k
        assert np.array_equal(outs[k][1].cpu().numpy(), d), k
    return outs


@pytest.mark.parametrize("per_row", [1, 2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("ragged", [False, True])
def test_step_bit_exact_short_rows(env, per_row, ragged):
    from learnmultigrid_b200.engine import DeviceSell
    A = rows_matrix(3000 + 17 * per_row, per_row, ragged, per_row + 100 * ragged)
    S = DeviceSell(env["torch"], A, env["dev"])
    assert S.max_len <= 8
    check_steps(env, S, A, per_row)


def test_step_bit_exact_long_rows_and_wide_path(env):
    from learnmultigrid_b200.engine import DeviceSell
    lib = env["lib"]
    A = rows_matrix(2500, 12, True, 5)
    S = DeviceSell(env["torch"], A, env["dev"])
    assert S.max_len > 8
    old = lib.mg_set_wide_min_len(0)            # thread-per-row kernel, LEN = 0 (chunks of 4 + remainder)
    try:
        check_steps(env, S, A, 1)
    finally:
        lib.mg_set_wide_min_len(old)
    # 19-point (uniform) and 16..37-point (ragged) quasi-L2 Galerkin rows: warps-per-slice kernel
    for A in (structured(64, 1, quasi=True), structured(64, 2, quasi=True)):
        S = DeviceSell(env["torch"], A, env["dev"])
        assert S.max_len >= 9
        check_steps(env, S, A, 2)


def test_step_bit_exact_with_every_switch(env):
    """value dictionary, implied columns and implied values on a structured 5-point level, each on and off"""
    from learnmultigrid_b200.engine import DeviceSell
    lib = env["lib"]
    A = structured(128)
    old_floor = lib.mg_set_implied_min_rows(1)
    os.environ["MGB_IMPLIED_MIN_ROWS"] = "1"
    os.environ["MGB_VALUE_DICT_MIN_ROWS"] = "1"
    try:
        S = DeviceSell(env["torch"], A, env["dev"])
        assert S.val_idx is not None and S.slice_rec is not None and S.rec_vals is not None
        ref = None
        for dct in (0, 1):
            for impl in (0, 1):
                for impv in (0, 1):
                    lib.mg_set_value_dict(dct)
                    lib.mg_set_implied_columns(impl)
                    lib.mg_set_implied_values(impv)
                    outs = check_steps(env, S, A, 4)
                    if ref is None:
                        ref = outs
                    for (x1, d1), (x2, d2) in zip(outs, ref):
                        assert env["torch"].equal(x1, x2) and env["torch"].equal(d1, d2)
    finally:
        lib.mg_set_value_dict(1)
        lib.mg_set_implied_columns(1)
        lib.mg_set_implied_values(1)
        lib.mg_set_implied_min_rows(old_floor)
        os.environ.pop("MGB_IMPLIED_MIN_ROWS", None)
        os.environ.pop("MGB_VALUE_DICT_MIN_ROWS", None)


def test_step_rejects_aliasing_and_zero_c_d(env):
    from learnmultigrid_b200.engine import DeviceSell
    lib, torch = env["lib"], env["torch"]
    A = rows_matrix(100, 3, False, 1)
    S = DeviceSell(torch, A, env["dev"])
    v = torch.zeros(100, dtype=torch.float64, device=env["dev"])
    w = torch.zeros_like(v)
    assert lib.mg_sell_chebyshev(ctypes.byref(S.struct), v.data_ptr(), v.data_ptr(), v.data_ptr(), v.data_ptr(),
                                 v.data_ptr(), 0.5, 1.0, 0, st(env)) != 0
    assert lib.mg_sell_chebyshev(ctypes.byref(S.struct), v.data_ptr(), v.data_ptr(), v.data_ptr(), v.data_ptr(),
                                 w.data_ptr(), 0.0, 1.0, 0, st(env)) != 0


# ---- cycles ----------------------------------------------------------------------------------------------------------
def problem(case, N=64, levels=4):
    from learnmultigrid_b200 import problems as P
    coef = P.variable_coefficient if case == "variable" else None
    A = P.symmetric_dirichlet(P.structured_laplacian_2d(N, coef), P.boundary_nodes_2d(N))
    Qs = P.structured_hierarchy_2d(N, levels, transfer="quasi" if case == "quasi" else "linear")
    return A, P.structured_rhs_2d(N).ravel(), Qs


def run_cycles(h, b, x0, nu, cycles, use_graph):
    h.set_rhs(b)
    h.set_x(x0)
    params = h.make_params(nu_pre=nu, nu_post=nu)
    xs = []
    for _ in range(cycles):
        h.vcycle(params, use_graph=use_graph)
        xs.append(h.get_x().ravel().copy())
    return xs


@pytest.mark.parametrize("case", ["poisson", "quasi", "variable"])
@pytest.mark.parametrize("degree", [1, 2, 3])
@pytest.mark.parametrize("nu", [1, 2])
def test_cycle_matches_oracle(env, case, degree, nu):
    from learnmultigrid_b200.engine import DeviceHierarchy
    A, b, Qs = problem(case)
    h = DeviceHierarchy(A, Qs, smoother="chebyshev", cheby_degree=degree)
    assert len(h.cheby_coefficients) == len(Qs) and all(t.shape == (degree, 2) for t in h.cheby_coefficients)
    x0 = np.random.default_rng(7).standard_normal(A.shape[0])
    xg = run_cycles(h, b, x0, nu, 3, True)
    xe = run_cycles(h, b, x0, nu, 3, False)
    for g, e in zip(xg, xe):
        assert np.array_equal(g, e)                       # graph replay and eager launches: the same bits
    o = ChebyshevOracle(A, b, Qs, cheby_coefficients=h.cheby_coefficients, hoist_setup=True)
    o.build_hierarchy(len(Qs) + 1)
    x = x0.reshape(-1, 1)
    for got in xg:
        x = o.v_cycle(o.matrix, x, o.rhs, nu, len(Qs) + 1)
        want = x.ravel()
        assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want))


def lambda_max(A):
    s = sp.diags(1.0 / np.sqrt(A.diagonal()))
    return float(eigsh(sp.csr_matrix(s @ A @ s), k=1, which="LA", return_eigenvectors=False, tol=1e-12)[0])


@pytest.mark.parametrize("case", ["poisson", "quasi", "variable"])
def test_device_bounds_are_tight_and_deterministic(env, case):
    from learnmultigrid_b200 import formats as F
    from learnmultigrid_b200.engine import DeviceHierarchy
    A, b, Qs = problem(case)
    h1 = DeviceHierarchy(A, Qs, smoother="chebyshev")
    h2 = DeviceHierarchy(A, Qs, smoother="chebyshev")
    assert h1.cheby_lambda == h2.cheby_lambda
    Al = sp.csr_matrix(A)
    for l, Q in enumerate(Qs):
        lam = lambda_max(Al)
        assert 0.95 * lam <= h1.cheby_lambda[l] <= (1 + 1e-12) * lam
        assert h1.cheby_bounds[l] == (0.3 * h1.cheby_lambda[l], 1.1 * h1.cheby_lambda[l])
        assert np.array_equal(h1.cheby_coefficients[l], F.chebyshev_coefficients(*h1.cheby_bounds[l], 2))
        Al = sp.csr_matrix(Q.T @ Al @ Q)


def test_large_level_switches(env):
    """1025^2 (level 0 above 2^19 rows): implied columns and values are live on level 0, and cycles are the same bits
    with every switch off"""
    from learnmultigrid_b200.engine import DeviceHierarchy
    from learnmultigrid_b200 import problems as P
    lib = env["lib"]
    N = 1024
    A = P.structured_laplacian_2d(N)
    Qs = P.structured_hierarchy_2d(N, 5)
    b = P.structured_rhs_2d(N).ravel()
    h = DeviceHierarchy(A, Qs, smoother="chebyshev")
    lv0 = h.levels[0]
    assert lv0.perm is None and lv0.n > (1 << 19)
    assert lv0.A.slice_rec is not None and lv0.A.rec_vals is not None and lv0.A.val_idx is not None
    assert lv0.A.struct.nrec > 0 and lv0.A.struct.n_spec == 1
    x0 = np.random.default_rng(1).standard_normal(A.shape[0])
    on = run_cycles(h, b, x0, 1, 3, True)
    try:
        for f in (lib.mg_set_value_dict, lib.mg_set_implied_columns, lib.mg_set_implied_values):
            f(0)
        off = run_cycles(h, b, x0, 1, 3, False)
    finally:
        for f in (lib.mg_set_value_dict, lib.mg_set_implied_columns, lib.mg_set_implied_values):
            f(1)
    for a_, b_ in zip(on, off):
        assert np.array_equal(a_, b_)


@pytest.mark.parametrize("world", [2, 3, 4])
def test_partitioned_cycle_is_bit_identical_to_single_gpu(env, world):
    from learnmultigrid_b200.distributed import DistributedHierarchy, run_virtual_ranks
    from learnmultigrid_b200.engine import DeviceHierarchy
    N = 32
    A = poisson2d(N)
    Qs = [bilinear_P(N), bilinear_P(N // 2), bilinear_P(N // 4)]
    rng = np.random.default_rng(3)
    n = A.shape[0]
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    h = DeviceHierarchy(A, Qs, smoother="chebyshev")
    h.set_rhs(b)
    h.set_x(x0)
    params = h.make_params(nu_pre=1, nu_post=1)
    xs1, norms1 = [], []
    for _ in range(4):
        norms1.append(h.residual_norm())
        h.vcycle(params)
        xs1.append(h.get_x().copy())

    def body(fab):
        hd = DistributedHierarchy(A, Qs, fab, smoother="chebyshev", n_dist=2, region_bytes=1 << 20, max_sites=256,
                                  timeout_s=30.0)
        hd.set_rhs(b)
        hd.set_x(x0)
        p = hd.make_params(nu_pre=1, nu_post=1)
        xs, norms = [], []
        for it in range(4):
            if it % 2 == 0:
                norms.append(hd.residual_norm())
                hd.vcycle(p)
            else:
                hd.vcycle(p, with_norm=True)
                norms.append(hd.last_norm())
            xs.append(hd.get_x().copy())
        hd.check()
        bounds = hd.cheby_bounds
        hd.close()
        return xs, norms, bounds

    res = run_virtual_ranks(world, body)
    for xs, norms, bounds in res:
        assert bounds == h.cheby_bounds
        for got, want in zip(xs, xs1):
            assert np.array_equal(got, want)
        np.testing.assert_allclose(norms, norms1, rtol=1e-12)


def test_preconditioner_is_symmetric_and_cg_matches_oracle(env):
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.solvers.CG import CG
    from learnmultigrid_b200.solvers.Multigrid import SemiGeometricMG
    torch = env["torch"]
    N = 512
    A = P.symmetric_dirichlet(P.structured_laplacian_2d(N, P.variable_coefficient), P.boundary_nodes_2d(N))
    b = P.structured_rhs_2d(N)
    Qs = P.structured_hierarchy_2d(N, 6)
    mg = SemiGeometricMG(A, b, Qs)
    M = mg.as_preconditioner(levels=6, smoother="Chebyshev", smooth_steps=1)
    h = M.hierarchy
    n = A.shape[0]
    rng = np.random.default_rng(0)
    u, v = (torch.from_numpy(rng.standard_normal(n)).to(env["dev"]) for _ in range(2))
    Mu, Mv = torch.empty_like(u), torch.empty_like(v)
    M(u, Mu)
    M(v, Mv)
    asym = abs(float(torch.dot(u, Mv)) - float(torch.dot(v, Mu)))
    assert asym <= 1e-12 * float(torch.linalg.norm(u)) * float(torch.linalg.norm(Mv))
    cg = CG(A, b)
    cg.solve(max_iterations=200, error=1e-10, preconditioner=M)
    hist = np.asarray(cg.track_res).ravel()
    assert hist[-1] <= 1e-10
    o = ChebyshevOracle(A, b, Qs, cheby_coefficients=h.cheby_coefficients, hoist_setup=True)
    o.build_hierarchy(6)

    def precond(r):
        return o.v_cycle(o.matrix, np.zeros((n, 1)), r.reshape(-1, 1), 1, 6)
    _, want, its = pcg_solve(A, b, precond, max_iterations=200, error=1e-10)
    want = want.ravel()
    assert len(hist) == len(want)
    np.testing.assert_allclose(hist, want, rtol=1e-9, atol=1e-12 * want[0])


def test_api_solve_matches_oracle_and_honours_bounds(env):
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.solvers.Multigrid import SemiGeometricMG
    N = 64
    A = P.structured_laplacian_2d(N)
    b = P.structured_rhs_2d(N)
    Qs = P.structured_hierarchy_2d(N, 4)
    mg = SemiGeometricMG(A, b, Qs)
    mg.solve(levels=4, smoother="Chebyshev", smooth_steps=1, error=1e-9, max_iterations=40, cheby_degree=3)
    h = mg.get_hierarchy()
    assert h.smoother == "chebyshev" and h.cheby_degree == 3
    o = ChebyshevOracle(A, b, Qs, cheby_coefficients=h.cheby_coefficients, hoist_setup=True)
    o.solve(levels=4, smooth_steps=1, error=1e-9, max_iterations=40)
    assert mg.get_iterations() == len(o.track_res)
    scale = abs(A).sum(axis=1).max() * np.linalg.norm(o.solution)
    np.testing.assert_allclose(mg.track_res, o.track_res, rtol=1e-9, atol=1e-12 * scale)
    # given bounds are used as they are, and a new degree or new bounds build a new hierarchy
    bounds = [(0.2, 1.3), (0.25, 1.4), (0.3, 1.5)]
    mg.solve(levels=4, smoother="Chebyshev", smooth_steps=1, error=1e-9, max_iterations=5, cheby_bounds=bounds)
    h2 = mg.get_hierarchy()
    assert h2 is not h and h2.cheby_bounds == bounds and h2.cheby_lambda is None
    from learnmultigrid_b200 import formats as F
    for l, (lo, hi) in enumerate(bounds):
        assert np.array_equal(h2.cheby_coefficients[l], F.chebyshev_coefficients(lo, hi, 2))
    for kw in ({"cheby_degree": 0}, {"cheby_bounds": [(0.0, 1.0)] * 3}, {"cheby_bounds": [(1.0, 0.5)] * 3},
               {"cheby_bounds": [(0.1, 1.0)]}):
        with pytest.raises(ValueError):
            SemiGeometricMG(A, b, Qs).solve(levels=4, smoother="Chebyshev", max_iterations=2, **kw)
    with pytest.raises(ValueError):
        from learnmultigrid_b200.distributed import ThreadFabric
        from learnmultigrid_b200.distributed_strip import StripHierarchy
        StripHierarchy(None, [], [], ThreadFabric(1).view(0), 1, smoother="chebyshev")
