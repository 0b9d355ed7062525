"""Restarted GMRES on the device: the Krylov kernels against NumPy float64, DeviceHierarchy.gmres against the NumPy
oracle (tests/gmres_oracle.py) for every preconditioner kind, GMRES.solve through the public API, and partitioned runs
against one GPU."""
import numpy as np
import pytest

from gmres_oracle import gmres as oracle_gmres

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    import torch
    from learnmultigrid_b200 import _lib
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    return {"torch": torch, "lib": _lib.load(), "L": _lib, "dev": torch.device("cuda", 0)}


def up(env, a):
    return env["torch"].from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(env["dev"])


def stream(env):
    return env["torch"].cuda.current_stream().cuda_stream


def basis(rng, m, n):
    """m vectors of n entries at a stride ld > n (the columns of the device's column-major basis)"""
    ld = (n + 31) // 32 * 32 + 32
    V = np.zeros((m, ld))
    V[:, :n] = rng.uniform(0.5, 1.5, (m, n))
    return V, ld


@pytest.mark.parametrize("n", [1, 255, 257, 1000003])
def test_krylov_kernels_against_numpy(env, n):
    L, lib, torch = env["L"], env["lib"], env["torch"]
    rng = np.random.default_rng(n)
    for m in (1, 7, 8, 9, 17, 31):
        V, ld = basis(rng, m, n)
        w = rng.uniform(0.5, 1.5, n)
        dV, dw = up(env, V.ravel()), up(env, w)
        parts = torch.zeros(int(lib.mg_krylov_partials(n, m)), dtype=torch.float64, device=env["dev"])
        outs = []
        for _ in range(2):
            out = torch.full((m,), np.nan, dtype=torch.float64, device=env["dev"])
            L.check(lib.mg_multi_dot(n, dV.data_ptr(), ld, m, dw.data_ptr(), parts.data_ptr(), out.data_ptr(),
                                     stream(env)), "mg_multi_dot")
            outs.append(out.cpu().numpy())
        assert np.array_equal(outs[0], outs[1])
        np.testing.assert_allclose(outs[0], V[:, :n] @ w, rtol=1e-13)

        h = rng.uniform(-1.0, 1.0, m)
        want = w.copy()
        for k in range(m):
            want = want - h[k] * V[k, :n]
        res = []
        for _ in range(2):
            dw2 = up(env, w)
            nrm = torch.zeros(1, dtype=torch.float64, device=env["dev"])
            dh = up(env, h)                          # held: a temporary's block would be reused by the next upload
            L.check(lib.mg_multi_axpy_norm(n, dV.data_ptr(), ld, m, dh.data_ptr(), dw2.data_ptr(),
                                           parts.data_ptr(), nrm.data_ptr(), stream(env)), "mg_multi_axpy_norm")
            res.append((dw2.cpu().numpy(), float(nrm.item())))
        assert np.array_equal(res[0][0], want)                              # every operation rounded as in NumPy
        assert res[0][1] == res[1][1] and np.array_equal(res[0][0], res[1][0])
        np.testing.assert_allclose(res[0][1], want @ want, rtol=1e-13)

        # back substitution and update: R y = g, x += sum y_c z_c
        k = m
        H = np.zeros((k, k + 1))                                             # column-major (k + 1) x k
        for c in range(k):
            H[c, :c + 1] = rng.uniform(-1.0, 1.0, c + 1)
            H[c, c] = rng.uniform(1.0, 2.0) * (1 if c % 2 else -1)
        g = rng.uniform(-1.0, 1.0, k + 1)
        x = rng.uniform(-1.0, 1.0, n)
        y = np.zeros(k)
        for i in range(k - 1, -1, -1):
            acc = g[i]
            for c in range(i + 1, k):
                acc = acc - H[c, i] * y[c]
            y[i] = acc / H[i, i]
        xw = x.copy()
        for c in range(k):
            xw = xw + y[c] * V[c, :n]
        dx, dy = up(env, x), torch.zeros(k + 1, dtype=torch.float64, device=env["dev"])
        dH, dg = up(env, H.ravel()), up(env, g)
        L.check(lib.mg_gmres_solve_update(n, dH.data_ptr(), k + 1, dg.data_ptr(), k,
                                          dy.data_ptr(), dV.data_ptr(), ld, dx.data_ptr(), stream(env)),
                "mg_gmres_solve_update")
        assert np.array_equal(dy.cpu().numpy()[:k], y)
        assert np.array_equal(dx.cpu().numpy(), xw)

    # scale, including the lucky breakdown h = 0
    v = rng.standard_normal(n)
    for hv in (3.7, 0.0):
        dv, dh = up(env, v), up(env, [hv])
        L.check(lib.mg_scale_inv(n, dh.data_ptr(), dv.data_ptr(), stream(env)), "mg_scale_inv")
        got = dv.cpu().numpy()
        assert np.array_equal(got, v / hv if hv else v) and np.isfinite(got).all()


# ---- DeviceHierarchy.gmres against the oracle ----------------------------------------------------------------------
def oracle_precond(A, b, Qs, L, h, kind):
    from oracle.vcycle import OracleMultigrid
    from chebyshev_oracle import ChebyshevOracle
    if kind is None:
        return None
    if kind == "chebyshev":
        o = ChebyshevOracle(A, b, Qs, cheby_coefficients=h.cheby_coefficients, hoist_setup=True)
    else:
        o = OracleMultigrid(A, b, Qs, smoother={"mcgs": "mcgs", "lexgs": "gs", "jacobi": "jacobi"}[kind],
                            omega=2.0 / 3.0, colors=h.colors, hoist_setup=True)
    o.build_hierarchy(L)
    n = A.shape[0]
    return lambda v: o.v_cycle(o.matrix, np.zeros((n, 1)), v, 1, L)


def check_against_oracle(A, b, Qs, h, kind, restart, error, max_iterations, x0=None):
    L = len(Qs) + 1
    params = None if kind is None else h.make_params(nu_pre=1, nu_post=1, omega=2.0 / 3.0)
    x, hist, its, res = h.gmres(b, params, error=error, max_iterations=max_iterations, restart=restart, x0=x0)
    xo, ho, io, ro = oracle_gmres(A, b, oracle_precond(A, b, Qs, L, h, kind), error=error,
                                  max_iterations=max_iterations, restart=restart, x0=x0)
    assert its == io, (kind, restart, its, io)
    np.testing.assert_allclose(hist, ho, rtol=1e-6)
    np.testing.assert_allclose(x, xo, rtol=0, atol=1e-9 * np.linalg.norm(xo))
    assert res == pytest.approx(np.linalg.norm(b - A @ x), rel=1e-6, abs=1e-14 * np.linalg.norm(b))
    x2, hist2, its2, res2 = h.gmres(b, params, error=error, max_iterations=max_iterations, restart=restart, x0=x0)
    assert its2 == its and hist2 == hist and np.array_equal(x, x2) and res2 == res      # graphs replayed: same bits
    return its, hist, res


@pytest.fixture(scope="module")
def vc129():
    from learnmultigrid_b200 import problems as P
    N, L = 128, 5
    A = P.structured_laplacian_2d(N, P.variable_coefficient)                # row-Dirichlet: nonsymmetric
    return A, P.structured_rhs_2d(N), P.structured_hierarchy_2d(N, L, transfer="linear")


@pytest.mark.parametrize("restart", [30, 4])
def test_device_gmres_forward_gauss_seidel(env, vc129, restart):
    from learnmultigrid_b200.engine import DeviceHierarchy
    A, b, Qs = vc129
    h = DeviceHierarchy(A, Qs, smoother="mcgs")
    its, hist, res = check_against_oracle(A, b, Qs, h, "mcgs", restart, 1e-10, 200)
    assert res <= 1e-10 and its < 30
    if restart == 4:
        assert its > 4                                                       # several restarts


@pytest.mark.parametrize("kind", [None, "chebyshev", "lexgs", "jacobi"])
def test_device_gmres_other_preconditioners(env, vc129, kind):
    from learnmultigrid_b200.engine import DeviceHierarchy
    A, b, Qs = vc129
    h = DeviceHierarchy(A, Qs, smoother="mcgs" if kind is None else kind)
    if kind is None:
        # Unpreconditioned, this operator's Krylov sequence turns rounding-sensitive after ~21 steps: the oracle against
        # itself with exactly rounded dots (math.fsum) differs by 5e-7 at 30 steps and 5e-6 at 120, by 2e-11 over these
        # 20 steps with two restarts.  Beyond that no summation order is the right one to compare with.
        its, hist, res = check_against_oracle(A, b, Qs, h, kind, 8, 1e-10, 20)
        assert its == 20 and hist[-1] < hist[0]
    else:
        its, hist, res = check_against_oracle(A, b, Qs, h, kind, 30, 1e-10, 200)
        assert res <= 1e-10


def test_device_gmres_nonzero_initial_guess(env, vc129):
    from learnmultigrid_b200.engine import DeviceHierarchy
    A, b, Qs = vc129
    h = DeviceHierarchy(A, Qs, smoother="mcgs")
    x0 = np.random.default_rng(5).standard_normal((A.shape[0], 1)) * 1e-3
    its, hist, res = check_against_oracle(A, b, Qs, h, "mcgs", 30, 1e-10, 200, x0=x0)
    assert hist[0] == pytest.approx(np.linalg.norm(b - A @ x0), rel=1e-12) and res <= 1e-10


def test_device_gmres_convection_diffusion_with_amg(env):
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.solvers.Multigrid import AlgebraicMG
    N, L = 64, 4
    A = P.convection_diffusion_2d(N, 0.01, (1.0, 0.5))
    b = P.structured_rhs_2d(N)
    mg = AlgebraicMG(A, b)
    M = mg.as_preconditioner(levels=L, smoother="GaussSeidel", symmetric=False)
    Qs = [mg._ab().download(q) for q in mg.l_hierarchy]
    its, hist, res = check_against_oracle(A, b, Qs, M.hierarchy, "mcgs", 30, 1e-10, 300)
    assert res <= 1e-10


def test_device_gmres_refuses_bad_restart_and_huge_bases(env, vc129):
    from learnmultigrid_b200.engine import DeviceHierarchy
    A, b, Qs = vc129
    h = DeviceHierarchy(A, Qs, smoother="mcgs")
    with pytest.raises(ValueError, match="restart"):
        h.gmres(b, None, restart=0)
    free, _ = env["torch"].cuda.mem_get_info()
    with pytest.raises(ValueError, match="bytes"):
        h.gmres(b, None, restart=int(free // (16 * A.shape[0])) + 10)


# ---- public API ----------------------------------------------------------------------------------------------------
def api_problems():
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.neural2d import MassSurrogate
    from learnmultigrid_b200.solvers.Multigrid import AlgebraicMG, NeuralMG_2D, SemiGeometricMG, SmoothedAggregationMG
    N = 64
    A = P.structured_laplacian_2d(N, P.variable_coefficient)
    b = P.structured_rhs_2d(N)
    Qs = P.structured_hierarchy_2d(N, 4, transfer="linear")
    C = P.convection_diffusion_2d(N, 0.01, (1.0, -0.5))
    pb = P.irregular_p1_2d(32, seed=3)
    nn = NeuralMG_2D(pb["A"], pb["rhs"], MassSurrogate(), pb["M"], np.ones(43), np.zeros(43))
    nn.define_hierarchy(levels=3)
    return [("sgmg", A, b, SemiGeometricMG(A, b, Qs), 4), ("amg", C, b, AlgebraicMG(C, b), 4),
            ("sa", C, b, SmoothedAggregationMG(C, b), 4), ("nn", pb["A"], pb["rhs"], nn, 3)]


def test_gmres_solve_through_the_api(env):
    from learnmultigrid_b200.solvers.GMRES import GMRES
    from learn_multigrid.solvers.GMRES import GMRES as Alias
    assert Alias is GMRES
    for name, A, b, mg, levels in api_problems():
        for smoother in ("GaussSeidel", "Chebyshev"):
            M = mg.as_preconditioner(levels=levels, smoother=smoother, symmetric=False)
            s = GMRES(A, b)
            s.solve(error=1e-9, preconditioner=M, restart=30)
            x = s.get_solution() if hasattr(s, "get_solution") else s.solution
            true = np.linalg.norm(b - A @ x)
            assert true <= 1e-9 and s.residual == pytest.approx(true, rel=1e-6, abs=1e-15), (name, smoother)
            np.testing.assert_allclose(s.residual_vector, b - A @ x, rtol=0, atol=1e-12 * np.linalg.norm(b))
            first = s.iterations
            assert 0 < first == len(s.track_res) - 1
            s.solve(error=1e-9, preconditioner=M, restart=30, initial_guess=np.zeros_like(b))
            assert s.iterations == 2 * first
            # out of steps: the iterate of the last completed step, with its true residual
            s2 = GMRES(A, b)
            s2.solve(error=1e-30, max_iterations=3, preconditioner=M, restart=30)
            assert s2.iterations == 3 and len(s2.track_res) == 4
            assert s2.residual == pytest.approx(np.linalg.norm(b - A @ s2.solution), rel=1e-6)
            # zero right-hand side: nothing to do
            s3 = GMRES(A, np.zeros_like(b))
            s3.solve(preconditioner=M)
            assert s3.iterations == 0 and not s3.solution.any()
        s = GMRES(A, b)
        with pytest.raises(ValueError, match="preconditioner"):
            s.solve(preconditioner=None)
        with pytest.raises(ValueError, match="restart"):
            s.solve(preconditioner=M, restart=0)
    # a preconditioner of another matrix
    A2 = A.copy()
    A2.data = A2.data * 2.0
    with pytest.raises(ValueError, match="preconditioner"):
        GMRES(A2, b).solve(preconditioner=M)


# ---- partitioned ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("restart", [30, 4])
def test_device_gmres_single_and_partitioned(env, vc129, restart):
    """Same steps, histories to rtol 1e-7 -- down to the rounding floor 1e-14 ||b|| of an estimate that starts from a
    residual b - A x recomputed at a restart (its entries carry rounding of order u ||b||, summed in another order
    over the row blocks) --, the rank's rows of x to 1e-10 ||x||"""
    from learnmultigrid_b200.distributed import DistributedHierarchy, run_virtual_ranks
    from learnmultigrid_b200.engine import DeviceHierarchy
    A, b, Qs = vc129
    h = DeviceHierarchy(A, Qs, smoother="mcgs")
    params = h.make_params(nu_pre=1, nu_post=1)
    x, hist, its, res = h.gmres(b, params, error=1e-10, max_iterations=200, restart=restart)
    assert res <= 1e-10
    for world in (2, 3):
        def body(fab):
            hd = DistributedHierarchy(A, Qs, fab, smoother="mcgs", colors=h.colors, n_dist=2, region_bytes=1 << 20,
                                      max_sites=512, timeout_s=30.0)
            pd = hd.make_params(nu_pre=1, nu_post=1)
            xl, hl, il, rl = hd.gmres(b, pd, error=1e-10, max_iterations=200, restart=restart)
            hd.check()
            o0, o1 = int(hd.offsets[0][fab.rank]), int(hd.offsets[0][fab.rank + 1])
            hd.close()
            return xl, hl, il, rl, o0, o1
        for xl, hl, il, rl, o0, o1 in run_virtual_ranks(world, body):
            assert il == its
            np.testing.assert_allclose(hl, hist, rtol=1e-7, atol=1e-14 * np.linalg.norm(b))
            np.testing.assert_allclose(xl, x[o0:o1], rtol=0, atol=1e-10 * np.linalg.norm(x))
            assert rl <= 1e-10
