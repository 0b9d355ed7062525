"""Singular symmetric systems on the device: the pinned coarsest solves against the NumPy/SciPy restatement of
tests/nullspace_oracle.py, cycle histories against the emulated cycle, solves at scale, right-hand sides without a
solution, preconditioners and the errors."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

import nullspace_oracle as NO
from helpers import assert_history_close
from learnmultigrid_b200 import formats as F
from learnmultigrid_b200 import problems as P

pytestmark = pytest.mark.gpu


def torch_dev():
    import torch
    return torch, torch.device("cuda", torch.cuda.current_device())


def coarse_solver(A, dense_max, shuffle=None):
    from learnmultigrid_b200.coarse import build_coarse_solver
    torch, dev = torch_dev()
    A = F.canonical_csr(sp.csr_matrix(A))
    ip, ix, va = (torch.from_numpy(a).to(dev) for a in (A.indptr, A.indices, A.data))
    return build_coarse_solver(torch, dev, A.shape[0], ip, ix, va, dense_max, (A.indptr, A.indices), singular=True)


def apply(solver, b):
    from learnmultigrid_b200.coarse import apply_coarse
    torch, dev = torch_dev()
    out = torch.empty(len(b), dtype=torch.float64, device=dev)
    apply_coarse(solver, torch.from_numpy(np.ascontiguousarray(b, dtype=np.float64)).to(dev), out)
    return out.cpu().numpy()


def galerkin_coarsest(N, levels, transfer="linear", coef=P.variable_coefficient):
    A = sp.csr_matrix(P.structured_laplacian_2d(N, coef, boundary="neumann"))
    for Q in P.structured_hierarchy_2d(N, levels, transfer=transfer)[:levels - 1]:
        A = sp.csr_matrix(Q.T @ A @ Q)
    return A


def sparse_pinned_solve(A, b, k):
    """the oracle's A+ b with a sparse LU of A_pin (sizes where a dense pinv does not fit)"""
    n = A.shape[0]
    keep = np.ones(n)
    keep[k] = 0.0
    Z = sp.diags(keep)
    A_pin = sp.csc_matrix(Z @ A @ Z + sp.csr_matrix(([1.0], ([k], [k])), shape=(n, n)))
    lu = spla.splu(A_pin)
    a_k = np.asarray(A[:, [k]].todense()).ravel() * keep
    nu = -lu.solve(a_k)
    nu[k] = 1.0
    Pj = lambda v: v - (nu @ v) / (nu @ nu) * nu
    y = lu.solve(Pj(b) * keep)
    return Pj(y), nu


@pytest.mark.parametrize("transfer", ["linear", "quasi"])
def test_dense_pseudo_inverse_matches_oracle(transfer):
    A = galerkin_coarsest(64, 4, transfer)
    s = coarse_solver(A, 4096)
    o = NO.pinned(A)
    assert s.null_info["singular"] and s.null_info["pin"] == A.shape[0] - 1
    got = s.inv.view(A.shape[0], -1).cpu().numpy()
    assert np.abs(got - o["pinv"]).max() <= 1e-12 * np.abs(o["pinv"]).max()
    assert s.null_info["verify_ratio"] <= 1e-10


@pytest.mark.parametrize("shuffle", [False, True], ids=["natural", "shuffled"])
def test_bcr_257_matches_oracle(shuffle):
    """the 257^2 coarsest operator of a 4097^2 Neumann hierarchy (6 levels, linear transfers)"""
    from learnmultigrid_b200 import problems_device as PD
    from learnmultigrid_b200.engine import DeviceHierarchy
    N = 4096
    A = PD.structured_laplacian_2d(N, PD.variable_coefficient, boundary="neumann")
    h = DeviceHierarchy(A, PD.structured_hierarchy_2d(N, 5), smoother="mcgs", null_space="constant")
    assert h.null_info["singular"] and h.levels[-1].coarse_kind == 1
    Ac = sp.csr_matrix(h.level_matrix(4))
    assert Ac.shape[0] == 257 * 257
    rng = np.random.default_rng(3)
    if shuffle:
        p = rng.permutation(Ac.shape[0])
        Ac = F.canonical_csr(sp.csr_matrix(Ac[p][:, p]))
    s = coarse_solver(Ac, 4096)
    assert (s.perm is not None) == shuffle
    b = rng.standard_normal(Ac.shape[0])
    want, nu = sparse_pinned_solve(Ac, b, s.null_pin)
    got = apply(s, b)
    # two different direct solvers (block cyclic reduction, sparse LU) of the pinned system, whose condition number is
    # ~1e5 here: measured 1.2e-12 (natural) and 1.8e-12 (shuffled) relative on B200
    assert np.abs(got - want).max() <= 1e-11 * np.abs(want).max()
    # the derived null vectors (both ~ ones: linear transfers reproduce constants) differ by 5.9e-11 (measured)
    assert np.abs(s.null.cpu().numpy() - nu).max() <= 1e-9 * np.abs(nu).max()


def test_dense_coarse_max_forces_bcr():
    A = galerkin_coarsest(128, 3)
    s = coarse_solver(A, 256)
    assert s.kind == 1 and s.null_info["singular"]
    o = NO.pinned(A)
    b = F.chebyshev_start_vector(np.arange(A.shape[0], dtype=np.int64))
    want = o["pinv"] @ b
    assert np.abs(apply(s, b) - want).max() <= 1e-12 * np.abs(want).max()


def device_history(h, b, params, cycles):
    h.set_rhs(b)
    h.project_rhs()
    h.zero_x()
    out = [h.residual_norm()]
    for _ in range(cycles):
        h.vcycle(params)
        out.append(h.residual_norm())
    return np.array(out)


@pytest.mark.parametrize("smoother", ["mcgs", "jacobi"])
@pytest.mark.parametrize("transfer", ["linear", "quasi"])
@pytest.mark.parametrize("coef", [None, P.variable_coefficient], ids=["constant", "variable"])
@pytest.mark.parametrize("dense_max", [4096, 256], ids=["dense", "bcr"])
def test_cycle_history_matches_oracle(smoother, transfer, coef, dense_max):
    from learnmultigrid_b200.engine import DeviceHierarchy
    N, L = 128, 3
    A = P.structured_laplacian_2d(N, coef, boundary="neumann")
    Qs = P.structured_hierarchy_2d(N, L, transfer=transfer)
    h = DeviceHierarchy(A, Qs, smoother=smoother, dense_coarse_max=dense_max, null_space="constant")
    b = F.chebyshev_start_vector(np.arange(A.shape[0], dtype=np.int64))
    got = device_history(h, b, h.make_params(1, 1, omega=2.0 / 3.0), 10)
    want, x = NO.stationary_history(A, Qs, np.ones(A.shape[0]), b, smoother=smoother, cycles=10)
    assert_history_close(got, want, A, x)


@pytest.mark.parametrize("smoother", ["chebyshev", "lexgs"])
@pytest.mark.parametrize("coef", [None, P.variable_coefficient], ids=["constant", "variable"])
def test_chebyshev_and_index_order_histories_match_oracle(smoother, coef):
    from learnmultigrid_b200.engine import DeviceHierarchy
    N, L = 128, 3
    A = P.structured_laplacian_2d(N, coef, boundary="neumann")
    Qs = P.structured_hierarchy_2d(N, L)
    h = DeviceHierarchy(A, Qs, smoother=smoother, null_space="constant")
    b = F.chebyshev_start_vector(np.arange(A.shape[0], dtype=np.int64))
    got = device_history(h, b, h.make_params(1, 1), 10)
    want, x = NO.oracle_history(A, Qs, b, "gs" if smoother == "lexgs" else "chebyshev", 10,
                                cheby_coefficients=h.cheby_coefficients)
    assert_history_close(got, want, A, x)


def _mass_surrogate_transfers(d, levels):
    from learnmultigrid_b200.neural2d import MassSurrogate
    from learnmultigrid_b200.solvers.Multigrid import NeuralMG_2D
    nmg = NeuralMG_2D(d["A"], d["rhs"], MassSurrogate(), d["M"], np.ones(43), np.zeros(43))
    nmg.define_hierarchy(levels)
    return [sp.csr_matrix(q) for q in nmg.l_hierarchy]


@pytest.mark.parametrize("builder", ["amg", "sa", "nn"])
def test_amg_sa_nn_histories_match_oracle(builder):
    """irregular_p1_2d(64, boundary="neumann"): SA's coarse null vector is the aggregate norms, not ones -- the case the
    derived nu_L is for"""
    import amg_oracle as AO
    import sa_oracle as SO
    from learnmultigrid_b200.engine import DeviceHierarchy
    d = P.irregular_p1_2d(64, boundary="neumann")
    A = d["A"]
    Qs = {"amg": lambda: AO.hierarchy(A, 3)[0], "sa": lambda: SO.hierarchy(A, 3)[0],
          "nn": lambda: _mass_surrogate_transfers(d, 3)}[builder]()
    h = DeviceHierarchy(A, Qs, smoother="mcgs", null_space="constant")
    assert h.null_info["singular"]
    b = d["rhs"].ravel()
    got = device_history(h, b, h.make_params(1, 1), 10)
    want, x = NO.oracle_history(A, Qs, b, "mcgs", 10, colors=h.colors)
    assert_history_close(got, want, A, x)
    assert abs(h.rhs_null_component) > 1e-3             # f = -1 with natural conditions has no solution


def scale_problem(N=2048):
    A = P.structured_laplacian_2d(N, P.variable_coefficient, boundary="neumann")
    b = F.chebyshev_start_vector(np.arange(A.shape[0], dtype=np.int64)) * 1e-3
    return A, b, P.structured_hierarchy_2d(N, 6)


def test_at_scale_stationary_and_pcg():
    from learnmultigrid_b200.solvers.Multigrid import SemiGeometricMG
    from learnmultigrid_b200.solvers.CG import CG
    A, b, Qs = scale_problem()
    Asp = sp.csr_matrix(A)
    nu = np.ones(A.shape[0])
    mg = SemiGeometricMG(A, b, Qs).set_null_space("constant")
    mg.solve(levels=6, smoother="GaussSeidel", max_iterations=40, error=1e-10)
    h = mg.get_hierarchy()
    assert h.levels[-1].coarse_kind == 1 and h.null_info["singular"]      # 65^2 coarsest: block cyclic reduction
    hist = mg.track_res.ravel()
    assert hist[-1] <= 1e-10, hist
    # the cycle count the oracle's factor predicts (the emulated cycle at N = 512, same levels and coefficient), plus one
    Ao = P.structured_laplacian_2d(512, P.variable_coefficient, boundary="neumann")
    fo = NO.factor(NO.stationary_history(Ao, P.structured_hierarchy_2d(512, 6), np.ones(Ao.shape[0]),
                                         F.chebyshev_start_vector(np.arange(Ao.shape[0], dtype=np.int64)), cycles=10)[0])
    predicted = 1 + int(np.ceil(np.log(1e-10 / hist[1]) / np.log(fo)))
    print("stationary: %d cycles, oracle factor %.3f predicts %d" % (len(hist) - 1, fo, predicted))
    assert len(hist) - 1 <= predicted + 1
    x = mg.get_solution().ravel()
    assert abs(nu @ x) <= 1e-12 * np.linalg.norm(x) * np.linalg.norm(nu)
    bp = b - (nu @ b) / (nu @ nu) * nu
    r = np.linalg.norm(bp - Asp @ x)
    assert abs(r - hist[-1]) <= 1e-3 * hist[-1] + 1e-14 * np.abs(Asp).sum(axis=1).max() * np.linalg.norm(x)
    pre = mg.as_preconditioner(levels=6, smoother="GaussSeidel")
    cg = CG(A, b)
    cg.solve(preconditioner=pre, error=1e-10, max_iterations=60)
    th = cg.track_res.ravel()
    print("PCG: %d iterations, history %s" % (len(th) - 1, th))
    assert th[-1] <= 1e-10
    assert len(th) - 1 <= predicted        # CG with the symmetric cycle needs no more steps than the cycle alone
    assert abs(mg.rhs_null_component - (nu @ b) / np.linalg.norm(nu)) <= 1e-13 * np.abs(b).sum() / np.linalg.norm(nu)
    xc = cg.get_solution().ravel()
    assert abs(nu @ xc) <= 1e-12 * np.linalg.norm(xc) * np.linalg.norm(nu)
    rc = np.linalg.norm(bp - Asp @ xc)
    assert abs(rc - th[-1]) <= 1e-2 * th[-1] + 1e-14 * np.abs(Asp).sum(axis=1).max() * np.linalg.norm(xc)


def test_inconsistent_rhs_minimum_norm_least_squares():
    from learnmultigrid_b200.solvers.Multigrid import SemiGeometricMG
    from learnmultigrid_b200.solvers.Solver import DirectSolver
    N = 32
    A = P.structured_laplacian_2d(N, boundary="neumann")
    b = P.structured_rhs_2d(N, -1.0, boundary="neumann")
    nu = np.ones(A.shape[0])
    want_c = float(nu @ b.ravel()) / np.linalg.norm(nu)
    x_ls = np.linalg.pinv(sp.csr_matrix(A).toarray(), hermitian=True) @ b.ravel()
    mg = SemiGeometricMG(A, b, P.structured_hierarchy_2d(N, 3)).set_null_space("constant")
    mg.solve(levels=3, smoother="GaussSeidel", max_iterations=60, error=1e-14)
    assert abs(mg.rhs_null_component - want_c) <= 1e-14 * abs(want_c)
    assert np.abs(mg.get_solution().ravel() - x_ls).max() <= 1e-10 * np.abs(x_ls).max()
    for dense_max in (4096, 256):
        ds = DirectSolver(A, b)
        ds.DENSE_MAX = dense_max
        ds.solve(null_space="constant")
        assert abs(ds.rhs_null_component - want_c) <= 1e-14 * abs(want_c)
        assert np.abs(ds.get_solution().ravel() - x_ls).max() <= 1e-10 * np.abs(x_ls).max()


@pytest.mark.parametrize("smoother", ["GaussSeidel", "Chebyshev"])
def test_preconditioner_symmetric_on_range(smoother):
    import torch
    from learnmultigrid_b200.solvers.Multigrid import SemiGeometricMG
    N = 64
    A = P.structured_laplacian_2d(N, P.variable_coefficient, boundary="neumann")
    n = A.shape[0]
    mg = SemiGeometricMG(A, np.zeros(n), P.structured_hierarchy_2d(N, 4)).set_null_space("constant")
    pre = mg.as_preconditioner(levels=4, smoother=smoother)
    rng = np.random.default_rng(1)
    u, v = (w - w.mean() for w in rng.standard_normal((2, n)))
    dev = pre.hierarchy.device
    Mu, Mv = torch.zeros(n, dtype=torch.float64, device=dev), torch.zeros(n, dtype=torch.float64, device=dev)
    pre(torch.from_numpy(u).to(dev), Mu)
    pre(torch.from_numpy(v).to(dev), Mv)
    a, c = float(v @ Mu.cpu().numpy()), float(u @ Mv.cpu().numpy())
    assert abs(a - c) <= 1e-12 * (abs(a) + abs(c))


def test_gmres_forward_gs():
    from learnmultigrid_b200.solvers.Multigrid import SemiGeometricMG
    from learnmultigrid_b200.solvers.GMRES import GMRES
    N = 128
    A = P.structured_laplacian_2d(N, P.variable_coefficient, boundary="neumann")
    b = P.structured_rhs_2d(N, -1.0, boundary="neumann")
    mg = SemiGeometricMG(A, b, P.structured_hierarchy_2d(N, 4)).set_null_space("constant")
    pre = mg.as_preconditioner(levels=4, smoother="GaussSeidel", symmetric=False)
    g = GMRES(A, b)
    g.solve(preconditioner=pre, error=1e-10, max_iterations=60)
    assert g.track_res[-1, 0] <= 1e-10
    x = g.get_solution().ravel()
    assert abs(x.sum()) <= 1e-12 * np.abs(x).sum()
    assert abs(pre.hierarchy.rhs_null_component) > 1e-3


def test_errors_and_reset():
    from learnmultigrid_b200 import _lib
    from learnmultigrid_b200.engine import DeviceHierarchy
    from learnmultigrid_b200.distributed_strip import StripHierarchy
    from learnmultigrid_b200.solvers.Multigrid import SemiGeometricMG
    N = 32
    Qs = P.structured_hierarchy_2d(N, 3)
    An = P.structured_laplacian_2d(N, boundary="neumann")
    with pytest.raises(ValueError, match="not one of the operator"):
        DeviceHierarchy(P.symmetric_dirichlet(P.structured_laplacian_2d(N), P.boundary_nodes_2d(N)), Qs,
                        null_space="constant")
    with pytest.raises(ValueError, match="entries"):
        DeviceHierarchy(An, Qs, null_space=np.ones(7))
    with pytest.raises(ValueError):
        SemiGeometricMG(An, np.zeros(An.shape[0]), Qs).set_null_space(np.ones(7))
    B = sp.lil_matrix(sp.csr_matrix(An))
    B[0, 1] += 0.25
    B[0, 0] -= 0.25
    with pytest.raises(ValueError, match="symmetric"):
        DeviceHierarchy(F.canonical_csr(sp.csr_matrix(B)), Qs, null_space="constant")
    T = NO.two_squares(N)
    Q2 = sp.block_diag([Qs[0], Qs[0]], format="csr")
    with pytest.raises(_lib.MgError):
        DeviceHierarchy(T, [Q2], null_space="constant")
    with pytest.raises(ValueError, match="null space"):
        StripHierarchy(None, [], [], None, 1, null_space="constant")
    from learnmultigrid_b200.solvers.CG import CG
    mgc = SemiGeometricMG(An, np.zeros(An.shape[0]), Qs).set_null_space("constant")
    pre = mgc.as_preconditioner(levels=3)
    with pytest.raises(ValueError, match="inside its hierarchy"):
        CG(An, np.zeros(An.shape[0])).solve(preconditioner=pre, initial_guess=np.zeros((An.shape[0], 1)))
    mg = SemiGeometricMG(An, P.structured_rhs_2d(N, boundary="neumann"), Qs).set_null_space("constant")
    mg.solve(levels=3, smoother="GaussSeidel", max_iterations=3)
    assert mg.get_hierarchy().null is not None
    mg.set_null_space(None).solve(levels=3, smoother="GaussSeidel", max_iterations=3)
    h = mg.get_hierarchy()
    assert h.null is None and getattr(h.levels[-1].coarse, "null", None) is None
    assert mg.rhs_null_component is None


def test_launches_and_unchanged_without_null_space():
    """null_space=None: the iterates and launch counts of a hierarchy built without the argument, bit for bit; with
    "constant" a dense coarsest launches the same kernels (A+ replaces the inverse), a BCR coarsest adds two
    projections of two launches each.  (The iterates of "constant" and of the unpinned hierarchy are not compared: the
    unpinned factor of the singular coarsest operator is what the pinned one replaces.)"""
    from learnmultigrid_b200.engine import DeviceHierarchy
    N = 128
    A = P.structured_laplacian_2d(N, boundary="neumann")
    Qs = P.structured_hierarchy_2d(N, 3)
    b = F.chebyshev_start_vector(np.arange(A.shape[0], dtype=np.int64))
    b = b - b.mean()                                         # consistent
    counts, xs = {}, {}
    for dm in (4096, 256):
        for null in ("absent", None, "constant"):
            kw = {} if null == "absent" else {"null_space": null}
            h = DeviceHierarchy(A, Qs, smoother="mcgs", dense_coarse_max=dm, **kw)
            p = h.make_params(1, 1)
            h.set_rhs(b)
            h.zero_x()
            for _ in range(3):
                h.vcycle(p)
            counts[dm, null] = h.last_launches
            xs[dm, null] = h.get_x().ravel()
    for dm in (4096, 256):
        assert counts[dm, None] == counts[dm, "absent"] and np.array_equal(xs[dm, None], xs[dm, "absent"])
    assert counts[4096, "constant"] == counts[4096, "absent"]
    assert counts[256, "constant"] == counts[256, "absent"] + 4


@pytest.mark.parametrize("coef", [None, "variable"])
def test_device_neumann_generator_matches_host(coef):
    from learnmultigrid_b200 import problems_device as PD
    from learnmultigrid_b200.setup_device import DeviceSetup
    torch, dev = torch_dev()
    for N, Ny in ((8, None), (16, 24)):
        H = sp.csr_matrix(P.structured_laplacian_2d(N, None if coef is None else P.variable_coefficient, Ny=Ny,
                                                     boundary="neumann"))
        D = DeviceSetup(torch, dev).download(PD.structured_laplacian_2d(
            N, None if coef is None else PD.variable_coefficient, Ny=Ny, boundary="neumann"))
        assert np.array_equal(D.indptr, H.indptr) and np.array_equal(D.indices, H.indices)
        if coef is None:
            assert np.array_equal(D.data, H.data)
        else:                                   # the device's sin() may differ from NumPy's in the last bit
            np.testing.assert_allclose(D.data, H.data, rtol=1e-14, atol=1e-15)


def _partitioned_null(world, A, Qs, b, colors, cycles, pcg_its):
    from learnmultigrid_b200.distributed import DistributedHierarchy, run_virtual_ranks

    def body(fab):
        h = DistributedHierarchy(A, Qs, fab, smoother="mcgs", colors=colors, n_dist=1, dense_coarse_max=500,
                                 bcr_split_min_blocks=2, region_bytes=1 << 20, timeout_s=30.0, null_space="constant")
        assert h.levels[-1].coarse_bcr_dist is not None and h.null_info["singular"]
        h.set_rhs(b)
        h.project_rhs()
        h.zero_x()
        p = h.make_params(1, 1)
        xs = []
        for _ in range(cycles):
            h.vcycle(p)
            xs.append(h.get_x().ravel().copy())
        h.project_null(h.levels[0].x)
        xs.append(h.get_x().ravel().copy())
        comp = h.rhs_null_component
        xp, track, _ = h.pcg(b, h.make_params(1, 1, reverse_post=True), error=0.0, max_iterations=pcg_its)
        xp = h.global_rows(xp)[0].ravel()
        h.check()
        h.close()
        return xs, comp, xp, track

    return run_virtual_ranks(world, body)


@pytest.mark.parametrize("world", [2, 3, 4])
def test_partitioned_bit_identical_to_one_gpu(world):
    """ThreadFabric ranks, level 0 row-partitioned, split BCR coarsest: the projected solve's iterates and x are the
    bits of one GPU; PCG's x too (its dots are summed per rank, so its history agrees to rounding)"""
    from learnmultigrid_b200.engine import DeviceHierarchy
    N = 64
    A = P.structured_laplacian_2d(N, P.variable_coefficient, boundary="neumann")
    Qs = P.structured_hierarchy_2d(N, 2)                      # coarsest 33^2 = 1089 -> BCR with dense_coarse_max 500
    b = F.chebyshev_start_vector(np.arange(A.shape[0], dtype=np.int64))
    h1 = DeviceHierarchy(A, Qs, smoother="mcgs", dense_coarse_max=500, null_space="constant")
    assert h1.levels[-1].coarse_kind == 1
    h1.set_rhs(b)
    h1.project_rhs()
    h1.zero_x()
    p1 = h1.make_params(1, 1)
    want = []
    for _ in range(3):
        h1.vcycle(p1)
        want.append(h1.get_x().ravel().copy())
    h1.project_null(h1.levels[0].x)
    want.append(h1.get_x().ravel().copy())
    comp1 = h1.rhs_null_component
    xp1, track1, _ = h1.pcg(b, h1.make_params(1, 1, reverse_post=True), error=0.0, max_iterations=6)
    xp1 = xp1.ravel()
    for xs, comp, xp, track in _partitioned_null(world, A, Qs, b, h1.colors, 3, 6):
        for got, w in zip(xs, want):
            assert np.array_equal(got, w)
        assert comp == comp1
        np.testing.assert_allclose(track, track1, rtol=1e-10)
        np.testing.assert_allclose(xp, xp1, rtol=0, atol=1e-12 * np.abs(xp1).max())
