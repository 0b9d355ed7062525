"""GPU tests of the work the multicolour cycle no longer does (csrc/cycle.cu g_cycle_fusion, sell_core.cuh GS_RES /
GS_NORM, implied columns as the default): every shortcut must leave the SAME BITS as the operation-by-operation cycle,
which the other GPU tests pin to the CPU oracle."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import kernels as K

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    import torch
    from learnmultigrid_b200 import _lib
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    return {"torch": torch, "lib": _lib.load(), "L": _lib, "dev": torch.device("cuda", 0)}


def up(env, a):
    return env["torch"].from_numpy(np.ascontiguousarray(a)).to(env["dev"])


def st(env):
    return env["L"].stream_handle(env["torch"])


def banded(n, per_row, seed, uniform):
    """symmetric-pattern matrix with about `per_row` entries per row and a dominant diagonal; uniform: every row has
    exactly the same number of entries (the SELL builder then stores it 'uniform')"""
    from learnmultigrid_b200 import formats as F
    rng = np.random.default_rng(seed)
    if uniform:
        offs = np.unique(np.concatenate([[0], rng.integers(1, 3 * per_row, size=per_row // 2)]))
        offs = np.concatenate([-offs[:0:-1], offs])
        rows = np.repeat(np.arange(n), len(offs))
        cols = (rows + np.tile(offs, n)) % n
    else:
        rows = np.repeat(np.arange(n), per_row)
        cols = (rows + rng.integers(-3 * per_row, 3 * per_row + 1, size=rows.size)) % n
    M = sp.csr_matrix((rng.standard_normal(rows.size), (rows, cols)), shape=(n, n))
    M = M + M.T + sp.diags(rng.uniform(3.0, 5.0, n) * per_row)
    return F.canonical_csr(M)


@pytest.mark.parametrize("n,per_row,uniform", [(900, 2, False), (40000, 4, True), (40000, 5, False), (3000, 7, False),
                                                (5000, 16, False), (5000, 30, True), (700, 90, False)])
def test_sweep_with_fused_residual_and_norm_is_the_residual_pass(env, n, per_row, uniform):
    """mg_sell_gs_rows_tail on every colour of a proper colouring == mg_sell_gs_rows followed by mg_sell_residual, bit
    for bit (short rows: thread-per-row kernel; 9..64 entries: warps-per-slice kernel; longer: not offered)"""
    from learnmultigrid_b200 import formats as F
    from learnmultigrid_b200.engine import DeviceSell
    L, lib, torch = env["L"], env["lib"], env["torch"]
    A = banded(n, per_row, n + per_row, uniform)
    rng = np.random.default_rng(1)
    colors, nc = F.greedy_colors(A)
    perm, cptr = F.color_permutation(colors)
    iperm = F.inverse_permutation(perm)
    Ap = F.permute_csr(A, perm, iperm)
    S = DeviceSell(torch, Ap, env["dev"])
    x, b = rng.standard_normal(n), rng.standard_normal(n)
    ws = torch.zeros(int(lib.mg_norm_workspace_size(n)) + 8, dtype=torch.float64, device=env["dev"])
    for c in range(nc):
        r0, r1 = int(cptr[c]), int(cptr[c + 1])
        ok = lib.mg_sell_gs_tail_ok(ctypes.byref(S.struct), r0, r1)
        if S.max_len > 64:
            assert not ok
            rc = lib.mg_sell_gs_rows_tail(ctypes.byref(S.struct), 0, 0, r0, r1, 1, ws.data_ptr(), None, None, st(env))
            assert rc != 0 and b"too long" in lib.mg_last_error()
            continue
        assert ok
        x1, x2, x3 = up(env, x), up(env, x), up(env, x)
        db = up(env, b)
        L.check(lib.mg_sell_gs_rows(ctypes.byref(S.struct), x1.data_ptr(), db.data_ptr(), r0, r1, st(env)))
        r_ref = torch.empty(n, dtype=torch.float64, device=env["dev"])
        L.check(lib.mg_sell_residual(ctypes.byref(S.struct), x1.data_ptr(), db.data_ptr(), r_ref.data_ptr(), st(env)))
        r = torch.full((n,), 7.0, dtype=torch.float64, device=env["dev"])
        L.check(lib.mg_sell_gs_rows_tail(ctypes.byref(S.struct), x2.data_ptr(), db.data_ptr(), r0, r1, 1, r.data_ptr(),
                                         None, None, st(env)))
        assert torch.equal(x1, x2)
        assert torch.equal(r[r0:r1], r_ref[r0:r1])
        assert bool((r[:r0] == 7.0).all()) and bool((r[r1:] == 7.0).all())        # nothing outside the colour
        # the oracle's residual on the same iterate (the chain GPU sweep == oracle sweep is test_gpu_parity's)
        assert np.array_equal(r_ref.cpu().numpy(), K.residual(Ap, x1.cpu().numpy(), b))
        nb = ctypes.c_int(0)
        L.check(lib.mg_sell_gs_rows_tail(ctypes.byref(S.struct), x3.data_ptr(), db.data_ptr(), r0, r1, 2, None,
                                         ws.data_ptr(), ctypes.byref(nb), st(env)))
        assert torch.equal(x1, x3) and nb.value > 0
        # only the NORM is asked of this mode: the swept rows have just been solved, their residual is rounding noise
        # (formed with one FMA, not in storage order), so what is checked is its share of ||b - A x||^2
        got = float(ws[:nb.value].sum().item())
        rest = float((r_ref[:r0] ** 2).sum().item() + (r_ref[r1:] ** 2).sum().item())
        total = float((r_ref ** 2).sum().item())
        np.testing.assert_allclose(got + rest, total, rtol=1e-13)
        assert 0.0 <= got <= 1e-24 * max(total, 1.0) * (r1 - r0)
        # residual of the remaining rows by the row-range entry: the two halves make the full residual
        L.check(lib.mg_sell_residual_rows(ctypes.byref(S.struct), x2.data_ptr(), db.data_ptr(), r.data_ptr(), 0, r0, st(env)))
        L.check(lib.mg_sell_residual_rows(ctypes.byref(S.struct), x2.data_ptr(), db.data_ptr(), r.data_ptr(), r1, n, st(env)))
        assert torch.equal(r, r_ref)


def test_rows_with_zero_or_missing_diagonal_keep_their_value_and_their_residual(env):
    from learnmultigrid_b200 import formats as F
    from learnmultigrid_b200.engine import DeviceSell
    L, lib, torch = env["L"], env["lib"], env["torch"]
    n = 2000
    A = banded(n, 4, 5, False).tolil()
    for i in (3, 700, 1999):
        A[i, i] = 0.0
    A = F.canonical_csr(sp.csr_matrix(A))          # explicit zeros are dropped: rows without a diagonal entry
    colors, nc = F.greedy_colors(A)
    perm, cptr = F.color_permutation(colors)
    Ap = F.permute_csr(A, perm, F.inverse_permutation(perm))
    S = DeviceSell(torch, Ap, env["dev"])
    rng = np.random.default_rng(2)
    x, b = rng.standard_normal(n), rng.standard_normal(n)
    db = up(env, b)
    for c in range(nc):
        r0, r1 = int(cptr[c]), int(cptr[c + 1])
        x1, x2 = up(env, x), up(env, x)
        L.check(lib.mg_sell_gs_rows(ctypes.byref(S.struct), x1.data_ptr(), db.data_ptr(), r0, r1, st(env)))
        r_ref = torch.empty(n, dtype=torch.float64, device=env["dev"])
        L.check(lib.mg_sell_residual(ctypes.byref(S.struct), x1.data_ptr(), db.data_ptr(), r_ref.data_ptr(), st(env)))
        r = torch.zeros(n, dtype=torch.float64, device=env["dev"])
        L.check(lib.mg_sell_gs_rows_tail(ctypes.byref(S.struct), x2.data_ptr(), db.data_ptr(), r0, r1, 1, r.data_ptr(),
                                         None, None, st(env)))
        assert torch.equal(x1, x2) and torch.equal(r[r0:r1], r_ref[r0:r1])
    # the inspection reports the missing diagonals and that the greedy colouring is proper
    flag = torch.zeros(1, dtype=torch.int32, device=env["dev"])
    diag = torch.empty(n, dtype=torch.float64, device=env["dev"])
    cp = up(env, np.asarray(cptr, dtype=np.int64))
    L.check(lib.mg_level_inspect(ctypes.byref(S.struct), nc, cp.data_ptr(), diag.data_ptr(), flag.data_ptr(), st(env)))
    assert int(flag.item()) == 2
    assert np.array_equal(diag.cpu().numpy(), Ap.diagonal())
    # two coupled rows in one colour: not proper
    bad = np.asarray(cptr, dtype=np.int64).copy()
    bad[1] = bad[2]                                # merge colours 0 and 1
    flag.zero_()
    dbad = up(env, bad)
    L.check(lib.mg_level_inspect(ctypes.byref(S.struct), nc, dbad.data_ptr(), None, flag.data_ptr(), st(env)))
    assert int(flag.item()) & 1


def test_first_sweep_on_a_zero_iterate_without_the_matrix(env):
    from learnmultigrid_b200 import formats as F
    from learnmultigrid_b200.engine import DeviceSell
    L, lib, torch = env["L"], env["lib"], env["torch"]
    n = 5000
    A = banded(n, 5, 9, False)
    colors, nc = F.greedy_colors(A)
    perm, cptr = F.color_permutation(colors)
    Ap = F.permute_csr(A, perm, F.inverse_permutation(perm))
    S = DeviceSell(torch, Ap, env["dev"])
    b = np.random.default_rng(3).standard_normal(n)
    b[int(cptr[0]) + 5] = -0.0
    db = up(env, b)
    want = torch.zeros(n + 17, dtype=torch.float64, device=env["dev"])            # 17 halo entries behind the rows
    L.check(lib.mg_sell_gs_rows(ctypes.byref(S.struct), want.data_ptr(), db.data_ptr(), 0, int(cptr[1]), st(env)))
    got = torch.full((n + 17,), 3.0, dtype=torch.float64, device=env["dev"])
    dd = up(env, Ap.diagonal())
    L.check(lib.mg_sell_gs_zero_first(n + 17, 0, int(cptr[1]), dd.data_ptr(), db.data_ptr(), got.data_ptr(), st(env)))
    assert np.array_equal(got.cpu().numpy().view(np.int64), want.cpu().numpy().view(np.int64))    # signs of zero too


def _problem(kind, N, levels):
    from learnmultigrid_b200 import problems as P
    if kind == "irregular":
        pb = P.irregular_p1_2d(N, seed=7)
        from learnmultigrid_b200.neural2d import MassSurrogate
        from learnmultigrid_b200.solvers.Multigrid import NeuralMG_2D
        nmg = NeuralMG_2D(pb["A"], pb["rhs"], MassSurrogate(), pb["M"], np.ones(43), np.zeros(43))
        nmg.define_hierarchy(levels)
        return pb["A"], pb["rhs"], nmg.l_hierarchy
    coef = P.variable_coefficient if kind.endswith("var") else None
    A = P.structured_laplacian_2d(N, coef)
    return A, P.structured_rhs_2d(N), P.structured_hierarchy_2d(N, levels, transfer=kind.split("-")[0])


@pytest.mark.parametrize("kind,N,levels,nu,reverse", [("linear", 64, 4, 1, False), ("linear-var", 96, 4, 2, True),
                                                       ("quasi", 64, 3, 1, False), ("quasi", 128, 4, 2, True),
                                                       ("irregular", 32, 3, 3, False), ("linear", 1024, 5, 1, False)])
def test_fused_cycle_is_bit_identical_to_the_plain_cycle(env, kind, N, levels, nu, reverse):
    """g_cycle_fusion on/off, implied columns on/off (floor lowered so that small levels use them), value dictionary
    on/off, implied values on/off: same iterates, bit for bit, cycle after cycle; the norm the fused cycle leaves equals
    the stand-alone residual norm to rounding"""
    from learnmultigrid_b200.engine import DeviceHierarchy
    lib = env["lib"]
    A, rhs, Qs = _problem(kind, N, levels)
    old_floor = lib.mg_set_implied_min_rows(1)
    import os
    os.environ["MGB_IMPLIED_MIN_ROWS"] = "1"
    os.environ["MGB_VALUE_DICT_MIN_ROWS"] = "1"
    try:
        h = DeviceHierarchy(A, Qs, smoother="mcgs")
        flags = [int(getattr(lv, "flags", 0)) for lv in h.levels[:-1]]
        assert all(f == 3 for f in flags), flags                 # proper colouring, no zero diagonal: everything fuses
        if kind.startswith("linear") and N >= 512:               # (on small grids every slice holds a boundary node)
            assert h.levels[0].A.slice_off is not None           # structured stencil level: implied columns attached
            # ... and, the coefficient being constant, value records: the regular slices read nothing but their id
            assert (h.levels[0].A.rec_vals is not None) == (kind == "linear")
            if kind == "linear":
                assert h.levels[0].A.regular_slices > 0.9 * h.levels[0].A.struct.nslices
        params = h.make_params(nu_pre=nu, nu_post=nu, reverse_post=reverse)
        results = {}
        for fusion, implied, vdict, impv in ((0, 0, 0, 1), (1, 0, 0, 1), (0, 1, 0, 1), (1, 1, 0, 1), (0, 0, 1, 1),
                                             (1, 1, 1, 1), (1, 1, 1, 0), (0, 1, 1, 0)):
            if True:
                lib.mg_set_cycle_fusion(fusion)
                lib.mg_set_implied_columns(implied)
                lib.mg_set_value_dict(vdict)
                lib.mg_set_implied_values(impv)
                h.drop_graphs()
                h.set_rhs(rhs)
                h.zero_x()
                xs, norms = [], []
                for _ in range(3):
                    h.vcycle(params, with_norm=True)
                    norms.append(h.last_norm())
                    xs.append(h.levels[0].x.clone())
                    np.testing.assert_allclose(norms[-1], h.residual_norm(), rtol=1e-12)
                h.vcycle(params, use_graph=False)                # eager, without the norm
                xs.append(h.levels[0].x.clone())
                results[(fusion, implied, vdict, impv)] = (xs, norms, h.last_launches)
        base = results[(0, 0, 0, 1)]
        for key, (xs, norms, _) in results.items():
            for a, b_ in zip(xs, base[0]):
                assert env["torch"].equal(a, b_), key
        assert norms[-1] < norms[0]
        # the fused cycle launches no more kernels than the plain one
        assert results[(1, 1, 1, 1)][2] <= results[(0, 0, 0, 1)][2]
        if kind in ("linear", "linear-var"):                       # linear interpolation: {1, 0.5, 0} -> dictionaries
            assert h.levels[0].Q.val_idx is not None and h.levels[0].Q.distinct_values <= 4
            assert (h.levels[0].A.val_idx is not None) == (kind == "linear")    # variable coefficients: too many values
    finally:
        lib.mg_set_cycle_fusion(1)
        lib.mg_set_implied_columns(1)
        lib.mg_set_value_dict(1)
        lib.mg_set_implied_values(1)
        lib.mg_set_implied_min_rows(old_floor)
        os.environ.pop("MGB_IMPLIED_MIN_ROWS", None)
        os.environ.pop("MGB_VALUE_DICT_MIN_ROWS", None)


def test_preconditioner_application_from_an_uninitialised_iterate(env):
    """x0_zero: z = M^-1 r without zeroing z first == the cycle on a zeroed iterate"""
    from learnmultigrid_b200.engine import DeviceHierarchy
    torch = env["torch"]
    A, rhs, Qs = _problem("linear-var", 64, 4)
    h = DeviceHierarchy(A, Qs, smoother="mcgs")
    for sm_params in (dict(nu_pre=1, nu_post=1, reverse_post=True), dict(nu_pre=2, nu_post=2)):
        h.set_rhs(rhs)
        h.zero_x()
        h.vcycle(h.make_params(**sm_params))
        want = h.levels[0].x.clone()
        h.levels[0].x.fill_(float("nan"))
        h.vcycle(h.make_params(x0_zero=True, **sm_params))
        assert torch.equal(h.levels[0].x, want)
    hj = DeviceHierarchy(A, Qs, smoother="jacobi")
    for nu in (1, 2):
        hj.set_rhs(rhs)
        hj.zero_x()
        hj.vcycle(hj.make_params(nu_pre=nu, nu_post=nu, omega=0.8))
        want = hj.levels[0].x.clone()
        hj.levels[0].x.fill_(float("nan"))
        hj.levels[0].tmp.fill_(float("nan"))
        hj.vcycle(hj.make_params(nu_pre=nu, nu_post=nu, omega=0.8, x0_zero=True))
        assert torch.equal(hj.levels[0].x, want)


def test_improper_colouring_switches_the_shortcuts_off(env):
    """colours that put coupled rows into one block: the level is flagged and the cycle falls back to one pass per
    operation (the fused and the plain setting then launch the same kernels)"""
    from learnmultigrid_b200.engine import DeviceHierarchy
    lib = env["lib"]
    A, rhs, Qs = _problem("linear", 32, 3)
    n0, n1 = A.shape[0], Qs[0].shape[1]
    colors = [np.arange(n0, dtype=np.int32) % 3, np.arange(n1, dtype=np.int32) % 2, None]
    h = DeviceHierarchy(A, Qs, smoother="mcgs", colors=colors)
    assert all(not (int(lv.flags) & 1) for lv in h.levels[:-1])
    params = h.make_params(nu_pre=1, nu_post=1)
    counts = []
    for fusion in (0, 1):
        lib.mg_set_cycle_fusion(fusion)
        h.set_rhs(rhs)
        h.zero_x()
        h.vcycle(params, use_graph=False)
        counts.append(h.last_launches)
    lib.mg_set_cycle_fusion(1)
    assert counts[1] <= counts[0] <= counts[1] + len(h.levels)      # only the zero-guess shortcut may differ


def test_norm_workspace_covers_the_wide_kernel(env):
    """ADVICE r1: a 27-entry operator of ~200 k rows runs the eight-warps-per-slice kernel, one partial per 32 rows; the
    documented workspace must hold them (guard values behind it stay untouched)"""
    from learnmultigrid_b200.engine import DeviceSell
    L, lib, torch = env["L"], env["lib"], env["torch"]
    n = 200_000
    A = banded(n, 27, 4, True)
    S = DeviceSell(torch, A, env["dev"])
    assert 21 <= S.max_len <= 64
    rng = np.random.default_rng(0)
    x, b = rng.standard_normal(n), rng.standard_normal(n)
    size = int(lib.mg_norm_workspace_size(n))
    ws = torch.full((size + 4096,), -123.0, dtype=torch.float64, device=env["dev"])
    nrm = torch.zeros(1, dtype=torch.float64, device=env["dev"])
    dx, db = up(env, x), up(env, b)
    L.check(lib.mg_sell_residual_norm2(ctypes.byref(S.struct), dx.data_ptr(), db.data_ptr(), ws.data_ptr(),
                                       nrm.data_ptr(), st(env)))
    np.testing.assert_allclose(np.sqrt(nrm.item()), np.linalg.norm(b - A @ x), rtol=1e-13)
    assert bool((ws[size:] == -123.0).all())


@pytest.mark.parametrize("rpt", [2, 4])
def test_short_row_kernel_is_bit_identical(env, rpt):
    """transfer operators with one or two entries per row: R rows per thread (sell_short_kernel) against the oracle, whole
    matrix and row ranges that start and end inside a slice, out of place and in place"""
    from learnmultigrid_b200 import formats as F, problems as P
    from learnmultigrid_b200.engine import DeviceSell
    L, lib, torch = env["L"], env["lib"], env["torch"]
    Q = F.canonical_csr(P.linear_P_2d(96))
    onecol = F.canonical_csr(sp.csr_matrix((np.arange(1.0, 3001.0), (np.arange(3000), np.arange(3000) % 77)), shape=(3000, 77)))
    old_r, old_min = lib.mg_set_short_rows_per_thread(rpt), lib.mg_set_short_min_rows(0)
    try:
        for M in (Q, onecol):
            S = DeviceSell(torch, M, env["dev"])
            assert 1 <= S.max_len <= 2
            rng = np.random.default_rng(5)
            e, u = rng.standard_normal(M.shape[1]), rng.standard_normal(M.shape[0])
            de, du = up(env, e), up(env, u)
            out = torch.empty(M.shape[0], dtype=torch.float64, device=env["dev"])
            L.check(lib.mg_sell_spmv(ctypes.byref(S.struct), de.data_ptr(), out.data_ptr(), st(env)))
            assert np.array_equal(out.cpu().numpy(), K.spmv(M, e))
            L.check(lib.mg_sell_prolong_correct(ctypes.byref(S.struct), de.data_ptr(), du.data_ptr(), out.data_ptr(), st(env)))
            want = K.prolong_correct(M, e, u)
            assert np.array_equal(out.cpu().numpy(), want)
            for r0, r1 in ((0, 1), (37, M.shape[0] - 45), (513, 1301), (M.shape[0] - 1, M.shape[0])):
                part = up(env, u)                                   # in place on a row range
                L.check(lib.mg_sell_prolong_correct_rows(ctypes.byref(S.struct), de.data_ptr(), part.data_ptr(),
                                                         part.data_ptr(), r0, r1, st(env)))
                got = part.cpu().numpy()
                assert np.array_equal(got[r0:r1], want[r0:r1])
                assert np.array_equal(got[:r0], u[:r0]) and np.array_equal(got[r1:], u[r1:])
    finally:
        lib.mg_set_short_rows_per_thread(old_r)
        lib.mg_set_short_min_rows(old_min)


def test_device_pcg_single_and_partitioned(env):
    """BASELINE configs[4] on the device-side iteration (mg_pcg_start / mg_pcg_iterate: scalars on the device, p.Ap from
    the SpMV, r.r from the update, one graph per iteration): against the CPU oracle's PCG, and row-partitioned over 2 and
    3 virtual ranks against the single-GPU run (same iteration count, histories to rounding of the dot products)"""
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.distributed import DistributedHierarchy, run_virtual_ranks
    from learnmultigrid_b200.engine import DeviceHierarchy
    from oracle.vcycle import OracleMultigrid, pcg_solve
    N, L = 128, 5
    A = P.symmetric_dirichlet(P.structured_laplacian_2d(N, P.variable_coefficient), P.boundary_nodes_2d(N))
    rhs = P.structured_rhs_2d(N)
    Qs = P.structured_hierarchy_2d(N, L, transfer="linear")
    h = DeviceHierarchy(A, Qs, smoother="mcgs")
    params = h.make_params(nu_pre=1, nu_post=1, reverse_post=True)
    x, hist, its = h.pcg(rhs, params, error=1e-10, max_iterations=60)
    o = OracleMultigrid(A, rhs, Qs, smoother="mcgs", colors=h.colors, hoist_setup=True, reverse_post=True)
    o.build_hierarchy(L)
    n = A.shape[0]
    xo, ho, io = pcg_solve(A, rhs, lambda r: o.v_cycle(o.matrix, np.zeros((n, 1)), r, 1, L), 60, 1e-10)
    assert its == io and its < 15
    np.testing.assert_allclose(hist, np.asarray(ho).ravel(), rtol=1e-6)
    np.testing.assert_allclose(x, xo, rtol=0, atol=1e-9 * np.linalg.norm(xo))
    x2, hist2, its2 = h.pcg(rhs, params, error=1e-10, max_iterations=60)          # graphs replayed: same bits
    assert its2 == its and hist2 == hist and np.array_equal(x, x2)
    # plain CG through the same device iteration
    xc, hc, ic = h.pcg(rhs, None, error=1e-8, max_iterations=2000)
    assert ic > 5 * its and hc[-1] <= 1e-8
    np.testing.assert_allclose(xc, xo, rtol=0, atol=1e-6 * np.linalg.norm(xo))

    for world in (2, 3):
        def body(fab):
            hd = DistributedHierarchy(A, Qs, fab, smoother="mcgs", colors=h.colors, n_dist=2, region_bytes=1 << 20,
                                      max_sites=512, timeout_s=30.0)
            pd = hd.make_params(nu_pre=1, nu_post=1, reverse_post=True)
            xl, hl, il = hd.pcg(rhs, pd, error=1e-10, max_iterations=60)
            hd.check()
            o0, o1 = int(hd.offsets[0][fab.rank]), int(hd.offsets[0][fab.rank + 1])
            hd.close()
            return xl, hl, il, o0, o1
        for xl, hl, il, o0, o1 in run_virtual_ranks(world, body):
            assert il == its
            np.testing.assert_allclose(hl, hist, rtol=1e-7)
            np.testing.assert_allclose(xl, x[o0:o1], rtol=0, atol=1e-10 * np.linalg.norm(x))


def test_value_dictionary_kernels_are_bit_identical(env):
    """csrc/valdict.cu: a matrix with few distinct values is re-encoded as one byte per entry + table, every SELL mode
    gives the bits of the ordinary kernels (which the other tests pin to the oracle); a matrix with more than 256
    distinct values gets no dictionary; -0.0 and +0.0 are different entries"""
    from learnmultigrid_b200 import formats as F
    from learnmultigrid_b200.engine import DeviceSell
    L, lib, torch = env["L"], env["lib"], env["torch"]
    import os
    os.environ["MGB_VALUE_DICT_MIN_ROWS"] = "1"
    try:
        rng = np.random.default_rng(12)
        for n, per_row, uniform, nvals in ((30000, 5, True, 7), (30000, 1, False, 200), (9000, 1, False, 250), (9000, 2, True, 3)):
            A = banded(n, per_row, n + nvals, uniform)
            pool = np.concatenate([rng.standard_normal(nvals - 2), [-0.0, 0.5]])
            A.data[:] = pool[rng.integers(0, nvals, size=A.nnz)]
            A = sp.csr_matrix(A)
            A.setdiag(40.0)                                            # a diagonal that dominates (entries exist already)
            A = F.raw_csr(A.indptr.astype(np.int32), A.indices.astype(np.int32), A.data, A.shape)
            colors, nc = F.greedy_colors(A)
            perm, cptr = F.color_permutation(colors)
            Ap = F.permute_csr(A, perm, F.inverse_permutation(perm))
            S = DeviceSell(torch, Ap, env["dev"])
            assert S.val_idx is not None and S.distinct_values <= 256
            tab = S.val_table.cpu().numpy()
            assert np.array_equal(tab[S.val_idx.cpu().numpy().astype(np.int64)].view(np.int64),
                                  S.vals.cpu().numpy().view(np.int64))              # lossless, signs of zero included
            x, b, u = rng.standard_normal(n), rng.standard_normal(n), rng.standard_normal(n)
            ws = torch.zeros(int(lib.mg_norm_workspace_size(n)) + 8, dtype=torch.float64, device=env["dev"])
            outs = {}
            for use in (0, 1):
                lib.mg_set_value_dict(use)
                dx, db, du = up(env, x), up(env, b), up(env, u)
                y = torch.empty(n, dtype=torch.float64, device=env["dev"])
                r = torch.empty(n, dtype=torch.float64, device=env["dev"])
                xj = torch.empty(n, dtype=torch.float64, device=env["dev"])
                nrm = torch.zeros(1, dtype=torch.float64, device=env["dev"])
                dd = up(env, 1.0 / Ap.diagonal())
                L.check(lib.mg_sell_spmv(ctypes.byref(S.struct), dx.data_ptr(), y.data_ptr(), st(env)))
                L.check(lib.mg_sell_residual(ctypes.byref(S.struct), dx.data_ptr(), db.data_ptr(), r.data_ptr(), st(env)))
                L.check(lib.mg_sell_residual_norm2(ctypes.byref(S.struct), dx.data_ptr(), db.data_ptr(), ws.data_ptr(),
                                                   nrm.data_ptr(), st(env)))
                L.check(lib.mg_sell_jacobi(ctypes.byref(S.struct), dd.data_ptr(), dx.data_ptr(), db.data_ptr(),
                                           xj.data_ptr(), 0.7, st(env)))
                L.check(lib.mg_sell_prolong_correct(ctypes.byref(S.struct), dx.data_ptr(), du.data_ptr(), du.data_ptr(), st(env)))
                xg = up(env, x)
                rt = torch.zeros(n, dtype=torch.float64, device=env["dev"])
                for c in range(nc):
                    L.check(lib.mg_sell_gs_rows_tail(ctypes.byref(S.struct), xg.data_ptr(), db.data_ptr(), int(cptr[c]),
                                                     int(cptr[c + 1]), 1, rt.data_ptr(), None, None, st(env)))
                outs[use] = [t.clone() for t in (y, r, nrm, xj, du, xg, rt)]
            lib.mg_set_value_dict(1)
            for a_, b_ in zip(outs[0], outs[1]):
                assert torch.equal(a_, b_)
            assert np.array_equal(outs[1][0].cpu().numpy(), K.spmv(Ap, x))
        many = banded(20000, 5, 3, False)                              # random values: far more than 256 distinct
        S = DeviceSell(torch, many, env["dev"])
        assert S.val_idx is None and not S.struct.d_val_idx
    finally:
        lib.mg_set_value_dict(1)
        os.environ.pop("MGB_VALUE_DICT_MIN_ROWS", None)
