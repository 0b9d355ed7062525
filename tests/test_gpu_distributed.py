"""GPU parity tests of the row-partitioned V-cycle (SURVEY 8e).

The partitioned cycle must reproduce the single-GPU cycle BIT FOR BIT (same global colouring, same per-row
arithmetic; only the residual norm is summed block by block).  Most tests run `world` virtual ranks as threads on
ONE GPU (distributed.ThreadFabric): the exchange kernels, arenas and graphs are exactly the multi-process ones, only
the peers' arenas are plain pointers instead of CUDA-IPC mappings.  The torchrun test needs >= 2 GPUs.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import bilinear_P, free_port, poisson2d

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    return torch


@pytest.mark.parametrize("world", [2, 4, 7])
def test_exchange_and_allreduce_programs(torch_mod, world):
    """ring exchange with index lists + all-reduce, repeated programs (epochs, parity buffers, fence)"""
    torch = torch_mod
    from learnmultigrid_b200 import _lib
    from learnmultigrid_b200.distributed import PeerComm, run_virtual_ranks
    lib = _lib.load()
    n = 1000

    def body(fab):
        r, W = fab.rank, fab.world
        dev = torch.device("cuda", 0)
        comm = PeerComm(fab, torch, region_bytes=1 << 16, max_sites=8, timeout_s=20.0)
        st = _lib.stream_handle(torch)
        src = torch.arange(n, dtype=torch.float64, device=dev) + 1000.0 * r
        dst = torch.full((2 * n,), -1.0, dtype=torch.float64, device=dev)
        idx = torch.arange(n - 1, -1, -1, dtype=torch.int32, device=dev)          # send reversed
        left, right = (r - 1) % W, (r + 1) % W
        x = _lib.mg_xfer()
        peers = sorted({left, right})
        x.npeers = len(peers)
        for k, q in enumerate(peers):
            x.peer[k] = q
            x.d_send_idx[k] = idx.data_ptr()
            x.send_cnt[k] = n
            x.recv_off[k] = 0 if q == left else n
            x.recv_cnt[k] = n
        val = torch.zeros(1, dtype=torch.float64, device=dev)
        slots = torch.zeros(8, dtype=torch.float64, device=dev)
        out = torch.zeros(1, dtype=torch.float64, device=dev)
        sums = []
        for it in (-1, 0, 1, 2, 3, 4):
            comm.struct.dry_run = 1 if it < 0 else 0      # first pass: load the kernels (mgb200.h, mg_comm)
            if it == 0:
                torch.cuda.current_stream().synchronize()
                fab.barrier()
            val.fill_(float(r + 1) * (it + 1))
            src.add_(1.0)
            _lib.check(lib.mg_comm_begin(ctypes.byref(comm.struct)))
            _lib.check(lib.mg_comm_exchange(ctypes.byref(comm.struct), ctypes.byref(x), src.data_ptr(), dst.data_ptr(), st))
            if it % 2 == 0 or it < 0:      # odd programs have no all-pairs site: mg_comm_end adds the fence
                _lib.check(lib.mg_comm_allreduce_sum(ctypes.byref(comm.struct), val.data_ptr(), slots.data_ptr(),
                                                     out.data_ptr(), st))
            _lib.check(lib.mg_comm_end(ctypes.byref(comm.struct), st))
            torch.cuda.current_stream().synchronize()
            got = dst.cpu().numpy()
            if it < 0:
                src.sub_(1.0)
                continue
            sums.append(float(out.item()))
            base = np.arange(n - 1, -1, -1, dtype=np.float64) + (it + 1)
            if W == 2:
                assert np.array_equal(got[:n], base + 1000.0 * right)       # one peer: lands in its single slot
            else:
                assert np.array_equal(got[:n], base + 1000.0 * left)
                assert np.array_equal(got[n:], base + 1000.0 * right)
        comm.check()
        comm.close()
        return sums

    res = run_virtual_ranks(world, body)
    tot = world * (world + 1) / 2
    for sums in res:
        assert sums[0] == tot * 1 and sums[2] == tot * 3 and sums[4] == tot * 5


def _single(A, Qs, smoother, b, x0, nu, omega, cycles):
    from learnmultigrid_b200.engine import DeviceHierarchy
    h = DeviceHierarchy(A, Qs, smoother=smoother)
    h.set_rhs(b)
    h.set_x(x0)
    params = h.make_params(nu_pre=nu, nu_post=nu, omega=omega)
    xs, norms = [], []
    for _ in range(cycles):
        norms.append(h.residual_norm())
        h.vcycle(params)
        xs.append(h.get_x().copy())
    return h.colors, xs, norms


def _partitioned(world, A, Qs, smoother, colors, b, x0, nu, omega, cycles, n_dist, use_graph=True):
    from learnmultigrid_b200.distributed import DistributedHierarchy, run_virtual_ranks

    def body(fab):
        h = DistributedHierarchy(A, Qs, fab, smoother=smoother, colors=colors, n_dist=n_dist, region_bytes=1 << 20,
                                 max_sites=256, timeout_s=30.0)
        h.set_rhs(b)
        h.set_x(x0)
        params = h.make_params(nu_pre=nu, nu_post=nu, omega=omega)
        xs, norms = [], []
        for it in range(cycles):
            if it % 2 == 0:
                norms.append(h.residual_norm())
                h.vcycle(params, use_graph=use_graph)
            else:                                   # the fused outer step: norm + cycle in one program
                h.vcycle(params, use_graph=use_graph, with_norm=True)
                norms.append(h.last_norm())
            xs.append(h.get_x().copy())
        h.check()
        info = (h.n_dist, [lv.n for lv in h.levels], h.last_launches)
        h.close()
        return xs, norms, info

    return run_virtual_ranks(world, body)


@pytest.mark.parametrize("smoother,omega", [("mcgs", 1.0), ("jacobi", 2.0 / 3.0)])
@pytest.mark.parametrize("world,n_dist", [(2, 1), (2, 2), (3, 3), (4, 2)])
@pytest.mark.parametrize("nu", [1, 2])
def test_partitioned_cycle_is_bit_identical_to_single_gpu(torch_mod, smoother, omega, world, n_dist, nu):
    N = 32
    A = poisson2d(N)
    Qs = [bilinear_P(N), bilinear_P(N // 2), bilinear_P(N // 4)]
    rng = np.random.default_rng(3)
    n = A.shape[0]
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    colors, xs1, norms1 = _single(A, Qs, smoother, b, x0, nu, omega, 4)
    res = _partitioned(world, A, Qs, smoother, colors, b, x0, nu, omega, 4, n_dist)
    for xs, norms, info in res:
        assert info[0] == n_dist
        for got, want in zip(xs, xs1):
            assert np.array_equal(got, want)
        np.testing.assert_allclose(norms, norms1, rtol=1e-12)
    # every rank computed the same norm bits (summed in rank order)
    assert all(r[1] == res[0][1] for r in res)


def test_partitioned_quasi_l2_wide_halos_and_eager_mode(torch_mod):
    """19-/37-point Galerkin stencils (halo of several grid rows, > 4 colours), eager launches"""
    from learnmultigrid_b200 import problems as P
    N = 32
    A = P.structured_laplacian_2d(N, P.variable_coefficient)
    Qs = P.structured_hierarchy_2d(N, 4, transfer="quasi")
    rng = np.random.default_rng(5)
    n = A.shape[0]
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    colors, xs1, norms1 = _single(A, Qs, "mcgs", b, x0, 1, 1.0, 2)
    res = _partitioned(3, A, Qs, "mcgs", colors, b, x0, 1, 1.0, 2, 2, use_graph=False)
    for xs, norms, info in res:
        for got, want in zip(xs, xs1):
            assert np.array_equal(got, want)
        np.testing.assert_allclose(norms, norms1, rtol=1e-12)


@pytest.mark.parametrize("world", [2, 3])
def test_split_bcr_coarse_solve_is_bit_identical(torch_mod, world):
    """block cyclic reduction with its reduction levels and dense tail split over the ranks + all-gathers"""
    import scipy.sparse as sp
    torch = torch_mod
    from learnmultigrid_b200 import _lib, problems as P, formats as F, setup_device as SD
    from learnmultigrid_b200.coarse import BcrCoarse, half_bandwidth
    from learnmultigrid_b200.distributed import PeerComm, run_virtual_ranks
    lib = _lib.load()
    A = P.structured_laplacian_2d(80)
    Q = P.structured_hierarchy_2d(80, 2, transfer="linear")[0]
    Ac = F.canonical_csr(sp.csr_matrix(Q.T @ sp.csc_matrix(A) @ Q))
    n = Ac.shape[0]
    bw = half_bandwidth(Ac.indptr, Ac.indices)
    rhs = np.random.default_rng(1).standard_normal(n)

    def body(fab):
        dev = torch.device("cuda", 0)
        S = SD.DeviceSetup(torch, dev)
        Ad = S.upload(Ac)
        bcr = BcrCoarse(torch, dev, n, Ad.indptr, Ad.indices, Ad.values, bw, min_block=1, tail_blocks=5)
        d = bcr.make_dist(fab.rank, fab.world, min_blocks=4)
        assert sum(1 for s in range(32) if d.fwd_xfer[s]) >= 2 and d.tail_xfer
        comm = PeerComm(fab, torch, region_bytes=1 << 20, max_sites=64, timeout_s=30.0)
        d_rhs = torch.from_numpy(rhs).to(dev)
        x_rep = torch.zeros(n, dtype=torch.float64, device=dev)
        x_split = torch.zeros(n, dtype=torch.float64, device=dev)
        st = _lib.stream_handle(torch)
        _lib.check(lib.mg_bcr_solve(ctypes.byref(bcr.handle), d_rhs.data_ptr(), x_rep.data_ptr(), st))
        comm.struct.dry_run = 1                     # load the kernels before anybody spins (mgb200.h, mg_comm)
        _lib.check(lib.mg_bcr_solve_dist(ctypes.byref(comm.struct), ctypes.byref(bcr.handle), ctypes.byref(d),
                                         d_rhs.data_ptr(), x_split.data_ptr(), st))
        comm.struct.dry_run = 0
        torch.cuda.current_stream().synchronize()
        fab.barrier()
        for _ in range(3):
            x_split.zero_()
            _lib.check(lib.mg_bcr_solve_dist(ctypes.byref(comm.struct), ctypes.byref(bcr.handle), ctypes.byref(d),
                                             d_rhs.data_ptr(), x_split.data_ptr(), st))
            torch.cuda.current_stream().synchronize()
            assert torch.equal(x_rep, x_split)
        comm.check()
        out = x_split.cpu().numpy()
        comm.close()
        return out

    res = run_virtual_ranks(world, body)
    from scipy.sparse.linalg import spsolve
    want = spsolve(sp.csc_matrix(Ac), rhs)
    for got in res:
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-11 * np.linalg.norm(want))


def test_partitioned_cycle_with_split_bcr_coarsest_level(torch_mod):
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.engine import DeviceHierarchy
    from learnmultigrid_b200.distributed import DistributedHierarchy, run_virtual_ranks
    N = 64
    A = P.structured_laplacian_2d(N)
    Qs = P.structured_hierarchy_2d(N, 2, transfer="linear")          # coarsest = 33^2 = 1089 unknowns -> BCR
    rng = np.random.default_rng(0)
    b, x0 = rng.standard_normal(A.shape[0]), rng.standard_normal(A.shape[0])
    h1 = DeviceHierarchy(A, Qs, smoother="mcgs", dense_coarse_max=500)
    assert h1.levels[-1].coarse_kind == 1
    h1.set_rhs(b)
    h1.set_x(x0)
    p1 = h1.make_params(nu_pre=1, nu_post=1)
    want = []
    for _ in range(3):
        h1.vcycle(p1)
        want.append(h1.get_x().copy())

    def body(fab):
        h = DistributedHierarchy(A, Qs, fab, smoother="mcgs", colors=h1.colors, n_dist=1, dense_coarse_max=500,
                                 bcr_split_min_blocks=2, region_bytes=1 << 20, timeout_s=30.0)
        assert h.levels[-1].coarse_bcr_dist is not None
        h.set_rhs(b)
        h.set_x(x0)
        p = h.make_params(nu_pre=1, nu_post=1)
        got = []
        for _ in range(3):
            h.vcycle(p)
            got.append(h.get_x().copy())
        h.check()
        h.close()
        return got

    for got in run_virtual_ranks(3, body):
        for g, w in zip(got, want):
            assert np.array_equal(g, w)


def test_partitioned_api_solve_matches_oracle_history(torch_mod):
    """SemiGeometricMG.solve on a partitioned hierarchy: same iteration count and history as the CPU oracle"""
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.distributed import run_virtual_ranks
    from learnmultigrid_b200.solvers.Multigrid import SemiGeometricMG
    from oracle.vcycle import OracleMultigrid
    from helpers import assert_history_close
    N = 64
    A = P.structured_laplacian_2d(N)
    rhs = P.structured_rhs_2d(N)
    Qs = P.structured_hierarchy_2d(N, 4, transfer="linear")

    def body(fab):
        mg = SemiGeometricMG(A, rhs, Qs)
        mg.fabric = fab
        mg.dist_options = dict(n_dist=2, region_bytes=1 << 20, timeout_s=30.0)
        mg.solve(levels=4, smoother="GaussSeidel", smooth_steps=1, error=1e-9, max_iterations=30)
        out = (mg.get_iterations(), mg.track_res.copy(), mg.get_solution().copy(), mg.get_hierarchy().colors)
        mg.get_hierarchy().close()
        return out

    res = run_virtual_ranks(2, body)
    its, hist, sol, colors = res[0]
    o = OracleMultigrid(A, rhs, Qs, smoother="mcgs", colors=colors, hoist_setup=True)
    o.solve(levels=4, smooth_steps=1, error=1e-9, max_iterations=30)
    assert its == len(o.track_res)
    assert_history_close(hist, o.track_res, A, o.solution)
    np.testing.assert_allclose(sol, o.solution, rtol=0, atol=1e-12 * np.linalg.norm(o.solution))
    assert np.array_equal(res[1][2], sol)


def test_two_process_torchrun_over_cuda_ipc(torch_mod):
    """one process per GPU, arenas mapped through CUDA IPC, NVLink stores (needs >= 2 GPUs)"""
    if torch_mod.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    env = dict(os.environ, OMP_NUM_THREADS="1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", free_port(), os.path.join(ROOT, "tools", "dist_check.py"), "--size", "128"]
    out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert "DIST_CHECK_OK" in out.stdout, out.stdout[-4000:]


def test_partitioned_cycle_is_bit_identical_at_4m_dof(torch_mod):
    """larger blocks (interior CTAs really overlap the riding exchanges), automatic choice of the partitioned levels,
    structured 2/3-colourings, fused residual norm: 2049^2, 5 levels, 4 virtual ranks"""
    from learnmultigrid_b200 import problems as P
    N, L = 2048, 5
    A = P.structured_laplacian_2d(N, P.variable_coefficient)
    Qs = P.structured_hierarchy_2d(N, L, transfer="linear")
    cols = P.structured_colors_2d(N, L)
    rng = np.random.default_rng(4)
    n = A.shape[0]
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    from learnmultigrid_b200.engine import DeviceHierarchy
    from learnmultigrid_b200.distributed import DistributedHierarchy, run_virtual_ranks
    h1 = DeviceHierarchy(A, Qs, smoother="mcgs", colors=cols)
    h1.set_rhs(b)
    h1.set_x(x0)
    p1 = h1.make_params(nu_pre=1, nu_post=1)
    want, norms1 = [], []
    for _ in range(3):
        norms1.append(h1.residual_norm())
        h1.vcycle(p1)
        want.append(h1.get_x().copy())
    del h1

    def body(fab):
        h = DistributedHierarchy(A, Qs, fab, smoother="mcgs", colors=cols, timeout_s=30.0)
        h.set_rhs(b)
        h.set_x(x0)
        p = h.make_params(nu_pre=1, nu_post=1)
        got, norms = [], []
        for _ in range(3):
            h.vcycle(p, with_norm=True)
            norms.append(h.last_norm())
            got.append(h.get_x_local().copy())
        h.check()
        o = (int(h.levels[0].plan.o0), int(h.levels[0].plan.o1), h.n_dist)
        h.close()
        return got, norms, o

    for got, norms, (o0, o1, nd) in run_virtual_ranks(4, body):
        assert nd == 3                                  # 4.2 M / 1.05 M / 263 k rows: >= 65536 per rank; 66 k: replicated
        for g, w in zip(got, want):
            assert np.array_equal(g, w[o0:o1])
        np.testing.assert_allclose(norms, norms1, rtol=1e-12)
