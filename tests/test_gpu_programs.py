"""GPU tests of the program cache (engine.DeviceHierarchy._run / drop_graphs): which calls capture a CUDA graph, under
which key, and what dropping graphs does -- a recaptured program follows the library switches as they are now, the
programs of other kinds keep replaying, the bits never change."""
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    import torch
    from learnmultigrid_b200 import _lib
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    return {"torch": torch, "lib": _lib.load()}


@pytest.fixture(scope="module")
def problem():
    from learnmultigrid_b200 import problems as P
    N, levels = 64, 4
    return P.structured_laplacian_2d(N), P.structured_rhs_2d(N), P.structured_hierarchy_2d(N, levels, transfer="linear")


def handles(h, skip=None):
    """key -> graph exec handle of every cached program not of kind `skip`"""
    return {k: g[0].value for k, g in h._graphs.items() if k[0] != skip}


def test_drop_graphs_recaptures_with_the_current_switches(env, problem):
    """A stale graph keeps the fused cycle after mg_set_cycle_fusion(0); after drop_graphs() the recaptured program is
    the plain cycle, with the eager run's launch count; the iterates are the same bits throughout"""
    from learnmultigrid_b200.engine import DeviceHierarchy
    torch, lib = env["torch"], env["lib"]
    A, rhs, Qs = problem
    h = DeviceHierarchy(A, Qs, smoother="mcgs")
    assert all(int(lv.flags) == 3 for lv in h.levels[:-1])         # every level fuses
    params = h.make_params(nu_pre=1, nu_post=1)

    def cycles(use_graph=True):
        h.set_rhs(rhs)
        h.zero_x()
        xs = []
        for _ in range(3):
            h.vcycle(params, use_graph=use_graph, with_norm=True)
            xs.append(h.levels[0].x.clone())
        return xs, h.last_launches

    try:
        fused_x, fused = cycles()
        lib.mg_set_cycle_fusion(0)
        stale_x, stale = cycles()
        assert stale == fused
        h.drop_graphs()
        assert not h._graphs
        plain_x, plain = cycles()
        assert len(h._graphs) == 1
        eager_x, eager = cycles(use_graph=False)
        # coarse levels: the fused cycle replaces a fill and a sweep on the zero iterate by one launch
        assert plain == eager and plain > fused
        for xs in (stale_x, plain_x, eager_x):
            for a, b in zip(xs, fused_x):
                assert torch.equal(a, b)
    finally:
        lib.mg_set_cycle_fusion(1)


def test_drop_graphs_of_one_kind(env, problem):
    """drop_graphs("gmres") and a new restart length drop the GMRES steps only; V-cycle and PCG programs replay the
    graphs they had, with the same bits"""
    from learnmultigrid_b200.engine import DeviceHierarchy
    torch = env["torch"]
    A, rhs, Qs = problem
    h = DeviceHierarchy(A, Qs, smoother="mcgs")
    params = h.make_params(nu_pre=1, nu_post=1, reverse_post=True)

    def run(restart=30):
        h.set_rhs(rhs)
        h.zero_x()
        h.vcycle(params)
        x = h.levels[0].x.clone()
        cg = h.pcg(rhs, params, error=0.0, max_iterations=5)
        gm = h.gmres(rhs, params, error=0.0, max_iterations=6, restart=restart)
        return x, cg, gm

    def same(r1, r2):
        (x1, (c1, ct1, ci1), (g1, gt1, gi1, gr1)), (x2, (c2, ct2, ci2), (g2, gt2, gi2, gr2)) = r1, r2
        assert torch.equal(x1, x2)
        assert (c1 == c2).all() and ct1 == ct2 and ci1 == ci2
        assert (g1 == g2).all() and gt1 == gt2 and gi1 == gi2 and gr1 == gr2

    first = run()
    kinds = sorted(k[0] for k in h._graphs)
    assert kinds == ["gmres"] * 6 + ["pcg"] * 2 + ["vcycle"]
    others = handles(h, skip="gmres")
    size = len(h._graphs)
    h.drop_graphs("gmres")
    assert handles(h) == others
    same(first, run())
    assert len(h._graphs) == size and handles(h, skip="gmres") == others
    run(restart=4)
    assert handles(h, skip="gmres") == others
    assert sorted(k[1] for k in h._graphs if k[0] == "gmres") == [0, 1, 2, 3]      # steps of GMRES(4) only


def test_index_order_gauss_seidel_is_not_captured(env, problem):
    """cooperative launches cannot be captured: with a lexgs preconditioner PCG and GMRES run uncaptured; without a
    preconditioner nothing of it is in the program and CG is captured"""
    from learnmultigrid_b200.engine import DeviceHierarchy
    A, rhs, Qs = problem
    h = DeviceHierarchy(A, Qs, smoother="lexgs")
    params = h.make_params(nu_pre=1, nu_post=1)
    _, _, its = h.pcg(rhs, params, error=0.0, max_iterations=4)
    assert its == 4
    _, track, its, _ = h.gmres(rhs, params, error=0.0, max_iterations=4)
    assert its == 4 and track[-1] < track[0]
    assert not h._graphs
    h.pcg(rhs, None, error=0.0, max_iterations=2)
    assert sorted(k[:2] for k in h._graphs) == [("pcg", 0), ("pcg", 1)]


def test_partitioned_programs_are_cached_per_key(env, problem):
    """on two virtual ranks the cycle with its norm and its dry twin are two programs; a repeated call replays;
    close() empties the cache"""
    from learnmultigrid_b200.distributed import DistributedHierarchy, run_virtual_ranks
    A, rhs, Qs = problem

    def body(fab):
        hd = DistributedHierarchy(A, Qs, fab, smoother="mcgs", n_dist=2, region_bytes=1 << 20, max_sites=512,
                                  timeout_s=30.0)
        p = hd.make_params(nu_pre=1, nu_post=1)
        hd.set_rhs(rhs)
        hd.zero_x()
        hd.vcycle(p, norm_after=True)
        hd.vcycle(p, norm_after=True, dry=True)
        cached = handles(hd)
        hd.vcycle(p, norm_after=True)
        hd.check()
        again = handles(hd)
        hd.close()
        return cached, again, len(hd._graphs)

    for cached, again, left in run_virtual_ranks(2, body):
        assert again == cached and len(cached) == 2
        assert all(k[0] == "vcycle_dist" for k in cached)
        assert sorted(k[3] for k in cached) == [False, True]          # the dry field
        assert left == 0
