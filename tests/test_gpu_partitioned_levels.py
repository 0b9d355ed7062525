"""GPU tests of the partitioned levels that DistributedHierarchy (row blocks cut out of the global operators) and
StripHierarchy (row blocks built by the ranks themselves) construct.

Both classes must build the same level structs, field for field, so that the cycle launches the same kernels with the
same exchange sites; mg_level.flags of a partitioned level must be those of the global operator with the global
colours, proper or not; and a partitioned cycle with an improper colouring (shortcuts off) must run and converge.
Virtual ranks on one GPU (distributed.run_virtual_ranks)."""

import numpy as np
import pytest

pytestmark = [pytest.mark.gpu]

N, LEVELS = 32, 4
COMM = dict(region_bytes=1 << 20, max_sites=256, timeout_s=30.0)


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    return torch


def _problem(transfer):
    from learnmultigrid_b200 import formats as F, problems as P
    A = F.canonical_csr(P.structured_laplacian_2d(N, P.variable_coefficient))
    Qs = [F.canonical_csr(q) for q in P.structured_hierarchy_2d(N, LEVELS, transfer)]
    ns = [A.shape[0]] + [q.shape[1] for q in Qs]
    return A, Qs, ns


def _greedy_colors(A, Qs):
    from learnmultigrid_b200.engine import DeviceHierarchy
    h = DeviceHierarchy(A, Qs, smoother="mcgs")
    return [None if c is None else np.asarray(c, dtype=np.int32).copy() for c in h.colors]


def _improper_colors(ns):
    """the colours of test_improper_colouring_switches_the_shortcuts_off: (i % 3) puts the vertical neighbours of the
    33-wide fine grid into one colour, (i % 2) the diagonal neighbours of the 7-point coarse operators"""
    return [np.arange(n, dtype=np.int32) % (3 if l == 0 else 2) for l, n in enumerate(ns[:-1])] + [None]


def _both(fab, A, Qs, ns, smoother, colors, n_dist):
    """DistributedHierarchy from the global operators, StripHierarchy from this rank's row blocks, same colours"""
    from learnmultigrid_b200 import partition as PT
    from learnmultigrid_b200.distributed import DistributedHierarchy
    from learnmultigrid_b200.distributed_strip import StripHierarchy
    r, W = fab.rank, fab.world
    offs = [PT.block_offsets(n, W) for n in ns]
    hd = DistributedHierarchy(A, Qs, fab, smoother=smoother, colors=colors, n_dist=n_dist, **COMM)
    strip_colors = None
    if colors is not None:
        strip_colors = [c if (c is None or l >= n_dist) else c[offs[l][r]:offs[l][r + 1]] for l, c in enumerate(colors)]
    hs = StripHierarchy(A[offs[0][r]:offs[0][r + 1]], [q[offs[l][r]:offs[l][r + 1]] for l, q in enumerate(Qs)], offs,
                        fab, n_dist, smoother=smoother, colors=strip_colors, **COMM)
    return hd, hs


def _np(v):
    if v is None:
        return None
    return v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)


def _xfer(x):
    k = int(x.npeers)
    return [k] + [list(getattr(x, f)[:k]) for f in ("peer", "send_off", "send_cnt", "recv_off", "recv_cnt")]


def _levels(h):
    """everything of h's levels that reaches the cycle, as host values"""
    out = {"n_dist": h.n_dist, "offsets": [np.asarray(o, dtype=np.int64) for o in h.offsets],
           "global": (list(h._global_n), list(h._global_nnzA), list(h._global_nnzQ))}
    for l, lev in enumerate(h.levels):
        d = {"n": lev.n, "perm": _np(lev.perm), "color_ptr": _np(lev.color_ptr),
             "flags": getattr(lev, "flags", None)}
        if l < h.nlevels - 1:
            d["dinv"] = _np(lev.dinv)
            d["nnz"] = (lev.nnz_A, lev.nnz_Q)
            for name in ("A", "Q", "QT"):
                M = getattr(lev, name)
                d[name] = (tuple(M.shape), M.nnz, _np(M.slice_ptr), _np(M.cols), _np(M.vals))
        else:
            d["coarse_kind"] = lev.coarse_kind
        if l < h.n_dist:
            ds = lev.dist_struct
            d["n_halo"] = lev.n_halo
            d["local_nnz_A"] = lev.local_nnz_A
            d["masks"] = [_np(m) for m in lev.masks]
            d["peers"] = list(lev.peers)
            d["send_idx"] = {q: (_np(i), list(p)) for q, (i, p) in lev.send_idx.items()}
            d["xfer"] = [_xfer(ds.xfer_color[c]) for c in range(ds.ncolors)] + [_xfer(ds.xfer_all[0])]
            if ds.xfer_gather:
                d["gather"] = (_xfer(ds.xfer_gather[0]), int(ds.n_gather_own), _np(lev.gather_iperm))
        out[l] = d
    return out


def _assert_same(a, b, path="levels"):
    if isinstance(a, dict):
        assert isinstance(b, dict) and a.keys() == b.keys(), path
        for k in a:
            _assert_same(a[k], b[k], "%s[%r]" % (path, k))
    elif isinstance(a, (list, tuple)):
        assert isinstance(b, (list, tuple)) and len(a) == len(b), path
        for k, (x, y) in enumerate(zip(a, b)):
            _assert_same(x, y, "%s[%d]" % (path, k))
    elif isinstance(a, np.ndarray):
        assert isinstance(b, np.ndarray), path
        assert a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes(), path      # bit for bit
    else:
        assert a == b, (path, a, b)


@pytest.mark.parametrize("transfer", ["linear", "quasi"])
@pytest.mark.parametrize("smoother", ["mcgs", "jacobi"])
@pytest.mark.parametrize("n_dist", [1, 2, 3])
@pytest.mark.parametrize("world", [2, 3, 4])
def test_both_classes_build_the_same_levels(torch_mod, world, n_dist, smoother, transfer):
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.distributed import run_virtual_ranks
    A, Qs, ns = _problem(transfer)
    colors = _greedy_colors(A, Qs) if smoother == "mcgs" else None
    b = P.structured_rhs_2d(N)
    x0 = np.random.default_rng(11).standard_normal((A.shape[0], 1))

    def body(fab):
        out = []
        for h in _both(fab, A, Qs, ns, smoother, colors, n_dist):
            lv = _levels(h)
            h.set_rhs(b)
            h.set_x(x0)
            h.vcycle(h.make_params(nu_pre=1, nu_post=1, omega=2.0 / 3.0), use_graph=False)
            lv["last_launches"] = h.last_launches
            lv["x"] = h.get_x().copy()
            h.check()
            h.close()
            out.append(lv)
        return out

    for got_d, got_s in run_virtual_ranks(world, body):
        assert got_d["n_dist"] == n_dist
        _assert_same(got_d, got_s)


@pytest.mark.parametrize("kind", ["greedy", "structured", "improper"])
@pytest.mark.parametrize("world", [2, 3])
def test_partitioned_flags_are_those_of_the_global_operator(torch_mod, world, kind):
    from learnmultigrid_b200 import _lib, problems as P, setup_device as SD
    from learnmultigrid_b200.distributed import run_virtual_ranks
    torch = torch_mod
    A, Qs, ns = _problem("linear")
    colors = {"greedy": lambda: _greedy_colors(A, Qs), "structured": lambda: P.structured_colors_2d(N, LEVELS),
              "improper": lambda: _improper_colors(ns)}[kind]()
    n_dist = LEVELS - 1
    S = SD.DeviceSetup(torch, torch.device("cuda", 0))
    _, A_nat, _, _ = SD.build_natural(S, A, Qs)
    want = [S.coloring_flags(A_nat[l], colors[l]) for l in range(n_dist)]
    proper = [bool(f & _lib.MG_LEVEL_PROPER_COLORING) for f in want]
    assert proper == [kind != "improper"] * n_dist           # the improper case really is improper on every level
    assert all(f & _lib.MG_LEVEL_NONZERO_DIAG for f in want)

    def body(fab):
        out = []
        for h in _both(fab, A, Qs, ns, "mcgs", colors, n_dist):
            out.append([int(lev.flags) for lev in h.levels[:n_dist]])
            h.close()
        return out

    for got_d, got_s in run_virtual_ranks(world, body):
        assert got_d == want and got_s == want


@pytest.mark.parametrize("world", [2, 3])
def test_improper_colours_in_the_partitioned_cycle(torch_mod, world):
    """A partitioned cycle with the shortcuts switched off: both classes flag the improper levels, run the cycle with
    its exchanges (no site times out) and converge.  Not compared with the single-GPU cycle bit for bit: with an
    improper colouring a colour sweep reads rows it also updates, so its result depends on which rows share a thread,
    and a halo copy always holds the value from before the sweep."""
    from learnmultigrid_b200 import _lib, problems as P
    from learnmultigrid_b200.distributed import run_virtual_ranks
    A, Qs, ns = _problem("linear")
    colors = _improper_colors(ns)
    b = P.structured_rhs_2d(N)
    n_dist = 2

    def body(fab):
        out = []
        for hp in _both(fab, A, Qs, ns, "mcgs", colors, n_dist):
            assert all(not (int(lv.flags) & _lib.MG_LEVEL_PROPER_COLORING) for lv in hp.levels[:n_dist])
            hp.set_rhs(b)
            hp.zero_x()
            p = hp.make_params(nu_pre=1, nu_post=1)
            norms = [hp.residual_norm()]
            for _ in range(4):
                hp.vcycle(p)
                norms.append(hp.residual_norm())
            hp.check()
            hp.close()
            out.append(norms)
        return out

    for per_class in run_virtual_ranks(world, body):
        for norms in per_class:
            assert all(later < earlier for earlier, later in zip(norms, norms[1:])), norms
