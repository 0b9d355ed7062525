"""GPU tests of the implied transfer columns (sell_core.cuh sell_pattern_kernel, mg_set_implied_transfers): restriction
and prolongation from slice patterns must give the SAME BITS as the kernels that read the columns, on every hierarchy
kind; hierarchies without shared patterns (quasi-L2: long rows; irregular NN meshes) carry none and run as before."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    import torch
    from learnmultigrid_b200 import _lib
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    return {"torch": torch, "lib": _lib.load(), "L": _lib}


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


@pytest.mark.parametrize("kind,N,levels,nu,reverse", [("linear", 1024, 5, 1, False), ("linear-var", 512, 4, 2, True),
                                                       ("quasi", 128, 4, 1, False), ("irregular", 32, 3, 2, False)])
def test_cycle_with_implied_transfers_is_bit_identical(env, kind, N, levels, nu, reverse):
    """implied transfers on / off (floor lowered so that every level uses them): same iterates and norms, bit for bit;
    the level-0 restriction and prolongation launches alone give the same bits too; the structured hierarchy carries
    patterns on both transfer operators, quasi-L2 and irregular ones none"""
    from learnmultigrid_b200.engine import DeviceHierarchy
    torch, lib = env["torch"], env["lib"]
    A, rhs, Qs = _problem(kind, N, levels)
    old_floor = lib.mg_set_implied_min_rows(1)
    os.environ["MGB_IMPLIED_MIN_ROWS"] = "1"
    try:
        h = DeviceHierarchy(A, Qs, smoother="mcgs")
        lev0 = h.levels[0]
        if kind == "linear":
            for T in (lev0.Q, lev0.QT):
                assert T.pat_rec is not None and T.pattern_slices > 0.7 * T.struct.nslices and T.struct.nrec < 0
        elif kind in ("quasi", "irregular"):             # long rows / unstructured numbering: no pattern anywhere
            for lv in h.levels[:-1]:
                for T in (lv.Q, lv.QT):
                    assert T.pat_rec is None and T.struct.nrec >= 0
        # (variable coefficients: the Galerkin levels' first-fit colouring scatters the coarse numbering, so patterns
        # are kept only where at least half of the slices share one -- either way the bits must not change)
        params = h.make_params(nu_pre=nu, nu_post=nu, reverse_post=reverse)
        results = {}
        for on in (0, 1):
            lib.mg_set_implied_transfers(on)
            h.drop_graphs()
            h.set_rhs(rhs)
            h.zero_x()
            xs, norms = [], []
            for _ in range(3):
                h.vcycle(params, with_norm=True)
                norms.append(h.last_norm())
                xs.append(h.levels[0].x.clone())
            h.vcycle(params, use_graph=False)
            xs.append(h.levels[0].x.clone())
            # the transfers alone, over all rows and over a range that starts inside a slice
            g = torch.Generator(device="cuda").manual_seed(5)
            r = torch.randn(lev0.n, dtype=torch.float64, device="cuda", generator=g)
            e = torch.randn(h.levels[1].n, dtype=torch.float64, device="cuda", generator=g)
            yc = torch.zeros(h.levels[1].n, dtype=torch.float64, device="cuda")
            yf = r.clone()
            st = env["L"].stream_handle(torch)
            env["L"].check(lib.mg_sell_spmv(lev0.QT.struct, r.data_ptr(), yc.data_ptr(), st), "mg_sell_spmv")
            r0 = min(37, lev0.n - 1)
            env["L"].check(lib.mg_sell_prolong_correct_rows(lev0.Q.struct, e.data_ptr(), r.data_ptr(), yf.data_ptr(),
                                                            r0, lev0.n, st), "prolong")
            torch.cuda.synchronize()
            results[on] = (xs, norms, yc, yf)
        (x0, n0, yc0, yf0), (x1, n1, yc1, yf1) = results[0], results[1]
        for a, b in zip(x0, x1):
            assert torch.equal(a, b)
        assert n0 == n1
        assert torch.equal(yc0, yc1) and torch.equal(yf0, yf1)
    finally:
        lib.mg_set_implied_transfers(1)
        lib.mg_set_implied_min_rows(old_floor)
        os.environ.pop("MGB_IMPLIED_MIN_ROWS", None)
