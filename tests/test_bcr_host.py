"""Host checks of the coarsest-level block cyclic reduction: the NumPy restatement (bcr_oracle) solves to SuperLU's
accuracy on every geometry the reduction can take, its geometry of the production 257^2 coarsest levels, and the
rule that decides which systems go to BcrCoarse."""
import functools

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.linalg import spsolve

import bcr_oracle as O
from learnmultigrid_b200 import _lib, coarse as C

# (n, m): n a multiple of m, n = k m + 1 (last block one real row), nb = 4, and block counts whose reduction levels
# see odd and even na at every depth
GEOMETRIES = [(240, 20), (241, 20), (61, 20), (1000, 20), (660, 20), (801, 20), (1041, 16)]


def forward_error_bound(A, xs):
    """64 eps kappa(A) max|x|, the error SuperLU and the reduction may each make on a strictly diagonally dominant
    SPD system, with kappa bounded by Gershgorin's discs"""
    d = A.diagonal()
    r = np.asarray(abs(A).sum(axis=1)).ravel() - d
    kappa = (d + r).max() / (d - r).min()
    return [64 * np.finfo(np.float64).eps * kappa * np.abs(x).max() for x in xs]


def test_geometries_cover_both_parities_at_every_depth():
    seen = {}
    for n, m in GEOMETRIES:
        for s, na in enumerate(O.geometry(n, m, min_block=1, tail_blocks=1)["na"]):
            seen.setdefault(s, set()).add(na % 2)
    assert all(seen[s] == {0, 1} for s in range(6)), seen


@functools.lru_cache(maxsize=1)
def banded_system(n, m):
    """(A, right-hand sides, SuperLU solutions, error bounds); the second right-hand side lives on the last block's
    last real row"""
    A = O.banded_spd(n, m, seed=n + m)
    rng = np.random.default_rng(1)
    bs = (rng.standard_normal(n), np.eye(n)[n - 1])
    wants = [spsolve(sp.csc_matrix(A), b) for b in bs]
    return A, bs, wants, forward_error_bound(A, wants)


@pytest.mark.parametrize("n,m", GEOMETRIES)
@pytest.mark.parametrize("tail_blocks", [1, 2, 5, 8, 16])
def test_oracle_solves_like_spsolve(n, m, tail_blocks):
    A, bs, wants, tols = banded_system(n, m)
    assert C.half_bandwidth(A.indptr, A.indices) == m
    o = O.BcrOracle(A, m, min_block=1, tail_blocks=tail_blocks)
    g = o.geometry
    assert g["nb"] == -(-n // m) and g["tail_na"] <= max(tail_blocks, 1) and all(na > tail_blocks for na in g["na"])
    assert [lv["na"] for lv in o.levels] == g["na"] and o.last_inv.shape == (g["tail_na"] * m,) * 2
    for b, want, tol in zip(bs, wants, tols):
        np.testing.assert_allclose(o.solve(b), want, rtol=0, atol=tol)


def test_oracle_min_block_and_padding_rows():
    A = O.banded_spd(130, 5, seed=3)
    o = O.BcrOracle(A, 5, min_block=32, tail_blocks=1)           # m = 32: five blocks, the last with two real rows
    assert (o.m, o.nb, o.geometry["padding"], o.geometry["na"]) == (32, 5, 30, [5, 3, 2])
    D, _, _ = O.blocks(A, 32, 5)
    assert np.array_equal(D[4, 2:, 2:], np.eye(30)) and not D[4, :2, 2:].any() and not D[4, 2:, :2].any()
    b = np.random.default_rng(0).standard_normal(130)
    want = spsolve(sp.csc_matrix(A), b)
    np.testing.assert_allclose(o.solve(b), want, rtol=0, atol=forward_error_bound(A, [want])[0])


def test_oracle_rejects_entries_outside_the_band():
    A = O.banded_spd(100, 10).tolil()
    A[0, 45] = A[45, 0] = -0.5
    with pytest.raises(ValueError, match="outside the block-tridiagonal band"):
        O.BcrOracle(sp.csr_matrix(A), 10, min_block=1)


@pytest.mark.parametrize("transfer", ["linear", "quasi"])
def test_production_coarsest_geometry(transfer):
    A = O.coarse_257(transfer)
    n = A.shape[0]
    bw = C.half_bandwidth(A.indptr, A.indices)
    assert n == 257 * 257
    g = O.geometry(n, bw, tail_blocks=C.BcrCoarse.TAIL_BLOCKS)
    assert O.geometry_row(g) == O.PRODUCTION_GEOMETRY[transfer, "natural"]
    chosen, perm = C.bcr_ordering(n, A.indptr, A.indices)
    if transfer == "linear":
        assert (chosen, perm) == (bw, None)
        assert n - (g["nb"] - 1) * g["m"] == 1                  # the last block holds a single real row
    else:
        assert perm is not None and chosen == C.permuted_half_bandwidth(A.indptr, A.indices, perm)
        g = O.geometry(n, chosen, tail_blocks=C.BcrCoarse.TAIL_BLOCKS)
        assert O.geometry_row(g) == O.PRODUCTION_GEOMETRY[transfer, "rcm"]


def test_bcr_fits_limits():
    big = 16 * 4097
    assert C.bcr_fits(big, C.BCR_MAX_BLOCK) and C.BCR_MAX_BLOCK == 4096
    assert not C.bcr_fits(big, C.BCR_MAX_BLOCK + 1)
    assert C.bcr_fits(4 * 64, 1) and not C.bcr_fits(3 * 64, 1)      # blocks of at least 64 rows, at least four
    m = C.BCR_MAX_FACTOR_BYTES // (5 * 8 * 4096 * 4096)
    assert C.bcr_fits(m * 4096, 4096) and not C.bcr_fits((m + 1) * 4096, 4096)


def test_wide_band_system_is_refused_before_block_cyclic_reduction(monkeypatch):
    """26400 unknowns of half bandwidth ~8.8k (more after RCM): four blocks of the natural band would fit the factor
    memory, but the batched inverse takes blocks of at most 4096 rows, so no BcrCoarse may be attempted"""
    A = O.layered_graph_matrix()
    A.sort_indices()
    n = A.shape[0]
    bw = C.half_bandwidth(A.indptr, A.indices)
    assert n == 26400 and C.BCR_MAX_BLOCK < bw and (n + bw - 1) // bw == 4
    assert 5 * n * bw * 8 <= C.BCR_MAX_FACTOR_BYTES and bw * bw > 4 * n
    perm = C.rcm_ordering(A.indptr, A.indices, n)
    assert C.permuted_half_bandwidth(A.indptr, A.indices, perm) >= bw

    def no_bcr(*args, **kwargs):
        raise AssertionError("BcrCoarse attempted")
    monkeypatch.setattr(C, "BcrCoarse", no_bcr)
    with pytest.raises(_lib.MgError, match="neither small enough for a dense inverse nor banded enough"):
        C.build_coarse_solver(None, None, n, None, None, None, 4096, host_pattern=(A.indptr, A.indices))
