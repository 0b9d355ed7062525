"""tests/setup_oracle.py (the host reference of the device setup) pinned to formats' torch functions on host tensors, on
small inputs with the edges that matter at scale: a partial last slice, an all-irregular matrix, more than 256 slice
patterns, ties in frequency, the 9/10 value-carrying threshold on both sides, and 256 / 257 distinct values with +0.0
and -0.0 as distinct entries."""
import ctypes

import numpy as np
import pytest

import setup_oracle as O
from learnmultigrid_b200 import _lib
from learnmultigrid_b200 import formats as F
from learnmultigrid_b200 import problems as P
from learnmultigrid_b200.engine import DeviceSell

torch = pytest.importorskip("torch")


@pytest.fixture
def small_floors(monkeypatch):
    """the attach rules at test sizes: every matrix is above the row floors"""
    monkeypatch.setattr(DeviceSell, "VALUE_DICT_MIN_ROWS", 1)
    monkeypatch.setattr(DeviceSell, "IMPLIED_MIN_ROWS", 2)


def synthetic(cols, vals, nrows, ncols):
    """oracle SELL dict of a uniform matrix given as [nslices, L, 32] columns and values"""
    nsl, L, _ = cols.shape
    return {"slice_ptr": np.arange(nsl + 1, dtype=np.int64) * 32 * L, "cols": np.ascontiguousarray(cols, np.int32).ravel(),
            "vals": np.ascontiguousarray(vals, np.float64).ravel(), "max_len": L, "uniform_len": L, "nrows": nrows,
            "shape": (nrows, ncols)}


def product_slice_records(s, with_dict):
    """formats.slice_records on host tensors, fed as DeviceSell feeds it: kernel offsets (host twin), dictionary"""
    L = s["uniform_len"]
    nsl = len(s["slice_ptr"]) - 1
    off = np.zeros((nsl, 8), dtype=np.int32)
    off[:, :L] = F.sell_slice_offsets((s["slice_ptr"], s["cols"], s["vals"]), s["nrows"], L)
    vi = vt = None
    if with_dict:
        bits, inv = np.unique(s["vals"].view(np.int64), return_inverse=True)
        vi = torch.from_numpy(inv.reshape(-1).astype(np.uint8))
        vt = torch.from_numpy(np.concatenate([bits, np.zeros(256 - len(bits), np.int64)]).view(np.float64))
    ids, table, rvals, nreg = F.slice_records(torch, torch.from_numpy(off), vi, vt, L)
    return ids.numpy(), table.numpy(), None if rvals is None else rvals.numpy(), nreg


def fake_sell(n, L):
    """a DeviceSell shell (no device data) whose spec-block methods can run on host tensors"""
    d = DeviceSell.__new__(DeviceSell)
    d.shape = (n, n)
    d.struct = _lib.mg_sell(n, n, (n + 31) // 32, 0, 0, 0, L, L)
    return d


def spec_arrays(st, nb):
    rows = [st.h_spec_row[k] for k in range(nb + 1)]
    rec = [st.h_spec_rec[k] for k in range(9 * nb)]
    vals = None if not st.h_spec_vals else np.array([st.h_spec_vals[k] for k in range(8 * nb)])
    return rows, rec, vals


@pytest.mark.parametrize("coef", [None, P.variable_coefficient])
def test_slice_records_and_spec_blocks_of_a_colour_blocked_operator(small_floors, coef):
    """257^2 rows (partial last slice of one row) in first-fit colour order: constant coefficients carry values,
    variable ones have no dictionary and carry columns only; the spec blocks name a most used record per colour"""
    A = F.canonical_csr(P.structured_laplacian_2d(256, coef))
    col, _ = O.colors(A)
    perm, iperm, cptr = O.permutation(col)
    s = O.sell(A, perm, iperm)
    assert s["nrows"] % 32 == 1 and s["uniform_len"] == 5
    d = O.value_dict(s)
    assert d["attached"] == (coef is None)
    ref = O.slice_records(s, d["attached"])
    assert ref["attached"] and ref["with_values"] == (coef is None)
    assert ref["group"][-1] == -1                                  # the one-row slice is never regular
    ids, table, rvals, nreg = product_slice_records(s, d["attached"])
    O.check_slice_records(ref, s, ids, table, rvals)
    assert nreg == int((ref["group"] >= 0).sum())
    sh = fake_sell(s["nrows"], 5)
    sh.slice_rec, sh.rec_table = torch.from_numpy(ids), torch.from_numpy(table)
    sh.rec_vals = None if rvals is None else torch.from_numpy(rvals)
    sh.set_spec_blocks(cptr)
    O.check_offset_spec_blocks(cptr, *spec_arrays(sh.struct, len(cptr) - 1), ids, table, rvals)
    # a record that resolves to other columns, a dropped record, unordered ids: each is caught
    for bad in ("cols", "drop", "order"):
        i2, t2 = ids.copy(), table.copy()
        if bad == "cols":
            t2[0, 1] += 1
        elif bad == "drop":
            i2[np.nonzero(i2 >= 0)[0][3]] = -1
        else:
            z = len(t2) - 1                                        # the most and the least used record swap ids
            t2[[0, z]] = t2[[z, 0]]
            i2 = np.where(i2 == 0, z, np.where(i2 == z, 0, i2)).astype(i2.dtype)
        with pytest.raises(AssertionError):
            O.check_slice_records(ref, s, i2, t2, rvals)


@pytest.mark.parametrize("uniform", [18, 17])
def test_value_carrying_threshold_both_sides(small_floors, uniform):
    """20 column-regular slices: values are carried when at least 18 of them (nine tenths) hold one value per entry"""
    nsl, L = 20, 2
    rows = np.arange(nsl * 32).reshape(nsl, 1, 32)
    cols = np.concatenate([rows - 1, rows + 3], axis=1) + 8
    vals = np.ones((nsl, L, 32))
    vals[:, 1] = -0.5
    vals[uniform:, 0, 7] = 2.0                     # one lane differs: column-regular, not value-regular
    s = synthetic(cols, vals, nsl * 32, nsl * 32 + 16)
    ref = O.slice_records(s, True)
    assert ref["with_values"] == (uniform == 18)
    ids, table, rvals, _ = product_slice_records(s, True)
    assert (rvals is not None) == (uniform == 18)
    O.check_slice_records(ref, s, ids, table, rvals)


def test_all_irregular_matrix_keeps_no_records(small_floors):
    """columns at random: no slice is regular, no two slices share a pattern -- neither record kind is attached"""
    rng = np.random.default_rng(5)
    nsl, L = 40, 3
    cols = rng.integers(0, 5000, (nsl, L, 32))
    vals = rng.standard_normal((nsl, L, 32))
    for shape in ((nsl * 32, nsl * 32), (nsl * 32 - 5, 5000)):
        s = synthetic(cols, vals, shape[0], shape[1])
        ref = O.slice_records(s, False)
        assert ref["attempted"] and not ref["attached"] and ref["regular_columns"] == 0
        pr = O.pattern_records(s, False)
        assert pr["attempted"] == (shape[0] != shape[1]) and not pr["attached"]
        if pr["attempted"]:
            *_, nreg = F.pattern_records(torch, torch.from_numpy(s["cols"]), torch.from_numpy(s["vals"]), shape[0], L)
            assert nreg == pr["slices"] == 0


@pytest.mark.parametrize("layout", ["ties", "ranked"])
def test_more_than_256_patterns(small_floors, layout):
    """ties: 300 patterns used by two slices each (the 256-record cutoff falls inside a tie); ranked: 256 patterns used
    3..6 times and 44 used twice (the cutoff falls between counts); both with unique slices and a partial last slice"""
    rng = np.random.default_rng(11)
    npat, L = 300, 2
    use = np.full(npat, 2) if layout == "ties" else np.where(np.arange(npat) < 256, 3 + np.arange(npat) % 4, 2)
    which = rng.permutation(np.concatenate([np.repeat(np.arange(npat), use), npat + np.arange(50)]))
    nsl = len(which) + 1
    deltas = rng.integers(0, 40, (npat + 50, L, 32))
    pv = rng.integers(-3, 3, (npat + 50, L, 32)) * 0.25
    base = rng.integers(0, 10000, nsl)
    cols = np.concatenate([base[:-1, None, None] + deltas[which], np.full((1, L, 32), 7)])
    vals = np.concatenate([pv[which], np.zeros((1, L, 32))])
    cols[-1, 0, 0] = base[-1]
    s = synthetic(cols, vals, nsl * 32 - 20, 10100)
    ref = O.pattern_records(s, False)
    assert not ref["sampled"] and len(ref["kept"]) == 256
    assert (ref["cutoff"] is not None) == (layout == "ties")
    b, ids, delta, pvals, nreg = F.pattern_records(torch, torch.from_numpy(s["cols"]), torch.from_numpy(s["vals"]),
                                                   s["nrows"], L)
    assert nreg == ref["slices"] and ref["attached"] == (2 * nreg >= nsl)
    O.check_pattern_records(ref, s, ids.numpy(), delta.numpy(), pvals.numpy(), b.numpy())
    # pattern spec blocks: 11 blocks, capped at 8 with the last absorbing the rest
    sh = fake_sell(s["nrows"], L)
    sh.pat_rec = ids
    row_ptr = np.linspace(0, s["nrows"], 12).astype(np.int64)
    sh.set_pattern_blocks(row_ptr)
    nb = sh.struct.n_spec
    assert nb == 8
    rows, rec, _ = spec_arrays(sh.struct, nb)
    O.check_pattern_spec_blocks(row_ptr, rows, rec, ids.numpy(), ref["group"])
    rec[9 * 2 + 1] += 1
    with pytest.raises(AssertionError):
        O.check_pattern_spec_blocks(row_ptr, rows, rec, ids.numpy(), ref["group"])
    # a kept record split off from its group is caught
    i2 = ids.numpy().copy()
    i2[np.nonzero(i2 == 0)[0][0]] = -1
    with pytest.raises(AssertionError):
        O.check_pattern_records(ref, s, i2, delta.numpy(), pvals.numpy(), b.numpy())


def test_sampled_pattern_decision(small_floors):
    """more than 2 x 4096 slices: the evenly spaced sample decides first -- structured slices pass it, a matrix whose
    sampled slices share nothing is skipped although its other slices all share one pattern"""
    nsl, L = 2 * DeviceSell.PATTERN_SAMPLE + 100, 1
    cols = np.zeros((nsl, L, 32), dtype=np.int64) + np.arange(32)
    vals = np.ones((nsl, L, 32))
    s = synthetic(cols + np.arange(nsl)[:, None, None], vals, nsl * 32, nsl * 32 + 64)
    ref = O.pattern_records(s, False)
    assert ref["sampled"] and ref["sample_slices"] == DeviceSell.PATTERN_SAMPLE and ref["attached"]
    pick = O.pattern_sample(nsl)
    vals2 = vals.copy()
    vals2[pick, 0, 0] = np.arange(len(pick)) + 2.0
    s2 = synthetic(cols, vals2, nsl * 32, nsl * 32 + 64)
    ref2 = O.pattern_records(s2, False)
    assert ref2["sampled"] and ref2["sample_slices"] == 0 and not ref2["attached"]
    tp = torch.linspace(0, nsl - 2, DeviceSell.PATTERN_SAMPLE).long().numpy()        # the product's picks
    assert np.abs(tp - pick).max() <= 1
    sc = torch.from_numpy(np.ascontiguousarray(cols.reshape(nsl, -1)[tp], np.int32).ravel())
    sv = torch.from_numpy(np.ascontiguousarray(vals2.reshape(nsl, -1)[tp]).ravel())
    *_, nreg = F.pattern_records(torch, sc, sv, DeviceSell.PATTERN_SAMPLE * 32, L)
    assert 2 * nreg < DeviceSell.PATTERN_SAMPLE


@pytest.mark.parametrize("distinct", [256, 257])
def test_value_dict_256_and_257_distinct_values(distinct):
    """+0.0 and -0.0 are distinct entries (the padding is +0.0): 256 distinct values take a dictionary, 257 do not;
    a dictionary that decodes -0.0 as +0.0 is caught"""
    n = DeviceSell.VALUE_DICT_MIN_ROWS
    v = np.concatenate([[0.0, -0.0], 1.0 + np.arange(distinct - 2)])
    vals = np.resize(v, (n // 32, 2, 32))
    s = synthetic(np.zeros((n // 32, 2, 32)), vals, n, n)
    ref = O.value_dict(s)
    assert ref["count"] == distinct and ref["attached"] == (distinct <= 256)
    if not ref["attached"]:
        O.check_value_dict(ref, s, None, None, None)
        return
    bits, inv = np.unique(s["vals"].view(np.int64), return_inverse=True)
    table = np.zeros(256, dtype=np.int64)
    table[:len(bits)] = bits
    idx = inv.reshape(-1).astype(np.uint8)
    O.check_value_dict(ref, s, idx, table.view(np.float64), distinct)
    merged = idx.copy()
    merged[idx == np.searchsorted(bits, np.float64(-0.0).view(np.int64))] = np.searchsorted(bits, 0)
    with pytest.raises(AssertionError):
        O.check_value_dict(ref, s, merged, table.view(np.float64), distinct)


def test_level_flags_and_dedup():
    A = F.canonical_csr(P.structured_laplacian_2d(16))
    col, _ = O.colors(A)
    assert O.level_flags(A, col) == (True, True)
    assert O.level_flags(A, np.zeros_like(col))[0] is False
    B = A.copy()
    B.data[B.indptr[40] + 2] = 0.0                                    # the diagonal of an interior row
    assert B.indices[B.indptr[40] + 2] == 40 and O.level_flags(B, col)[1] is False
    keys = np.array([[1, 2], [3, 4], [1, 2], [5, 6], [3, 4], [1, 2]])
    labels, counts = O.dedup_rows(keys)
    assert list(labels) == [0, 1, 0, 2, 1, 0] and list(counts) == [3, 2, 1]
