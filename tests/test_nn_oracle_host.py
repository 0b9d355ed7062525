"""The NumPy stages of tests/nn_oracle.py (fold, normalise, cut, next_mass and their composition) against the golden
vectors of the reference's NeuralMG_2D (tests/golden/neural_2d_cases.npz) and against the plain running-mean loop of
test_neural2d_host.py, so that they can serve as the reference for the device builder at sizes the goldens do not
reach (tests/test_gpu_nn_scale.py)."""
import numpy as np
import pytest
import scipy.sparse as sp

import nn_oracle as O
from helpers import load_golden
from test_gpu_neural2d import Stub
from test_neural2d_host import CASES, fold_reference_rule, levels_of


def golden_cmap(d):
    n, nc = d["M"].shape[0], len(d["C"])
    cmap = np.full(n, -1, dtype=np.int32)
    cmap[d["C"]] = np.arange(nc, dtype=np.int32)
    return cmap


@pytest.mark.parametrize("case", CASES)
def test_fold_normalise_and_cut_reproduce_the_reference(case):
    """B bit for bit; Q to 1e-15 relative (about 4 ulp: the reference adds each dense row pairwise, the oracle in
    column order as the device does); the cut Galerkin product with the pattern of the next level's stored matrix and
    its values to 1e-15 relative (the reference multiplies dense matrices)"""
    g = load_golden("neural_2d_cases.npz")
    lv = levels_of(g, case)
    for l, d in enumerate(lv):
        n, nc = d["M"].shape[0], len(d["C"])
        cmap = golden_cmap(d)
        rows, cols, vals, dn = O.contributions(d["fill"], d["pred"], cmap, n, nc)
        assert np.array_equal(dn, d["dn"])
        B = O.fold(rows, cols, vals, n, nc)
        assert B.has_sorted_indices and B.nnz == np.count_nonzero(d["B"])
        assert np.array_equal(B.toarray(), d["B"])
        assert np.array_equal(B.toarray(), fold_reference_rule(rows, cols, vals, n, nc, n))
        Q = O.normalise(B)
        assert np.array_equal(Q.indptr, B.indptr) and np.array_equal(Q.indices, B.indices)
        np.testing.assert_allclose(Q.toarray(), d["Q"], rtol=1e-15, atol=0)
        if l + 1 < len(lv):
            want = lv[l + 1]["M"]
            got = O.cut(O.next_mass(d["M"], sp.csr_matrix(d["Q"])), d["dn"])
            assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
            np.testing.assert_allclose(got.data, want.data, rtol=1e-15, atol=0)


def test_normalise_adds_each_row_in_column_order():
    """rows whose sum depends on the order of the additions: the oracle adds in column order"""
    x = np.array([1.0, 1e-16, 1e-16, 1e-16, 1e-16])
    B = sp.csr_matrix(np.vstack([x, x[::-1]]))
    sums = []
    for row in (x, x[::-1]):
        s = 0.0
        for v in row:
            s += v
        sums.append(s)
    assert sums[0] != sums[1]
    np.testing.assert_array_equal(O.normalise(B).data, np.concatenate([x / sums[0], x[::-1] / sums[1]]))


def test_cut_keeps_the_diagonal_and_the_listed_neighbours_only():
    M = sp.csr_matrix(np.array([[4.0, 1.0, 2.0, 0.0],
                                [1.0, 4.0, 0.0, 3.0],
                                [2.0, 5.0, 0.0, 1.0],
                                [0.0, 3.0, 1.0, 4.0]]))
    M.data[M.indptr[2] + 1] = 0.0                        # M[2, 1]: an explicitly stored zero
    dn = np.array([[2, -1, -1, -1, -1, -1], [-1] * 6, [1, 3, -1, -1, -1, -1], [0, 1, 2, -1, -1, -1]], dtype=np.int32)
    got = O.cut(M, dn)
    assert np.array_equal(got.toarray(), [[4, 0, 2, 0], [0, 4, 0, 0], [0, 0, 0, 1], [0, 3, 1, 4]])
    assert got.nnz == 7                                   # the zero diagonal of row 2 and the stored zero are gone


@pytest.mark.parametrize("seed", range(6))
def test_fold_equals_the_running_mean_loop(seed):
    """random contributions with many collisions, values from a small set so that runs cancel to exactly 0 and start
    again, exact-0 predictions, and unused slots"""
    rng = np.random.default_rng(seed)
    n, nc, m = 23, 9, 500
    rows = rng.integers(0, n + 3, size=m).astype(np.int32)          # rows >= n are unused slots
    cols = rng.integers(0, nc, size=m).astype(np.int32)
    vals = rng.choice([-1.0, -0.5, 0.0, 0.0, 0.5, 1.0, 0.75, 2.0], size=m)
    stats = {}
    B = O.fold(rows, cols, vals, n, nc, stats)
    want = fold_reference_rule(rows, cols, vals, n, nc, n)
    assert np.array_equal(B.toarray(), want)
    assert B.nnz == np.count_nonzero(want) and B.has_sorted_indices
    assert stats["restarts"] > 0 and stats["cancelled"] >= stats["restarts"] and stats["dropped"] > 0


def test_fold_on_hand_made_runs():
    rows = np.array([0, 0, 0, 0, 1, 1, 1, 2, 2, 1, 3], dtype=np.int32)
    cols = np.array([0, 0, 0, 1, 0, 0, 0, 1, 1, 1, 0], dtype=np.int32)
    vals = np.array([1.0, -1.0, 3.0, 0.0, 2.0, 0.0, 4.0, 5.0, -5.0, 7.0, 1.0])
    stats = {}
    B = O.fold(rows, cols, vals, 3, 2, stats)          # row 3 is the unused row
    # (0,0): 1 -> 0 -> 3 ; (0,1): 0 dropped ; (1,0): 2 -> (2+0)/2=1 -> (1+4)/2 ; (2,1): 5 -> 0 dropped ; (1,1): 7
    assert np.array_equal(B.toarray(), [[3.0, 0.0], [2.5, 7.0], [0.0, 0.0]])
    assert stats == {"cancelled": 2, "restarts": 1, "dropped": 2}


@pytest.mark.parametrize("case", CASES)
def test_oracle_hierarchy_reproduces_the_reference(case):
    """the composed oracle with the golden predictor: coarse sets and fill indices exact on every level; the level-0
    patches, B and Q as above; coarser levels to the bars of the device's define_hierarchy test (the reference forms
    Q^T M Q densely)"""
    g = load_golden("neural_2d_cases.npz")
    lv = levels_of(g, case)
    mean, std = (g["mean2"], g["std2"]) if case in ("r77", "i289", "f169") else (np.zeros(43), np.ones(43))
    got = O.define_hierarchy(lv[0]["M"], Stub(), mean, std, len(lv) + 1)
    assert len(got) == len(lv)
    for l, (o, d) in enumerate(zip(got, lv)):
        assert np.array_equal(o["clist"], d["C"]) and np.array_equal(o["fill"], d["fill"])
        assert np.array_equal(o["dneigh"], d["dn"])
        assert np.array_equal(o["M"].indptr, d["M"].indptr) and np.array_equal(o["M"].indices, d["M"].indices)
        np.testing.assert_allclose(o["M"].data, d["M"].data, rtol=1e-13)
        if l == 0:
            assert np.array_equal(o["patches"], d["patches"]) and np.array_equal(o["B"].toarray(), d["B"])
            np.testing.assert_allclose(o["Q"].toarray(), d["Q"], rtol=1e-15, atol=0)
            extra = o["fill"].shape[0] - len(d["C"])
            assert int(o["not_last"].sum()) == extra and o["not_last"][len(d["C"]):].sum() < max(extra, 1)
        else:
            np.testing.assert_allclose(o["patches"], d["patches"], rtol=1e-13)
            np.testing.assert_allclose(o["Q"].toarray(), d["Q"], rtol=1e-12, atol=1e-300)
