"""formats.pattern_records (the slice patterns behind the implied transfer columns, sell_core.cuh sell_pattern_kernel)
on host tensors, against its host twin formats.sell_slice_patterns."""
import numpy as np
import scipy.sparse as sp

from learnmultigrid_b200 import formats as F
from learnmultigrid_b200 import problems as P


def _transfers(N, levels=3):
    A = P.structured_laplacian_2d(N)
    Qs = P.structured_hierarchy_2d(N, levels, transfer="linear")
    lv = F.build_host_hierarchy(A, Qs, "mcgs")
    return [(lv[l][k], lv[l][k + "_sell"]) for l in range(levels - 1) for k in ("Q", "QT")]


def test_pattern_records_rebuild_the_transfer_operators():
    """every slice with a record id has exactly the columns base + delta[id] and the values vals[id] (same bits) in all
    32 rows; ids are ordered by frequency, a kept record serves at least two slices, the ragged last slice has none,
    and on the structured hierarchy most slices of the level-0 restriction and prolongation have one"""
    import torch
    for M, sell in _transfers(256):
        slice_ptr, cols, vals = sell
        nsl = len(slice_ptr) - 1
        L = int(slice_ptr[1]) // 32
        assert slice_ptr[-1] == nsl * 32 * L                         # linear transfers are uniform
        base_h, delta_h, vals_h, full = F.sell_slice_patterns(sell, M.shape[0], L)
        base, ids, delta, pv, nrec = F.pattern_records(torch, torch.from_numpy(cols), torch.from_numpy(vals),
                                                       M.shape[0], L, chunk=97)
        base, ids, delta, pv = base.numpy(), ids.numpy(), delta.numpy(), pv.numpy()
        assert np.array_equal(base, base_h)
        reg = ids >= 0
        assert nrec == reg.sum() and not np.any(reg & ~full)
        r = np.maximum(ids, 0)
        assert np.array_equal((base[:, None, None] + delta[r].astype(np.int64))[reg],
                              cols.reshape(nsl, L, 32)[reg])
        assert np.array_equal(delta[r][reg], delta_h[reg])
        assert np.array_equal(pv[r][reg].view(np.int64), vals_h[reg].view(np.int64))
        counts = np.bincount(ids[reg], minlength=len(delta))
        assert np.all(np.diff(counts) <= 0) and counts.min() >= 2
        # every full slice whose pattern is shared with another full slice has a record (at most 256 kept)
        if len(delta) < 256:
            keys = [(delta_h[s].tobytes(), vals_h[s].tobytes()) for s in range(nsl) if full[s]]
            from collections import Counter
            shared = Counter(keys)
            want = sum(1 for s in range(nsl) if full[s] and shared[(delta_h[s].tobytes(), vals_h[s].tobytes())] >= 2)
            assert nrec == want
    (Q0, s0), (QT0, t0) = _transfers(256)[:2]
    for M, sell in ((Q0, s0), (QT0, t0)):
        L = int(sell[0][1]) // 32
        *_, nrec = F.pattern_records(torch, torch.from_numpy(sell[1]), torch.from_numpy(sell[2]), M.shape[0], L)
        assert nrec > 0.7 * (len(sell[0]) - 1)


def test_pattern_records_of_an_unstructured_numbering_keep_nothing():
    """rows and columns of a transfer operator shuffled at random: no two slices share a pattern, no record is kept"""
    import torch
    (Q, _), = _transfers(128, 2)[:1]
    rng = np.random.default_rng(3)
    Qp = F.canonical_csr(sp.csr_matrix(Q)[rng.permutation(Q.shape[0])][:, rng.permutation(Q.shape[1])])
    slice_ptr, cols, vals = F.csr_to_sell(Qp)
    L = int(slice_ptr[1]) // 32
    assert slice_ptr[-1] == (len(slice_ptr) - 1) * 32 * L
    base, ids, delta, pv, nrec = F.pattern_records(torch, torch.from_numpy(cols), torch.from_numpy(vals), Qp.shape[0], L)
    assert nrec == 0 and delta.shape[0] == 0 and np.all(ids.numpy() == -1)
