"""Host reference of the device hierarchy setup (setup_device.py and the extras engine.DeviceSell attaches), one
function per stage, for tests/test_gpu_setup_scale.py.

Where formats holds an independent host restatement it is reused: SciPy's Galerkin product, the serial first-fit
colouring (greedy_colors), the colour permutation, permute_csr / csr_to_sell and the slice offsets / patterns.  The
deduplicated records (formats.slice_records, formats.pattern_records) and the spec blocks (engine.DeviceSell) are the
product's own torch code, so they are restated here in plain NumPy, and the device's output is compared by meaning:
record ids depend on how ties in frequency are ordered, so a check asks that every slice with an id resolves to exactly
its own columns and value bits, that the slices with an id are the reference's, that ids are ordered by use and that
each block's by-value record is one of the most used in that block.

check_* functions take host arrays (downloaded device tensors, or the torch functions' output on CPU tensors) and
raise AssertionError with the stage in the message.
"""
import numpy as np
import scipy.sparse as sp

from learnmultigrid_b200 import formats as F
from learnmultigrid_b200.engine import DeviceSell

SLICE = F.SLICE
VALUE_DICT_MAX = 256
SLICE_RECORDS_MAX = 32766          # formats.slice_records' max_records
PATTERN_RECORDS_MAX = 256          # formats.pattern_records' max_records
PATTERN_MIN_SLICES = 2             # formats.pattern_records' min_slices
PATTERN_BLOCKS = 8                 # blocks the pattern launcher knows; later rows count to the last one
CHUNK = 1 << 18                    # slices per vectorised step: bounds the temporaries at benchmark sizes


# ---- stages that formats restates on the host ------------------------------------------------------------------
def galerkin(A, Q):
    """csr_matrix(Q.T @ A @ Q) with sorted indices, as the reference evaluates it (A stored CSC at level 0)"""
    C = sp.csr_matrix(Q.T @ A @ Q)
    C.sort_indices()
    return F.canonical_csr(C)


def colors(A):
    """(colours, number of colours) of the serial first-fit helper"""
    return F.greedy_colors(A)


def permutation(col):
    """(perm new -> old, inverse, colour offsets)"""
    perm, cptr = F.color_permutation(col)
    return perm, F.inverse_permutation(perm), cptr


def sell(A, row_perm=None, col_iperm=None):
    """SELL-32 arrays of A in the colour-blocked ordering, with max_len and uniform_len as DeviceSell reports them"""
    slice_ptr, cols, vals = F.csr_to_sell(F.permute_csr(A, row_perm, col_iperm))
    d = np.diff(slice_ptr) // SLICE
    max_len = int(d.max()) if len(d) else 0
    uniform_len = max_len if len(d) and int(d.min()) == max_len else 0
    return {"slice_ptr": slice_ptr, "cols": cols, "vals": vals, "max_len": max_len, "uniform_len": uniform_len,
            "nrows": A.shape[0], "shape": A.shape}


def dinv(A, perm=None):
    with np.errstate(divide="ignore"):
        d = 1.0 / A.diagonal()
    return d if perm is None else d[perm]


def level_flags(A, col):
    """(proper, nonzero_diag): no row couples to another row of its colour; every row has a non-zero diagonal"""
    rows = np.repeat(np.arange(A.shape[0], dtype=np.int64), np.diff(A.indptr))
    off = rows != A.indices
    proper = not np.any(col[rows[off]] == col[A.indices[off]])
    return proper, bool(np.all(A.diagonal() != 0.0))


# ---- value dictionary ----------------------------------------------------------------------------------------------
def value_dict(s, chunk=1 << 20):
    """the distinct value bit patterns of a SELL matrix (padding included: the kernels read it) and whether
    DeviceSell attaches a dictionary: at most 256 of them, 1 <= max_len <= 8, at least VALUE_DICT_MIN_ROWS rows.
    The values are scanned chunk by chunk against the distinct ones found so far, and the scan stops once there are
    more than 256: count is exact up to 257 and a lower bound beyond (a variable-coefficient operator is not sorted)."""
    v = s["vals"].view(np.int64)
    bits = np.zeros(0, dtype=np.int64)
    for a in range(0, v.size, chunk):
        c = v[a:a + chunk]
        if bits.size:
            i = np.minimum(np.searchsorted(bits, c), bits.size - 1)
            c = c[bits[i] != c]
        if c.size:
            bits = np.union1d(bits, c)
        if bits.size > VALUE_DICT_MAX:
            break
    attached = (1 <= s["max_len"] <= 8 and s["nrows"] >= DeviceSell.VALUE_DICT_MIN_ROWS and s["vals"].size > 0
                and len(bits) <= VALUE_DICT_MAX)
    return {"bits": bits, "count": len(bits), "attached": attached}


def check_value_dict(ref, s, val_idx, val_table, count):
    """val_idx / val_table / count: the device's (None when none is attached)"""
    assert (val_idx is not None) == ref["attached"], "value dictionary attached: %s, reference %s" % (
        val_idx is not None, ref["attached"])
    if not ref["attached"]:
        return
    assert count == ref["count"], "value dictionary: %d distinct values, reference %d" % (count, ref["count"])
    table = np.asarray(val_table).view(np.int64)
    assert np.array_equal(np.sort(table[:count]), ref["bits"]), "value dictionary table is not the distinct values"
    assert int(np.asarray(val_idx).max()) < count, "value dictionary index beyond the table"
    for a in range(0, s["vals"].size, CHUNK * SLICE):
        b = min(a + CHUNK * SLICE, s["vals"].size)
        assert np.array_equal(table[np.asarray(val_idx[a:b], dtype=np.int64)], s["vals"][a:b].view(np.int64)), \
            "value dictionary does not decode to the values (entries %d..%d)" % (a, b)


# ---- exact deduplication -----------------------------------------------------------------------------------------
def dedup_rows(keys):
    """(labels, counts) of the distinct rows of an int64 matrix: labels[i] = group of row i, groups numbered by first
    occurrence.  A 64-bit hash groups the rows, every row is then compared with its group's first row entry by entry;
    a collision falls back to sorting the rows themselves, so the grouping is exact."""
    keys = np.ascontiguousarray(keys, dtype=np.int64)
    n = keys.shape[0]
    if n == 0:
        return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    w = np.random.default_rng(7).integers(1, 1 << 62, keys.shape[1], dtype=np.int64) | 1
    with np.errstate(over="ignore"):
        h = keys @ w
    _, first_idx, inv = np.unique(h, return_index=True, return_inverse=True)
    exact = True
    for a in range(0, n, CHUNK):
        b = min(a + CHUNK, n)
        if not np.array_equal(keys[a:b], keys[first_idx[inv[a:b]]]):
            exact = False
            break
    if not exact:
        v = keys.view(np.dtype((np.void, keys.shape[1] * 8))).ravel()
        _, first_idx, inv = np.unique(v, return_index=True, return_inverse=True)
    order = np.argsort(first_idx, kind="stable")            # number groups by first occurrence
    relabel = np.empty(len(order), dtype=np.int64)
    relabel[order] = np.arange(len(order))
    labels = relabel[inv.reshape(-1)]
    return labels, np.bincount(labels, minlength=len(order))


# ---- slice records (implied columns / values) --------------------------------------------------------------------
def slice_records(s, dict_attached):
    """formats.slice_records as DeviceSell._attach_slice_offsets applies it: whether records are attached, whether they
    carry values, and per slice the group of its record (-1: no record).  A uniform matrix with 1..8 entries per row and
    at least IMPLIED_MIN_ROWS / 2 rows gets offsets; they are kept when at least half of the slices are regular; with a
    value dictionary a record carries the values (a slice then also needs one value per entry in all 32 rows) if that
    loses at most a tenth of the regular slices."""
    L, n = s["uniform_len"], s["nrows"]
    nsl = len(s["slice_ptr"]) - 1
    out = {"attempted": 1 <= L <= 8 and n >= max(DeviceSell.IMPLIED_MIN_ROWS // 2, 1), "attached": False}
    if not out["attempted"]:
        return out
    off = F.sell_slice_offsets((s["slice_ptr"], s["cols"], s["vals"]), n, L)
    regular = off[:, 0] != F.SLICE_IRREGULAR
    n_regular = int(regular.sum())
    out["regular_columns"] = n_regular
    if 2 * n_regular < nsl:
        return out
    keys = off.astype(np.int64)
    with_values = False
    if dict_attached:
        vb = s["vals"].view(np.int64).reshape(nsl, L, SLICE)
        same = np.all(vb == vb[:, :, :1], axis=(1, 2))
        full = regular & same
        if n_regular > 0 and 10 * int(full.sum()) >= 9 * n_regular:
            with_values = True
            regular = full
            keys = np.concatenate([keys, vb[:, :, 0]], axis=1)
        del vb, same, full
    labels, counts = dedup_rows(keys[regular])
    assert len(counts) <= SLICE_RECORDS_MAX, "more slice records than the table holds"
    group = np.full(nsl, -1, dtype=np.int64)
    group[regular] = labels
    out.update(attached=True, with_values=with_values, group=group, counts=counts)
    return out


def check_slice_records(ref, s, ids, rec_table, rec_vals):
    """the device's ids [nslices] / rec_table [nrec, 8] / rec_vals [nrec, 8] or None against the reference's meaning"""
    assert (ids is not None) == ref["attached"], "slice records attached: %s, reference %s" % (
        ids is not None, ref["attached"])
    if not ref["attached"]:
        return
    L = s["uniform_len"]
    nsl = len(s["slice_ptr"]) - 1
    ids = np.asarray(ids).astype(np.int64)
    assert (rec_vals is not None) == ref["with_values"], "slice records carry values: %s, reference %s" % (
        rec_vals is not None, ref["with_values"])
    assert np.array_equal(ids >= 0, ref["group"] >= 0), "the slices with a record differ from the reference (%d vs %d)" % (
        int((ids >= 0).sum()), int((ref["group"] >= 0).sum()))
    nrec = rec_table.shape[0]
    assert nrec == len(ref["counts"]), "%d slice records, reference %d distinct" % (nrec, len(ref["counts"]))
    assert np.all(rec_table[:, L:] == 0), "slice record entries beyond uniform_len are not zero"
    cols = s["cols"].reshape(nsl, L, SLICE)
    vb = s["vals"].view(np.int64).reshape(nsl, L, SLICE)
    lane = np.arange(SLICE, dtype=np.int64)
    for a in range(0, nsl, CHUNK):
        b = min(a + CHUNK, nsl)
        sl = a + np.nonzero(ids[a:b] >= 0)[0]
        rows = sl[:, None, None] * SLICE + lane[None, None, :]
        want = rows + rec_table[ids[sl]][:, :L, None].astype(np.int64)
        assert np.array_equal(cols[sl], want), "slice record does not resolve to the slice's columns (slices %d..%d)" % (a, b)
        if rec_vals is not None:
            rv = np.asarray(rec_vals).view(np.int64)[ids[sl]][:, :L, None]
            assert np.all(vb[sl] == rv), "slice record does not resolve to the slice's values (slices %d..%d)" % (a, b)
    # one record per reference group: the records are distinct, and a record's slices are one group
    keys = rec_table.astype(np.int64)
    if rec_vals is not None:
        keys = np.concatenate([keys, np.asarray(rec_vals).view(np.int64)], axis=1)
    assert len(dedup_rows(keys)[1]) == nrec, "two slice records are equal"
    use = np.bincount(ids[ids >= 0], minlength=nrec)
    assert np.all(np.diff(use) <= 0), "slice record ids are not ordered by use"
    assert np.array_equal(np.sort(use), np.sort(ref["counts"])), "slice record use differs from the reference groups"


# ---- slice patterns (implied transfer columns) ---------------------------------------------------------------------
def pattern_sample(nsl):
    """the evenly spaced slices DeviceSell._attach_patterns deduplicates first (float64 here: a pick may differ by one
    slice from the device's float32 linspace; only the decision is compared)"""
    return np.linspace(0, nsl - 2, DeviceSell.PATTERN_SAMPLE).astype(np.int64)


def _pattern_keys(cols, vals, L, sl):
    c = cols.reshape(-1, L * SLICE)[sl].astype(np.int64)
    return np.concatenate([c - c[:, :1], vals.view(np.int64).reshape(-1, L * SLICE)[sl]], axis=1)


def _pattern_kept(cols, vals, L, sl, full):
    """(group [len(sl)], counts, kept group ids in rank order, cutoff count) of formats.pattern_records restated:
    exact dedup over the full slices of [delta, value bits]; records used by >= 2 slices, the 256 most used"""
    group = np.full(len(sl), -1, dtype=np.int64)
    f = np.nonzero(full)[0]
    labels, counts = dedup_rows(np.concatenate([_pattern_keys(cols, vals, L, sl[f[a:a + CHUNK]])
                                                for a in range(0, len(f), CHUNK)]) if len(f) else
                                np.zeros((0, 2 * L * SLICE), dtype=np.int64))
    group[f] = labels
    rank = np.argsort(-counts, kind="stable")
    rank = rank[counts[rank] >= PATTERN_MIN_SLICES]
    kept = rank[:PATTERN_RECORDS_MAX]
    tie = len(rank) > PATTERN_RECORDS_MAX and counts[rank[PATTERN_RECORDS_MAX]] == counts[kept[-1]]
    cutoff = int(counts[kept[-1]]) if tie else None          # the count the 256-record cutoff falls inside
    return group, counts, kept, cutoff


def pattern_records(s, slice_records_attached):
    """formats.pattern_records as DeviceSell._attach_patterns applies it: tried on a rectangular uniform matrix with
    1..8 entries per row and at least IMPLIED_MIN_ROWS rows that has no slice records; with more than 2 x 4096 slices a
    sample must keep a record for at least half of its slices first; kept when at least half of all slices have one."""
    L, n = s["uniform_len"], s["nrows"]
    nsl = len(s["slice_ptr"]) - 1
    out = {"attempted": (not slice_records_attached and s["shape"][0] != s["shape"][1] and 1 <= L <= 8
                         and n >= max(DeviceSell.IMPLIED_MIN_ROWS, 1)), "attached": False, "sampled": False}
    if not out["attempted"]:
        return out
    cols, vals = s["cols"], s["vals"]
    if nsl > 2 * DeviceSell.PATTERN_SAMPLE:
        pick = pattern_sample(nsl)
        _, counts, kept, _ = _pattern_kept(cols, vals, L, pick, np.ones(len(pick), dtype=bool))
        out.update(sampled=True, sample_slices=int(counts[kept].sum()))
        if 2 * out["sample_slices"] < DeviceSell.PATTERN_SAMPLE:
            return out
    full = (np.arange(nsl) + 1) * SLICE <= n
    group, counts, kept, cutoff = _pattern_kept(cols, vals, L, np.arange(nsl), full)
    with_rec = np.isin(group, kept)
    out.update(group=group, counts=counts, kept=kept, cutoff=cutoff, with_record=with_rec,
               slices=int(with_rec.sum()))
    out["attached"] = 2 * out["slices"] >= nsl
    return out


def check_pattern_records(ref, s, ids, delta, pvals, base):
    """the device's ids [nslices], delta [nrec, L, 32], pvals [nrec, L, 32], base [nslices] (None when no patterns are
    attached) against the reference's meaning"""
    assert (ids is not None) == ref["attached"], "slice patterns attached: %s, reference %s" % (
        ids is not None, ref["attached"])
    if not ref["attached"]:
        return
    L = s["uniform_len"]
    nsl = len(s["slice_ptr"]) - 1
    ids = np.asarray(ids).astype(np.int64)
    cols = s["cols"].reshape(nsl, L, SLICE)
    vb = s["vals"].view(np.int64).reshape(nsl, L, SLICE)
    assert np.array_equal(base, cols[:, 0, 0]), "slice pattern base is not the slice's first column"
    nrec = delta.shape[0]
    assert nrec == len(ref["kept"]), "%d slice patterns, reference %d" % (nrec, len(ref["kept"]))
    has = ids >= 0
    for a in range(0, nsl, CHUNK):
        b = min(a + CHUNK, nsl)
        sl = a + np.nonzero(has[a:b])[0]
        want = base[sl].astype(np.int64)[:, None, None] + delta[ids[sl]].astype(np.int64)
        assert np.array_equal(cols[sl], want), "slice pattern does not resolve to the slice's columns (slices %d..%d)" % (a, b)
        assert np.array_equal(vb[sl], np.asarray(pvals).view(np.int64)[ids[sl]]), \
            "slice pattern does not resolve to the slice's values (slices %d..%d)" % (a, b)
    use = np.bincount(ids[has], minlength=nrec)
    assert np.all(np.diff(use) <= 0), "slice pattern ids are not ordered by use"
    # Deliberately stricter than formats.pattern_records promises: its hash groups may collide, and a collision may
    # cost a slice its record (never a wrong column).  With its fixed weights no collision occurs on these operators,
    # so every slice of an exact group must have the record; a failure below after a change of data or weights may
    # be such a collision rather than a wrong record -- the resolve checks above still hold in that case.
    assert use.min() >= PATTERN_MIN_SLICES, "a slice pattern serves fewer than 2 slices"
    # the same groups: every slice of a reference group has a record, and that record's slices are the whole group
    g = ref["group"]
    assert not np.any(has & (g < 0)), "a slice beyond the matrix has a slice pattern"
    first = np.full(nrec, -1, dtype=np.int64)
    first[ids[has][::-1]] = g[has][::-1]
    assert np.array_equal(g[has], first[ids[has]]), "one slice pattern serves slices of different reference groups"
    assert len(np.unique(first)) == nrec, "two slice patterns are the same reference group"
    assert np.array_equal(use, ref["counts"][first]), "a slice pattern does not serve its whole reference group"
    want_use = np.sort(ref["counts"][ref["kept"]])
    assert np.array_equal(np.sort(use), want_use), "slice pattern use differs from the reference's 256 most used"
    if ref["cutoff"] is None:
        assert np.array_equal(has, ref["with_record"]), "the slices with a pattern differ from the reference"
    else:                # ties at the 256-record cutoff: the identities of the last records may differ, the counts not
        above = (g >= 0) & (ref["counts"][np.maximum(g, 0)] > ref["cutoff"])
        assert np.all(has[above]), "a slice of a group above the 256-record cutoff has no pattern"
        assert np.all(ref["counts"][g[has & ~above]] == ref["cutoff"]), "a pattern below the cutoff was kept"


# ---- spec blocks ---------------------------------------------------------------------------------------------------
def _block_slices(row_ptr, k):
    return row_ptr[k] // SLICE, max((row_ptr[k + 1] + SLICE - 1) // SLICE, row_ptr[k] // SLICE + 1)


def pattern_block_rows(row_ptr):
    """the row blocks the pattern launcher is told about: 8 at most, the last absorbs the rest"""
    row_ptr = [int(v) for v in row_ptr]
    return row_ptr[:PATTERN_BLOCKS] + row_ptr[-1:] if len(row_ptr) > PATTERN_BLOCKS + 1 else row_ptr


def check_offset_spec_blocks(row_ptr, spec_rows, spec_rec, spec_vals, ids, rec_table, rec_vals):
    """by-value offset record of every colour block: its record (and values) are one of the block's most used"""
    row_ptr = [int(v) for v in row_ptr]
    nb = len(row_ptr) - 1
    assert list(spec_rows) == row_ptr, "spec blocks are not the colour blocks"
    ids = np.asarray(ids).astype(np.int64)
    for k in range(nb):
        s0, s1 = _block_slices(row_ptr, k)
        blk = ids[s0:s1]
        blk = blk[blk >= 0]
        best = int(spec_rec[9 * k])
        if blk.size:
            use = np.bincount(blk, minlength=rec_table.shape[0])
            assert use[best] == use.max(), "block %d: by-value record %d is used %d times, the most used %d" % (
                k, best, use[best], use.max())
        else:
            assert best == 0, "block %d has no record but names %d" % (k, best)
        assert list(spec_rec[9 * k + 1:9 * k + 9]) == list(rec_table[best]), "block %d: by-value offsets" % k
        if rec_vals is not None:
            assert np.array_equal(np.asarray(spec_vals[8 * k:8 * k + 8]).view(np.int64),
                                  np.asarray(rec_vals[best]).view(np.int64)), "block %d: by-value values" % k


def check_pattern_spec_blocks(row_ptr, spec_rows, spec_rec, ids, ref_group):
    """by-value slice pattern of every block (colour blocks, 8 at most): one of the block's most used, and the share of
    the most used one in per mille of the block's slices, from the reference groups"""
    row_ptr = pattern_block_rows(row_ptr)
    nb = len(row_ptr) - 1
    assert list(spec_rows) == row_ptr, "pattern spec blocks are not the (capped) colour blocks"
    ids = np.asarray(ids).astype(np.int64)
    for k in range(nb):
        s0, s1 = _block_slices(row_ptr, k)
        n = len(ids[s0:s1])
        blk = ids[s0:s1]
        has = blk >= 0
        best = int(spec_rec[9 * k])
        if has.any():
            use = np.bincount(blk[has])
            assert best < len(use) and use[best] == use.max(), "block %d: by-value pattern is not the most used" % k
            most = int(np.bincount(ref_group[s0:s1][has]).max())
        else:
            assert best == 0, "block %d has no pattern but names %d" % (k, best)
            most = 0
        assert int(spec_rec[9 * k + 1]) == 1000 * most // max(n, 1), "block %d: per-mille share %d, reference %d" % (
            k, spec_rec[9 * k + 1], 1000 * most // max(n, 1))
