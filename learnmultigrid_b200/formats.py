"""Host-side sparse-format plumbing (NumPy, vectorised): canonical CSR, level permutations, SELL-32 layout.

These routines only rearrange integers and copy values; all floating-point work happens in the CUDA kernels.
They are also the host cross-check of the device setup kernels (tests compare the two).
"""
import ctypes

import numpy as np
import scipy.sparse as sp

from . import _lib

SLICE = 32


def solver_csr(A):
    """The CSR form of what the reference's Solver holds, `csc_matrix(matrix)` (Solver.py:18).  A CSR matrix that is
    already canonical (sorted, duplicate-free) comes back from the CSR -> CSC -> CSR round trip unchanged, so it is
    taken as it is (the round trip costs seconds at 10^8 entries)."""
    if sp.isspmatrix_csr(A) and A.dtype == np.float64 and A.has_canonical_format:
        return canonical_csr(A)
    return canonical_csr(sp.csc_matrix(A))


def canonical_csr(A):
    """scipy CSR with sorted, duplicate-free int32 indices and float64 data (what SciPy hands to its kernels)."""
    if not sp.issparse(A):
        A = sp.csr_matrix(np.asarray(A, dtype=np.float64))
    A = sp.csr_matrix(A, dtype=np.float64)
    A.sum_duplicates()
    A.sort_indices()
    if A.nnz >= 2 ** 31 or max(A.shape) >= 2 ** 31:
        raise OverflowError("matrix does not fit the int32 index contract")
    A.indptr = A.indptr.astype(np.int32, copy=False)
    A.indices = A.indices.astype(np.int32, copy=False)
    return A


def raw_csr(indptr, indices, data, shape):
    """CSR container that never re-sorts or merges (entries keep the given order)."""
    M = sp.csr_matrix(shape, dtype=np.float64)
    M.indptr = np.ascontiguousarray(indptr, dtype=np.int32)
    M.indices = np.ascontiguousarray(indices, dtype=np.int32)
    M.data = np.ascontiguousarray(data, dtype=np.float64)
    return M


def permute_csr(A, row_perm=None, col_iperm=None):
    """rows: new row i = old row row_perm[i]; columns relabelled old j -> col_iperm[j].
    Entries keep their ORIGINAL order inside every row (so row sums round exactly as in natural ordering)."""
    indptr, indices, data = A.indptr, A.indices, A.data
    if row_perm is not None:
        lens = np.diff(indptr)[row_perm]
        new_ptr = np.zeros(len(row_perm) + 1, dtype=np.int64)
        np.cumsum(lens, out=new_ptr[1:])
        # source position of every new entry
        src = np.repeat(indptr[:-1][row_perm].astype(np.int64) - new_ptr[:-1], lens) + np.arange(new_ptr[-1])
        indices = indices[src]
        data = data[src]
        indptr = new_ptr
        nrows = len(row_perm)
    else:
        nrows = A.shape[0]
    if col_iperm is not None:
        indices = np.asarray(col_iperm, dtype=np.int32)[indices]
    return raw_csr(indptr, indices, data, (nrows, A.shape[1]))


def transpose_csr(Q):
    """CSR of Q^T whose row entries are in ascending original-row order (the order SciPy's csc_matvec adds
    them in `i.T @ res`, Multigrid.py:93)."""
    QT = sp.csr_matrix(sp.csc_matrix(Q).T) if not sp.isspmatrix_csr(Q) else Q.T.tocsr()
    QT.sort_indices()
    return canonical_csr(QT)


def sell_is_uniform(max_len, sum_len, nslices):
    """pad all slices to the longest one when that costs at most 3 % extra entries -- 25 % for rows of one or two
    entries, whose kernel then needs no slice pointer (same rule as mg_sell_layout)"""
    return max_len > 0 and nslices * max_len * 100 <= (125 if max_len <= 2 else 103) * sum_len


def csr_to_sell(A):
    """(slice_ptr int64[nslices+1], cols int32[total], vals float64[total]) of the SELL-32 layout."""
    n = A.shape[0]
    indptr = A.indptr.astype(np.int64)
    indices, data = A.indices, A.data
    lens = np.diff(indptr)
    nsl = (n + SLICE - 1) // SLICE
    lens_p = np.zeros(nsl * SLICE, dtype=np.int64)
    lens_p[:n] = lens
    sl_len = lens_p.reshape(nsl, SLICE).max(axis=1) if nsl else np.zeros(0, dtype=np.int64)
    if nsl and sell_is_uniform(int(sl_len.max()), int(sl_len.sum()), nsl):
        sl_len = np.full(nsl, sl_len.max(), dtype=np.int64)      # pad every slice to the longest one
    slice_ptr = np.zeros(nsl + 1, dtype=np.int64)
    np.cumsum(sl_len * SLICE, out=slice_ptr[1:])
    total = int(slice_ptr[-1])
    lastcol = np.zeros(nsl * SLICE, dtype=np.int32)
    nz = lens > 0
    lastcol[:n][nz] = indices[indptr[1:][nz] - 1]
    cols = np.repeat(lastcol.reshape(nsl, SLICE), sl_len, axis=0).reshape(-1)
    cols = np.ascontiguousarray(cols, dtype=np.int32)
    vals = np.zeros(total, dtype=np.float64)
    if len(data):
        rows = np.repeat(np.arange(n, dtype=np.int64), lens)
        k = np.arange(len(data), dtype=np.int64) - indptr[rows]
        dest = slice_ptr[rows >> 5] + k * SLICE + (rows & 31)
        cols[dest] = indices
        vals[dest] = data
    return slice_ptr, cols, vals


def sell_padding_ratio(A):
    slice_ptr, _, _ = csr_to_sell(A) if not isinstance(A, tuple) else A
    return float(slice_ptr[-1])


def greedy_colors(A):
    """First-fit colouring in index order on the symmetrised pattern (C helper in libmgb200, host code)."""
    A = canonical_csr(A)
    n = A.shape[0]
    colors = np.empty(n, dtype=np.int32)
    lib = _lib.load()
    nc = lib.mg_host_greedy_color(n, A.indptr.ctypes.data, A.indices.ctypes.data, colors.ctypes.data)
    if nc < 0:
        _lib.check(nc, "mg_host_greedy_color")
    return colors, int(nc)


def lex_levels(A):
    """(level_ptr int64[nlev+1], level_rows int32[n]) of the index-order Gauss-Seidel dependency levels."""
    A = canonical_csr(A)
    n = A.shape[0]
    level = np.empty(n, dtype=np.int32)
    lib = _lib.load()
    nlev = lib.mg_host_lex_levels(n, A.indptr.ctypes.data, A.indices.ctypes.data, level.ctypes.data)
    if nlev < 0:
        _lib.check(int(nlev), "mg_host_lex_levels")
    order = np.argsort(level, kind="stable").astype(np.int32)
    counts = np.bincount(level, minlength=int(nlev))
    level_ptr = np.zeros(int(nlev) + 1, dtype=np.int64)
    np.cumsum(counts, out=level_ptr[1:])
    return level_ptr, order


def color_permutation(colors):
    """perm (new -> old) that groups rows by colour, natural order inside a colour; colour offsets."""
    colors = np.asarray(colors)
    ncolors = int(colors.max()) + 1 if len(colors) else 0
    perm = np.argsort(colors, kind="stable").astype(np.int32)
    color_ptr = np.zeros(ncolors + 1, dtype=np.int64)
    np.cumsum(np.bincount(colors, minlength=ncolors), out=color_ptr[1:])
    return perm, color_ptr


def inverse_permutation(perm):
    iperm = np.empty(len(perm), dtype=np.int32)
    iperm[perm] = np.arange(len(perm), dtype=np.int32)
    return iperm


def geometric_interpolator_csr(dimension):
    """Sparse form of the reference's dense 1D linear interpolation (Multigrid.interpolator,
    learn_multigrid/solvers/Multigrid.py:126-147): n x (floor((n-1)/2)+1), interior columns [1/2, 1, 1/2],
    first column [1, 1/2], last column [1/2, 1]."""
    rows_n = int(dimension)
    cols_n = int(np.floor((rows_n - 1) / 2)) + 1
    r, c, v = [0, 1], [0, 0], [1.0, 0.5]
    j = np.arange(1, cols_n - 1)
    i0 = 1 + 2 * (j - 1)
    r += list(np.concatenate([i0, i0 + 1, i0 + 2]))
    c += list(np.concatenate([j, j, j]))
    v += [0.5] * len(j) + [1.0] * len(j) + [0.5] * len(j)
    if cols_n >= 2 or rows_n >= 2:
        r += [rows_n - 1, rows_n - 2]
        c += [cols_n - 1, cols_n - 1]
        v += [1.0, 0.5]
    M = sp.coo_matrix((np.array(v), (np.array(r), np.array(c))), shape=(rows_n, cols_n))
    # duplicates (tiny n) follow the dense assignment semantics: last write wins, so rebuild via dense then
    if rows_n <= 4:
        D = np.zeros((rows_n, cols_n))
        ii = 1
        for jj in range(1, cols_n - 1):
            D[ii, jj] = 1; ii += 1
            D[ii, jj] = 2; ii += 1
            D[ii, jj] = 1
        D[0, 0] = 2; D[1, 0] = 1; D[-1, -1] = 2; D[-2, -1] = 1
        return canonical_csr(sp.csr_matrix(D / 2))
    return canonical_csr(M.tocsr())


def build_host_hierarchy(A, Q_list, smoother, colors=None, with_sell=True):
    """Pure NumPy/SciPy construction of every level's data in the engine's orderings (no device work).

    Returns a list of dicts (one per level) with: n, nnz_A, A_nat (canonical CSR, natural ordering), perm / iperm
    (None = natural), colors, color_ptr, and for all but the coarsest level: A (permuted CSR, entries in natural
    order inside rows), dinv, Q, QT (permuted CSR), Q_nat, nnz_Q, and with smoother == "lexgs" lex_ptr / lex_rows.
    With with_sell=True the SELL-32 arrays of A, Q, QT are added as (slice_ptr, cols, vals) under *_sell.
    The Galerkin products are SciPy's `csr_matrix(Q.T @ A @ Q)` (learn_multigrid/solvers/Multigrid.py:97-98).
    """
    L = len(Q_list) + 1
    A_nat = [solver_csr(A)]                            # Solver.py:18 stores csc_matrix(matrix)
    Q_nat = [canonical_csr(q) for q in Q_list]
    for l in range(L - 1):
        if Q_nat[l].shape[0] != A_nat[l].shape[0]:
            raise ValueError("Q_%d has %d rows, level operator has %d" % (l, Q_nat[l].shape[0], A_nat[l].shape[0]))
        A_nat.append(canonical_csr(sp.csr_matrix(Q_nat[l].T @ A_nat[l] @ Q_nat[l])))
    levels = []
    for l in range(L):
        d = {"n": A_nat[l].shape[0], "nnz_A": int(A_nat[l].nnz), "A_nat": A_nat[l]}
        if smoother == "mcgs" and l < L - 1:
            if colors is not None and colors[l] is not None:
                col = np.ascontiguousarray(colors[l], dtype=np.int32)
            else:
                col = greedy_colors(A_nat[l])[0]
            d["colors"] = col
            d["perm"], d["color_ptr"] = color_permutation(col)
            d["iperm"] = inverse_permutation(d["perm"])
        else:
            d["colors"] = d["perm"] = d["iperm"] = d["color_ptr"] = None
        levels.append(d)
    for l in range(L - 1):
        d, dc = levels[l], levels[l + 1]
        d["A"] = permute_csr(A_nat[l], d["perm"], d["iperm"])
        with np.errstate(divide="ignore"):
            dinv = 1.0 / A_nat[l].diagonal()
        d["dinv"] = np.ascontiguousarray(dinv if d["perm"] is None else dinv[d["perm"]])
        d["Q_nat"] = Q_nat[l]
        d["nnz_Q"] = int(Q_nat[l].nnz)
        d["Q"] = permute_csr(Q_nat[l], d["perm"], dc["iperm"])
        d["QT"] = permute_csr(transpose_csr(Q_nat[l]), dc["perm"], d["iperm"])
        if smoother == "lexgs":
            d["lex_ptr"], d["lex_rows"] = lex_levels(A_nat[l])
        if with_sell:
            for k in ("A", "Q", "QT"):
                d[k + "_sell"] = csr_to_sell(d[k])
    return levels


def greedy_colors_by_rounds(A):
    """The colouring of greedy_colors evaluated by dependency rounds (csrc/color_kernels.cu, host emulation of the
    device algorithm with the same per-row code): (colours, number of colours, rounds).  Test infrastructure for the
    device colouring; the product calls setup_device.DeviceSetup.first_fit_colors."""
    A = canonical_csr(A)
    n = A.shape[0]
    T = sp.csr_matrix((np.ones(A.nnz), A.indices, A.indptr), shape=A.shape).T.tocsr()
    T.sort_indices()
    tip, tix = T.indptr.astype(np.int32), T.indices.astype(np.int32)
    lib = _lib.load_testing()                    # the host emulation lives in libmgb200_testing.so
    colors = np.empty(max(n, 1), dtype=np.int32)
    work = np.zeros(int(lib.mg_color_workspace_size(n)), dtype=np.uint8)
    rounds = ctypes.c_int64(0)
    rc = lib.mg_host_color_rounds(n, A.indptr.ctypes.data, A.indices.ctypes.data, tip.ctypes.data, tix.ctypes.data,
                                  colors.ctypes.data, work.ctypes.data, ctypes.byref(rounds))
    if rc:
        _lib.check(rc, "mg_host_color_rounds")
    colors = colors[:n]
    return colors, (int(colors.max()) + 1 if n else 0), int(rounds.value)


SLICE_IRREGULAR = -2 ** 31


def sell_slice_offsets(sell, nrows, length):
    """Slice-relative columns of a UNIFORM SELL-32 matrix (every slice `length` entries per row): off[s, j] such that
    entry j of EVERY row r of slice s has column r + off[s, j]; slices where that does not hold (or that hold rows
    beyond the matrix) get off[s, 0] = SLICE_IRREGULAR.  On a structured stencil level nearly all slices are regular,
    so a kernel can compute the columns instead of loading them: 4*length bytes per slice instead of 128*length
    (csrc/sell_kernels.cu, mg_set_implied_columns).  Host twin of mg_sell_slice_offsets."""
    slice_ptr, cols, _ = sell
    nsl = len(slice_ptr) - 1
    off = np.full((nsl, max(length, 1)), SLICE_IRREGULAR, dtype=np.int32)
    if nsl == 0 or length <= 0:
        return off
    c = np.asarray(cols, dtype=np.int64).reshape(nsl, length, SLICE)          # [slice][entry][lane]
    rows = (np.arange(nsl, dtype=np.int64) * SLICE)[:, None, None] + np.arange(SLICE, dtype=np.int64)[None, None, :]
    rel = c - rows
    regular = np.all(rel == rel[:, :, :1], axis=(1, 2)) & ((np.arange(nsl) + 1) * SLICE <= nrows)
    off[regular] = rel[regular][:, :, 0].astype(np.int32)
    return off


def sell_slice_patterns(sell, nrows, length):
    """Slice patterns of a UNIFORM SELL-32 matrix (every slice `length` entries per row): base[s] = the column of entry 0
    of lane 0, delta[s, j, lane] = column - base[s] and vals[s, j, lane] the values, so that entry j of row 32 s + lane
    has column base[s] + delta[s, j, lane].  Unlike sell_slice_offsets this holds for every slice, whichever index space
    the columns live in (transfer operators: another level's colour-blocked numbering); what makes a slice cheap is that
    many slices share one (delta, vals) pattern.  full[s] = the slice holds no row beyond the matrix.  Host twin of
    pattern_records (which deduplicates the patterns on any torch device)."""
    slice_ptr, cols, vals = sell
    nsl = len(slice_ptr) - 1
    c = np.asarray(cols, dtype=np.int64).reshape(nsl, length, SLICE)          # [slice][entry][lane]
    base = c[:, 0, 0].copy() if nsl else np.zeros(0, dtype=np.int64)
    delta = c - base[:, None, None]
    full = (np.arange(nsl) + 1) * SLICE <= nrows
    return base, delta, np.asarray(vals, dtype=np.float64).reshape(nsl, length, SLICE), full


def pattern_records(torch, cols, vals, nrows, length, max_records=256, min_slices=2, chunk=1 << 16):
    """Deduplicated slice patterns of a uniform SELL-32 matrix with `length` <= 8 entries per row (engine.DeviceSell;
    sell_core.cuh, sell_pattern_kernel).  A slice keeps a 32-bit base column and a 16-bit record id; record r holds
    delta[r][j][lane] (int32) and vals[r][j][lane] (float64), and entry j of lane `lane` of the slice has the column
    base + delta and exactly that value (sell_slice_patterns defines base and delta).  Records are ranked by how many
    slices use them; at most `max_records` of those used by at least `min_slices` slices are kept (the table stays
    L1-sized), every other slice -- and a slice with rows beyond the matrix -- gets id -1 (0xffff to the kernels) and
    keeps reading its columns and values.

    Two 62-bit sums of the slice's pattern with fixed weights group the slices; each slice is then compared with the
    first slice of its group, entry by entry, so a hash collision only costs a slice its record, never a wrong column.
    Pure tensor code (any device): the CPU suite runs it on host tensors against sell_slice_patterns.
    Returns (base int32 [nslices], ids int16 [nslices], delta int32 [nrec, length, 32], vals f64 [nrec, length, 32],
    slices with a record)."""
    dev = cols.device
    nsl = int(cols.numel()) // (32 * length)
    K = 32 * length
    c = cols.view(nsl, K)
    base = c[:, 0].contiguous()
    vbits = vals.view(nsl, K).view(torch.int64)
    gen = torch.Generator().manual_seed(20251)
    w = torch.randint(1, 1 << 20, (2, 3, K), generator=gen, dtype=torch.int64).to(dev)

    def pattern(s):               # [n, 3K] int64 of the slices s (a range or an index tensor), elements in [-2^32, 2^32)
        d = c[s].to(torch.int64) - base[s].to(torch.int64)[:, None]
        v = vbits[s]
        return torch.cat([d, v >> 32, v & 0xffffffff], dim=1)

    keys = torch.empty(nsl, 2, dtype=torch.int64, device=dev)
    for s0 in range(0, nsl, chunk):      # |element| < 2^33, weight < 2^20, 3K <= 768 terms: no int64 overflow
        s = slice(s0, min(s0 + chunk, nsl))
        p = pattern(s)
        keys[s, 0] = (p * w[0].reshape(1, -1)).sum(dim=1)
        keys[s, 1] = (p * w[1].reshape(1, -1)).sum(dim=1)
    _, inverse, counts = torch.unique(keys, dim=0, return_inverse=True, return_counts=True)
    first = torch.full((counts.numel(),), nsl, dtype=torch.int64, device=dev)
    first.scatter_reduce_(0, inverse, torch.arange(nsl, device=dev), reduce="amin")
    ok = (torch.arange(nsl, device=dev) + 1) * 32 <= nrows
    for s0 in range(0, nsl, chunk):      # exact check against the group's first slice
        s = slice(s0, min(s0 + chunk, nsl))
        ok[s] &= (pattern(s) == pattern(first[inverse[s]])).all(dim=1)
    counts = torch.bincount(inverse[ok], minlength=counts.numel())
    order = torch.argsort(counts, descending=True, stable=True)
    order = order[counts[order] >= min_slices][:max_records]
    rank_of = torch.full((counts.numel(),), -1, dtype=torch.int64, device=dev)
    rank_of[order] = torch.arange(order.numel(), device=dev)
    ids = torch.where(ok, rank_of[inverse], torch.full_like(inverse, -1)).to(torch.int16)
    rep = first[order]
    delta = (c[rep].to(torch.int64) - base[rep, None].to(torch.int64)).to(torch.int32).view(-1, length, 32).contiguous()
    rvals = vals.view(nsl, K)[rep].view(-1, length, 32).contiguous()
    return base.to(torch.int32), ids, delta, rvals, int((ids >= 0).sum().item())


def slice_records(torch, off, val_idx=None, val_table=None, uniform_len=0, max_records=32766):
    """Deduplicated slice records of a uniform SELL-32 matrix (engine.DeviceSell; sell_core.cuh IMPL / IMPV kernels).

    off      : [nslices, 8] int32 tensor, the per-slice column offsets of mg_sell_slice_offsets (entries beyond
               uniform_len zero, irregular slices flagged by SLICE_IRREGULAR in column 0)
    val_idx  : optional uint8 tensor laid out like the matrix' values (value dictionary), val_table its <= 256 doubles

    A slice keeps two bytes, the id of its record (most frequent record = 0; -1, read as 0xffff by the kernels, = the
    slice is not regular).  With a dictionary, and if at most a tenth of the column-regular slices would be lost, a
    record also carries the VALUES: a slice then counts as regular only if its 32 rows hold the same value per entry
    (constant-coefficient stencil levels), and rec_vals[id] are those values.  Pure tensor code (any device): the CPU
    suite runs it on host tensors (tests/test_host_logic.py).
    Returns (ids int16 [nslices], rec_table int32 [nrec, 8], rec_vals float64 [nrec, 8] or None, regular_slices)."""
    nsl = int(off.shape[0])
    dev = off.device
    regular = off[:, 0] != SLICE_IRREGULAR
    n_regular = int(regular.sum().item())
    vrec = None
    if val_idx is not None and val_table is not None and uniform_len >= 1 and val_idx.numel() == nsl * 32 * uniform_len:
        v = val_idx.view(nsl, uniform_len, 32)
        same = (v == v[:, :, :1]).all(dim=2).all(dim=1)
        full = regular & same
        if n_regular > 0 and 10 * int(full.sum().item()) >= 9 * n_regular:
            vrec = torch.zeros(nsl, 8, dtype=torch.int32, device=dev)
            vrec[:, :uniform_len] = v[:, :, 0].to(torch.int32)
            regular = full
        del v, same, full
    keys = off if vrec is None else torch.cat([off, vrec], dim=1)
    recs, inverse, counts = torch.unique(keys[regular], dim=0, return_inverse=True, return_counts=True)
    order = torch.argsort(counts, descending=True)[:max_records]       # ids by frequency
    rank_of = torch.full((recs.shape[0],), -1, dtype=torch.int64, device=dev)
    rank_of[order] = torch.arange(order.numel(), device=dev)
    ids = torch.full((nsl,), -1, dtype=torch.int16, device=dev)
    ids[regular] = rank_of[inverse].to(torch.int16)
    rec_table = recs[order][:, :8].contiguous().to(torch.int32)
    rec_vals = None if vrec is None else val_table[recs[order][:, 8:16].long()].contiguous()
    return ids, rec_table, rec_vals, int((ids >= 0).sum().item())



# ---- Chebyshev smoother: coefficients, start vector, Lanczos (host twin) -------------------------------------------
CHEBY_LANCZOS_STEPS = 10
CHEBY_INTERVAL = (0.3, 1.1)       # default [lo, hi] as fractions of the Lanczos estimate of lambda_max(D^-1 A)


def chebyshev_check(degree, bounds=None):
    """ValueError unless degree is an integer >= 1 and bounds (None, or one (lo, hi) pair per smoothing level) has
    0 < lo < hi, both finite."""
    if isinstance(degree, bool) or not isinstance(degree, (int, np.integer)) or int(degree) < 1:
        raise ValueError("Chebyshev degree must be an integer >= 1, got %r" % (degree,))
    if bounds is None:
        return
    for b in bounds:
        lo, hi = (float(v) for v in b)
        if not (np.isfinite(lo) and np.isfinite(hi) and lo > 0.0 and hi > lo):
            raise ValueError("Chebyshev bounds need 0 < lo < hi, got (%r, %r)" % (lo, hi))


def chebyshev_coefficients(lo, hi, degree):
    """The (degree, 2) table of (c_d, c_r) of the Chebyshev smoother over [lo, hi] (c_d of step 0 is unused, 0 here).
    Step k of one application: dn = c_r t (k = 0) or (c_d d) + (c_r t), x += dn, d = dn, with t = D^-1 (b - A x).
    The error after `degree` steps is T_deg((theta - lambda)/delta) / T_deg(sigma) times the start error in every
    eigenvector of D^-1 A with eigenvalue lambda.  float64, in this exact order (the device cycle and the oracle read
    the same table)."""
    chebyshev_check(degree, [(lo, hi)])
    lo, hi = float(lo), float(hi)
    theta = (hi + lo) / 2.0
    delta = (hi - lo) / 2.0
    sigma = theta / delta
    rho = 1.0 / sigma
    out = np.zeros((int(degree), 2), dtype=np.float64)
    out[0, 1] = 1.0 / theta
    for k in range(1, int(degree)):
        rho_k = 1.0 / (2.0 * sigma - rho)
        out[k, 0] = rho_k * rho
        out[k, 1] = 2.0 * rho_k / delta
        rho = rho_k
    return out


def chebyshev_start_vector(idx):
    """Lanczos start vector: a counter-based hash of the GLOBAL row index (NumPy or torch int64 array, indices below
    2^31), uniform in [-1/2, 1/2).  Integer arithmetic only, so it is the same bits on the host, on any device, in any
    row ordering and on every rank."""
    M = 0xffffffff
    h = (idx * 2654435761) & M
    h = h ^ (h >> 16)
    h = (h * 0x45d9f3b) & M
    h = h ^ (h >> 16)
    h = (h * 0x45d9f3b) & M
    h = h ^ (h >> 16)
    f = h.astype(np.float64) if isinstance(h, np.ndarray) else h.double()
    return f * (1.0 / 4294967296.0) - 0.5


def lanczos_tridiagonal_max(alphas, betas):
    """largest eigenvalue of the symmetric tridiagonal Lanczos matrix (NumPy, float64)"""
    k = len(alphas)
    T = np.diag(np.asarray(alphas, dtype=np.float64))
    if k > 1:
        off = np.asarray(betas[:k - 1], dtype=np.float64)
        T += np.diag(off, 1) + np.diag(off, -1)
    return float(np.linalg.eigvalsh(T)[-1])


def lanczos_breakdown(beta, alphas):
    """Lanczos stops early when the new vector has (numerically) vanished: the Krylov space is invariant"""
    return not (beta > 1e-14 * max(abs(a) for a in alphas))


def chebyshev_lambda_max_host(A, steps=CHEBY_LANCZOS_STEPS):
    """Host twin (NumPy) of the device estimate of lambda_max(D^-1 A): `steps` Lanczos steps on D^-1/2 A D^-1/2 from
    chebyshev_start_vector, the same sequence of operations as setup_device.chebyshev_lambda_max."""
    A = sp.csr_matrix(A)
    d = A.diagonal()
    if not np.all(d > 0.0):
        raise ValueError("the Chebyshev smoother needs a positive diagonal")
    s = np.sqrt(1.0 / d)
    n = A.shape[0]
    v = chebyshev_start_vector(np.arange(n, dtype=np.int64))
    v = v * (1.0 / np.sqrt(np.dot(v, v)))
    v_prev = None
    alphas, betas = [], []
    beta = 0.0
    for k in range(int(steps)):
        w = s * (A @ (s * v))
        a = float(np.dot(w, v))
        w = w - a * v
        if v_prev is not None:
            w = w - beta * v_prev
        alphas.append(a)
        beta = float(np.sqrt(np.dot(w, w)))
        if k == steps - 1 or lanczos_breakdown(beta, alphas):
            break
        betas.append(beta)
        v_prev, v = v, w * (1.0 / beta)
    return lanczos_tridiagonal_max(alphas, betas)
