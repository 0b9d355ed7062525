"""Float64 host reference of the 2D NN transfer-operator builder (learnmultigrid_b200/neural2d.py), stage by stage, at
any size.

Coarsening, patch extraction and the fill_B contributions run the per-node code of csrc/nn_kernels.cu serially through
the mg_host_nn_* entry points of libmgb200_testing.so (pinned to the reference's golden vectors by
test_neural2d_host.py); compared with the device they check the parallel orchestration around that code: the
independent-set rounds, the launch indexing, where patch variants land, which patch's d_neighs survives.  The remaining
stages are plain NumPy / SciPy, independent of the CUDA code:

  fold        fill_B's running mean (Multigrid.py:687-732): contributions ordered by (row, col) with application order
              kept inside a run; an empty or exactly-0 entry takes the value, otherwise the mean of old and new; entries
              that end at exactly 0 are not stored
  normalise   Q = B / rowsum(B), the row sum added sequentially in column order (Multigrid.py:758-759)
  cut         pre_process (Multigrid.py:735-739): the diagonal plus the predicted neighbours, stored zeros dropped
  next_mass   csr_matrix(Q.T @ csc_matrix(M) @ Q), the expression DeviceSetup.galerkin reproduces bit for bit
"""
import ctypes

import numpy as np
import scipy.sparse as sp

from learnmultigrid_b200 import _lib
from learnmultigrid_b200 import formats as F


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _csr_arrays(M):
    return (np.ascontiguousarray(M.indptr, dtype=np.int32), np.ascontiguousarray(M.indices, dtype=np.int32),
            np.ascontiguousarray(M.data, dtype=np.float64))


def coarsen(M):
    """lexicographically first independent set (serial): (cmap, clist)"""
    lib = _lib.load_testing()
    n = M.shape[0]
    ip, ix, va = _csr_arrays(F.canonical_csr(M.T))
    cmap = np.empty(n, dtype=np.int32)
    clist = np.empty(n, dtype=np.int32)
    nc = lib.mg_host_nn_coarsen(n, _ptr(ip), _ptr(ix), _ptr(va), _ptr(cmap), _ptr(clist))
    if nc <= 0:
        raise _lib.MgError("mg_host_nn_coarsen: %s" % lib.mg_last_error().decode())
    return cmap, clist[:nc].copy()


def extract(M, cmap, clist):
    """patches (rows x 43) and fill indices (rows x 31); rows nc.. hold the extra variants in node order"""
    lib = _lib.load_testing()
    ip, ix, va = _csr_arrays(M)
    nc = len(clist)
    rows = lib.mg_host_nn_extract_patches(nc, _ptr(ip), _ptr(ix), _ptr(va), _ptr(cmap), _ptr(clist), None, None)
    patches = np.empty((rows, 43))
    fill = np.empty((rows, 31), dtype=np.int32)
    rc = lib.mg_host_nn_extract_patches(nc, _ptr(ip), _ptr(ix), _ptr(va), _ptr(cmap), _ptr(clist), _ptr(patches),
                                        _ptr(fill))
    if rc != rows:
        raise _lib.MgError("mg_host_nn_extract_patches: %s" % lib.mg_last_error().decode())
    return patches, fill


def not_last(fill, nc):
    """1 for every patch followed by another patch of the same node (only the last one sets d_neighs)"""
    node = fill[:, 0]
    last = np.full(int(node.max()) + 1, -1, dtype=np.int64)
    np.maximum.at(last, node, np.arange(len(node)))
    return (last[node] != np.arange(len(node))).astype(np.int32)


def contributions(fill, pred, cmap, n, nc):
    """(rows, cols, vals) of every prediction in application order (row n = unused) and the d_neighs table, written
    patch after patch"""
    lib = _lib.load_testing()
    m = fill.shape[0]
    fill = np.ascontiguousarray(fill, dtype=np.int32)
    pred = np.ascontiguousarray(pred, dtype=np.float64)
    rows = np.empty((m, 31), dtype=np.int32)
    cols = np.empty((m, 31), dtype=np.int32)
    vals = np.empty((m, 31))
    dn = np.full((nc, 6), -1, dtype=np.int32)
    _lib.check(lib.mg_host_nn_contributions(m, _ptr(fill), _ptr(pred), _ptr(cmap), n, _ptr(rows), _ptr(cols),
                                            _ptr(vals), _ptr(dn)), "mg_host_nn_contributions")
    return rows, cols, vals, dn


def fold(rows, cols, vals, n, nc, stats=None):
    """fill_B's running mean over contributions given in application order (entries with row >= n are unused).
    stats (a dict): receives 'cancelled', how often a contribution brought a nonzero entry back to exactly 0,
    'restarts', the contributions that then found it at 0, and 'dropped', the entries that end at exactly 0."""
    r, c, v = (np.asarray(a).ravel() for a in (rows, cols, vals))
    use = r < n
    r, c, v = r[use], c[use], v[use]
    o = np.lexsort((c, r))                          # by row, then column; stable, so application order within a run
    r, c, v = r[o], c[o], v[o]
    head = np.ones(len(r), dtype=bool)
    head[1:] = (r[1:] != r[:-1]) | (c[1:] != c[:-1])
    start = np.flatnonzero(head)
    run = np.cumsum(head) - 1
    pos = np.arange(len(r)) - start[run]
    cur = np.zeros(len(start))
    held = np.zeros(len(start), dtype=bool)             # the run's entry has been nonzero
    restarts = cancelled = 0
    for p in range(int(pos.max()) + 1 if len(r) else 0):
        at = pos == p
        k, x = run[at], v[at]
        empty = cur[k] == 0.0
        restarts += int((empty & held[k]).sum())
        cur[k] = np.where(empty, x, (cur[k] + x) / 2.0)
        cancelled += int((~empty & (cur[k] == 0.0)).sum())
        held[k] |= cur[k] != 0.0
    keep = cur != 0.0
    br, bc, bv = r[start][keep], c[start][keep], cur[keep]
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(br, minlength=n), out=indptr[1:])
    if stats is not None:
        stats["restarts"] = restarts
        stats["cancelled"] = cancelled
        stats["dropped"] = int((~keep).sum())
    return F.raw_csr(indptr, bc, bv, (n, nc))


def normalise(B):
    """Q = B / rowsum(B), each row sum added in column order one entry at a time"""
    n = B.shape[0]
    lens = np.diff(B.indptr)
    s = np.zeros(n)
    for p in range(int(lens.max()) if n else 0):
        rows = np.flatnonzero(lens > p)
        s[rows] += B.data[B.indptr[rows] + p]
    return F.raw_csr(B.indptr, B.indices, B.data / np.repeat(s, lens), B.shape)


def cut(M, dneigh):
    """pre_process: of row i keep the diagonal and the columns dneigh[i] lists (-1 = none); stored zeros dropped"""
    n = M.shape[0]
    row = np.repeat(np.arange(n), np.diff(M.indptr))
    keep = (M.indices == row) | (np.asarray(dneigh)[row] == M.indices[:, None]).any(axis=1)
    keep &= M.data != 0.0
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(row[keep], minlength=n), out=indptr[1:])
    return F.raw_csr(indptr, M.indices[keep], M.data[keep], M.shape)


def next_mass(M, Q):
    A = sp.csr_matrix(Q.T @ sp.csc_matrix(M) @ Q)
    A.sort_indices()
    return F.raw_csr(A.indptr, A.indices, A.data, A.shape)


def define_hierarchy(M, predictor, mean, std, levels):
    """NeuralMG_2D.define_hierarchy (Multigrid.py:741-765) with every intermediate kept, one dict per level:
    M (the level's matrix, cut for levels >= 1), M_full (before the cut, levels >= 1), cmap, clist, patches, fill,
    not_last, pred, B, dneigh, Q and stats (fold's counters)"""
    mean = np.broadcast_to(np.asarray(mean, dtype=np.float64), (43,))
    std = np.broadcast_to(np.asarray(std, dtype=np.float64), (43,))
    mass = F.canonical_csr(M)
    out, dneigh = [], None
    for i in range(levels - 1):
        lv = {}
        if dneigh is not None:
            lv["M_full"] = mass
            mass = cut(mass, dneigh)
        n = mass.shape[0]
        cmap, clist = coarsen(mass)
        nc = len(clist)
        patches, fill = extract(mass, cmap, clist)
        pred = np.ascontiguousarray(predictor.predict((patches - mean) / std), dtype=np.float64)
        rows, cols, vals, dneigh = contributions(fill, pred, cmap, n, nc)
        stats = {}
        B = fold(rows, cols, vals, n, nc, stats)
        Q = normalise(B)
        lv.update(M=mass, cmap=cmap, clist=clist, patches=patches, fill=fill, not_last=not_last(fill, nc), pred=pred,
                  B=B, dneigh=dneigh, Q=Q, stats=stats)
        out.append(lv)
        if i + 1 < levels - 1:
            mass = next_mass(mass, Q)
    return out
