"""NumPy/SciPy restatement of the classical AMG setup (test infrastructure), written from the definition in DESIGN.md
§4.10, not from the CUDA:

  1. strength      j != i is in S_i iff -a_ij > 0 and -a_ij >= theta * max_{k != i}(-a_ik); theta in [0, 1)
  2. weights       w_i = |S^T_i| + r_i, r_i = formats.chebyshev_start_vector(i) + 0.5; (w_i, i) compared lexicographically
  3. PMIS          points with an empty S^T_i start F, the others undecided; per round: select (an undecided i turns C iff
                   its (w_i, i) beats every undecided j in S_i and S^T_i), then mark (an undecided i with a C point in S_i
                   turns F); until nothing is undecided
  4. promotion     an F point with a non-empty S_i and no C point in S_i turns C (one pass over the final states)
  5. numbering     C points in ascending fine index
  6. interpolation C row: 1 at cmap[i]; F row: sn_all = sum_{k != i, a_ik < 0} a_ik, sp_all = sum_{k != i, a_ik > 0} a_ik,
                   sn_str = sum_{k in S_i n C} a_ik (storage order), alpha = sn_all / sn_str, d = a_ii + sp_all,
                   coef = -alpha / d, Q[i, cmap[j]] = coef * a_ij for j in S_i n C
  7. recursion     A_c = Q^T A Q (oracle.vcycle.galerkin); a level with n_c = 0 or n_c = n is a ValueError

NumPy rounds every elementwise product, sum and quotient on its own, and the sums below run over the row entries in
storage order, one entry position at a time for all rows -- the order of the device's one-thread-per-row loops.
"""
import numpy as np
import scipy.sparse as sp

from learnmultigrid_b200 import formats as F
from oracle.vcycle import galerkin

UNDECIDED, C_POINT, F_POINT = 0, 1, 2


def check_theta(theta):
    theta = float(theta)
    if not 0.0 <= theta < 1.0:
        raise ValueError("theta must be in [0, 1)")
    return theta


def _csr_from_mask(A, keep):
    """the entries of A flagged in `keep` (one flag per stored entry), in storage order, as a CSR matrix"""
    n = A.shape[0]
    rows = np.repeat(np.arange(n), np.diff(A.indptr))
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(rows[keep], minlength=n), out=indptr[1:])
    return F.raw_csr(indptr, A.indices[keep], A.data[keep], A.shape)


def strength(A, theta=0.25):
    theta = check_theta(theta)
    A = F.canonical_csr(A)
    n = A.shape[0]
    rows = np.repeat(np.arange(n), np.diff(A.indptr))
    neg = -A.data
    off = A.indices != rows
    m = np.zeros(n)
    sel = off & (neg > 0.0)
    np.maximum.at(m, rows[sel], neg[sel])
    thr = theta * m
    return _csr_from_mask(A, off & (neg > 0.0) & (neg >= thr[rows]))


def transpose_counts(S):
    return np.bincount(S.indices, minlength=S.shape[0])


def weights(S):
    n = S.shape[0]
    return transpose_counts(S).astype(np.float64) + (F.chebyshev_start_vector(np.arange(n, dtype=np.int64)) + 0.5)


def _pattern(M):
    P = sp.csr_matrix((np.ones(len(M.indices)), M.indices, M.indptr), shape=M.shape)
    return P


def _row_max(G, v):
    """max over the stored columns j of row i of v[j] (0 for an empty row)"""
    out = np.zeros(G.shape[0])
    vals = v[G.indices]
    nonempty = np.flatnonzero(np.diff(G.indptr) > 0)
    if len(nonempty):
        out[nonempty] = np.maximum.reduceat(vals, G.indptr[nonempty])
    return out


def pmis(S):
    """(states before promotion, rounds, [(C points chosen, F points marked) per round])"""
    n = S.shape[0]
    w = weights(S)
    order = np.lexsort((np.arange(n), w))            # ascending (w, i)
    rank = np.empty(n, dtype=np.float64)
    rank[order] = np.arange(1, n + 1)
    Sp = _pattern(S)
    G = sp.csr_matrix(Sp + Sp.T)
    G.sort_indices()
    state = np.where(transpose_counts(S) == 0, F_POINT, UNDECIDED).astype(np.int32)
    history = []
    while np.any(state == UNDECIDED):
        und = state == UNDECIDED
        best = _row_max(G, np.where(und, rank, 0.0))
        new_c = und & (rank > best)
        state[new_c] = C_POINT
        has_c = (Sp @ (state == C_POINT).astype(np.float64)) > 0
        new_f = (state == UNDECIDED) & has_c
        state[new_f] = F_POINT
        history.append((np.flatnonzero(new_c), np.flatnonzero(new_f)))
        if len(history) > n:
            raise RuntimeError("PMIS made no progress")
    return state, len(history), history


def promote(S, state):
    Sp = _pattern(S)
    has_c = (Sp @ (state == C_POINT).astype(np.float64)) > 0
    promo = (state == F_POINT) & (np.diff(S.indptr) > 0) & ~has_c
    out = state.copy()
    out[promo] = C_POINT
    return out, np.flatnonzero(promo)


def _storage_order_sum(M, take):
    """per row: sum of M's values where take (per stored entry) holds, added one entry position at a time"""
    n = M.shape[0]
    lens = np.diff(M.indptr)
    acc = np.zeros(n)
    for k in range(int(lens.max()) if n else 0):
        r = np.flatnonzero(lens > k)
        p = M.indptr[r] + k
        t = take[p]
        acc[r[t]] = acc[r[t]] + M.data[p[t]]
    return acc


def interpolate(A, S, state):
    """(Q as canonical CSR n x n_c, cmap)"""
    A = F.canonical_csr(A)
    n = A.shape[0]
    is_c = state == C_POINT
    cmap = np.where(is_c, np.cumsum(is_c) - 1, -1).astype(np.int64)
    nc = int(is_c.sum())
    rows = np.repeat(np.arange(n), np.diff(A.indptr))
    off = A.indices != rows
    sn_all = _storage_order_sum(A, off & (A.data < 0.0))
    sp_all = _storage_order_sum(A, off & (A.data > 0.0))
    a_ii = np.zeros(n)
    a_ii[rows[~off]] = A.data[~off]
    srows = np.repeat(np.arange(n), np.diff(S.indptr))
    s_c = is_c[S.indices]
    sn_str = _storage_order_sum(S, s_c)
    f_int = (state == F_POINT) & (np.bincount(srows[s_c], minlength=n) > 0)
    with np.errstate(divide="ignore", invalid="ignore"):
        alpha = sn_all / sn_str
        d = a_ii + sp_all
        coef = -alpha / d
    bad = np.flatnonzero(f_int & (d == 0.0))
    if len(bad):
        raise ValueError("a_ii + sp_all is 0 in row %d" % bad[0])
    take = f_int[srows] & s_c
    r = np.concatenate([np.flatnonzero(is_c), srows[take]])
    c = np.concatenate([cmap[is_c], cmap[S.indices[take]]])
    v = np.concatenate([np.ones(nc), coef[srows[take]] * S.data[take]])
    o = np.lexsort((c, r))
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(r, minlength=n), out=indptr[1:])
    return F.raw_csr(indptr, c[o], v[o], (n, nc)), cmap


def level(A, theta=0.25):
    """one level: dict with S, the PMIS states, rounds, per-round history, the promoted points, final states, Q, cmap"""
    S = strength(A, theta)
    st0, rounds, history = pmis(S)
    st1, promoted = promote(S, st0)
    Q, cmap = interpolate(A, S, st1)
    return {"S": S, "pmis_state": st0, "rounds": rounds, "history": history, "promoted": promoted, "state": st1,
            "Q": Q, "cmap": cmap}


def hierarchy(A, levels, theta=0.25):
    """(Q list, level operators A_0 .. A_{levels-1}, per-level dicts of `level`)"""
    theta = check_theta(theta)
    Al = F.canonical_csr(A)
    Qs, As, info = [], [Al], []
    for l in range(levels - 1):
        d = level(Al, theta)
        nc = d["Q"].shape[1]
        if nc == 0 or nc == Al.shape[0]:
            raise ValueError("AMG coarsening of level %d stalls (%d of %d points C)" % (l, nc, Al.shape[0]))
        Qs.append(d["Q"])
        info.append(d)
        Al = galerkin(Al, d["Q"])
        As.append(Al)
    return Qs, As, info


def convergence_factor(track_res):
    """geometric mean reduction per cycle, from the second history entry on (the first is the sqrt(n) quirk)"""
    r = np.asarray(track_res).ravel()
    return float((r[-1] / r[1]) ** (1.0 / (len(r) - 2)))


def random_m_matrix(n=600, degree=6, seed=5):
    """seeded symmetric positive definite M-matrix: a random weighted graph Laplacian plus a small diagonal shift"""
    rng = np.random.default_rng(seed)
    i = np.repeat(np.arange(n), degree)
    j = rng.integers(0, n, size=n * degree)
    keep = i != j
    W = sp.coo_matrix((rng.uniform(0.1, 1.0, size=int(keep.sum())), (i[keep], j[keep])), shape=(n, n)).tocsr()
    W = W + W.T
    L = sp.diags(np.asarray(W.sum(axis=1)).ravel() + rng.uniform(0.0, 0.05, size=n)) - W
    return F.canonical_csr(L)


def zero_denominator_matrix():
    """6 x 6: identity rows except row 4 = [0, -2, 0, 0, -1, 1].  Row 4 is F and interpolates from the C point 1, and
    a_44 + sp_all = -1 + 1 = 0: direct interpolation is undefined there"""
    A = sp.lil_matrix(sp.identity(6))
    A[4, 1], A[4, 4], A[4, 5] = -2.0, -1.0, 1.0
    return F.canonical_csr(sp.csr_matrix(A))


def cpu_problems():
    """the matrices of the CPU tests: Poisson with row-replaced Dirichlet rows, a variable coefficient, an irregular
    P1 mesh and a random M-matrix"""
    from helpers import poisson2d
    from learnmultigrid_b200 import problems as P
    return {"poisson": poisson2d(32), "variable": P.structured_laplacian_2d(32, P.variable_coefficient),
            "irregular": P.irregular_p1_2d(32)["A"], "random": random_m_matrix()}


# V(1,1) convergence factors of the oracle's cycles with the oracle's operators on the problems above (right-hand side
# standard normal with seed 0, zero start, until ||r|| <= 1e-10 ||b|| or 60 cycles), measured on the CPU, rounded up to
# two digits with a margin of 0.02.  The device cycles are held to the same bounds.
#   measured (levels 3 / 4):  poisson    gs .529/.566  jacobi .643/.694  mcgs .518/.557  cheby .556/.598
#                             variable   gs .489/.549  jacobi .618/.673  mcgs .474/.537  cheby .513/.583
#                             irregular  gs .550/.590  jacobi .695/.736  mcgs .544/.588  cheby .585/.621
#                             random     gs .066/.066  jacobi .410/.410  mcgs .065/.065  cheby .042/.042
FACTOR_BOUNDS = {
    "poisson": {3: {"gs": 0.55, "jacobi": 0.67, "mcgs": 0.54, "cheby": 0.58},
                4: {"gs": 0.59, "jacobi": 0.72, "mcgs": 0.58, "cheby": 0.62}},
    "variable": {3: {"gs": 0.51, "jacobi": 0.64, "mcgs": 0.50, "cheby": 0.54},
                 4: {"gs": 0.57, "jacobi": 0.70, "mcgs": 0.56, "cheby": 0.61}},
    "irregular": {3: {"gs": 0.57, "jacobi": 0.72, "mcgs": 0.57, "cheby": 0.61},
                  4: {"gs": 0.62, "jacobi": 0.76, "mcgs": 0.61, "cheby": 0.65}},
    "random": {3: {"gs": 0.09, "jacobi": 0.43, "mcgs": 0.09, "cheby": 0.07},
               4: {"gs": 0.09, "jacobi": 0.43, "mcgs": 0.09, "cheby": 0.07}},
}
