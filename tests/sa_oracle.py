"""NumPy/SciPy restatement of the smoothed aggregation setup (test infrastructure), written from the definition in
DESIGN.md §4.11, not from the CUDA:

  1. strength      j in S_i iff j != i, a_ij != 0 and a_ij * a_ij >= theta2 * (|a_ii| * |a_jj|), theta2 = theta * theta,
                   theta in [0, 1); S keeps the values a_ij in storage order
  2. graph         N_i = S_i u S^T_i; a point with an empty N_i is isolated
  3. MIS(2)        keys (state, r_i, i) compared lexicographically, r_i = formats.chebyshev_start_vector(i) + 0.5,
                   OUT = 0 < UNDECIDED = 1 < IN = 2; isolated points start OUT, the others undecided; per round
                   K1_i = max over {i} u N_i of K0_j, K2_i = max over {i} u N_i of K1_j, then an undecided i turns IN if
                   K2_i is its own key, OUT if K2_i has state IN; until nothing is undecided
  4. numbering     roots (IN) in ascending fine index
  5. aggregation   pass 1: a non-root non-isolated i with a root in N_i joins it (that root is unique); pass 2: a point
                   still unassigned joins the aggregate of its pass-1-assigned neighbour j with the largest (r_j, j)
  6. tentative     nu_a = sqrt(sum_{i in a} B_i * B_i) in ascending i, T[i, agg(i)] = B_i / nu_agg(i), next B = nu
  7. smoothing     omega_hat = omega / lambda_max, s_i = omega_hat / a_ii, At_ij = -(s_i * a_ij) (j != i),
                   At_ii = 1 - s_i * a_ii on A's pattern, P = At @ T (SciPy; exact zeros pruned; columns sorted)
  8. recursion     A_c = P^T A P (oracle.vcycle.galerkin); a level with n_c = 0 or n_c = n is a ValueError

lambda_max per level is an input: the device's value for bit comparisons, formats.chebyshev_lambda_max_host otherwise.
NumPy rounds every elementwise product, sum, quotient and square root on its own.
"""
import numpy as np
import scipy.sparse as sp

from learnmultigrid_b200 import formats as F
from oracle.vcycle import galerkin

OUT, UNDECIDED, IN = 0, 1, 2


def check_theta(theta):
    theta = float(theta)
    if not 0.0 <= theta < 1.0:
        raise ValueError("theta must be in [0, 1)")
    return theta


def check_omega(omega):
    omega = float(omega)
    if not 0.0 < omega < 2.0:
        raise ValueError("omega must be in (0, 2)")
    return omega


def r_hash(n):
    return F.chebyshev_start_vector(np.arange(n, dtype=np.int64)) + 0.5


def diagonal(A):
    """the stored a_ii of every row, 0 where none is stored"""
    n = A.shape[0]
    rows = np.repeat(np.arange(n), np.diff(A.indptr))
    d = np.zeros(n)
    on = A.indices == rows
    d[rows[on]] = A.data[on]
    return d


def strength(A, theta=0.0):
    theta = check_theta(theta)
    A = F.canonical_csr(A)
    n = A.shape[0]
    theta2 = theta * theta
    rows = np.repeat(np.arange(n), np.diff(A.indptr))
    d = np.abs(diagonal(A))
    a = A.data
    keep = (A.indices != rows) & (a != 0.0) & (a * a >= theta2 * (d[rows] * d[A.indices]))
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(rows[keep], minlength=n), out=indptr[1:])
    return F.raw_csr(indptr, A.indices[keep], A.data[keep], A.shape)


def neighbours(S):
    """the pattern of S u S^T (no diagonal) as CSR with sorted columns, and the isolated points"""
    P = sp.csr_matrix((np.ones(S.nnz), S.indices, S.indptr), shape=S.shape)
    G = sp.csr_matrix(P + P.T)
    G.sort_indices()
    return G, np.diff(G.indptr) == 0


def _row_max_self(G, v):
    """max of v over {i} u (the columns of row i)"""
    out = v.copy()
    nonempty = np.flatnonzero(np.diff(G.indptr) > 0)
    if len(nonempty):
        out[nonempty] = np.maximum(out[nonempty], np.maximum.reduceat(v[G.indices], G.indptr[nonempty]))
    return out


def mis2(S):
    """(final states, rounds, [(points turned IN, points turned OUT) per round])"""
    n = S.shape[0]
    G, isolated = neighbours(S)
    r = r_hash(n)
    idx = np.arange(n)
    state = np.where(isolated, OUT, UNDECIDED).astype(np.int32)
    history = []
    while np.any(state == UNDECIDED):
        # the key (state, r, i) of every point as its rank among all keys of the round
        order = np.lexsort((idx, r, state))
        rank = np.empty(n, dtype=np.int64)
        rank[order] = np.arange(n)
        k2 = _row_max_self(G, _row_max_self(G, rank))
        und = state == UNDECIDED
        new_in = und & (k2 == rank)
        new_out = und & ~new_in & (state[order[k2]] == IN)
        state = state.copy()
        state[new_in], state[new_out] = IN, OUT
        history.append((np.flatnonzero(new_in), np.flatnonzero(new_out)))
        if len(history) > n:
            raise RuntimeError("MIS(2) made no progress")
    return state, len(history), history


def aggregate(S, state):
    """(agg per point, -1 for an unaggregated point; number of aggregates).  ValueError names a point with two roots
    among its neighbours or a non-isolated point left unassigned"""
    n = S.shape[0]
    G, isolated = neighbours(S)
    is_root = state == IN
    cmap = np.where(is_root, np.cumsum(is_root) - 1, -1)
    nc = int(is_root.sum())
    grow = np.repeat(np.arange(n), np.diff(G.indptr))
    root_nb = is_root[G.indices]
    n_roots = np.bincount(grow[root_nb], minlength=n)
    two = np.flatnonzero(~is_root & (n_roots > 1))
    if len(two):
        raise ValueError("point %d has two roots among its neighbours" % two[0])
    agg1 = np.full(n, -1, dtype=np.int64)
    agg1[is_root] = cmap[is_root]
    join = root_nb & ~is_root[grow]
    agg1[grow[join]] = cmap[G.indices[join]]
    # pass 2: the pass-1-assigned neighbour with the largest (r_j, j), as its rank (1..n) among all points
    r = r_hash(n)
    order = np.lexsort((np.arange(n), r))
    rank = np.empty(n, dtype=np.int64)
    rank[order] = np.arange(1, n + 1)
    best = np.zeros(n, dtype=np.int64)
    nonempty = np.flatnonzero(np.diff(G.indptr) > 0)
    if len(nonempty):
        best[nonempty] = np.maximum.reduceat(np.where(agg1[G.indices] >= 0, rank[G.indices], 0), G.indptr[nonempty])
    agg = agg1.copy()
    todo = (agg1 < 0) & ~isolated
    take = todo & (best > 0)
    agg[take] = agg1[order[best[take] - 1]]
    left = np.flatnonzero(todo & (best == 0))
    if len(left):
        raise ValueError("point %d is left unassigned" % left[0])
    return agg, nc


def tentative(agg, nc, B):
    """(T as canonical CSR n x n_c, nu)"""
    n = len(agg)
    on = agg >= 0
    members = np.flatnonzero(on)                       # ascending i
    a = agg[members]
    nu2 = np.zeros(nc)
    # sum in ascending member index, one member position at a time for all aggregates
    o = np.argsort(a, kind="stable")
    a_sorted, m_sorted = a[o], members[o]
    starts = np.searchsorted(a_sorted, np.arange(nc))
    pos = np.arange(len(a_sorted)) - starts[a_sorted]
    for k in range(int(pos.max()) + 1 if len(pos) else 0):
        sel = pos == k
        b = B[m_sorted[sel]]
        nu2[a_sorted[sel]] = nu2[a_sorted[sel]] + b * b
    nu = np.sqrt(nu2)
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(on, out=indptr[1:])
    return F.raw_csr(indptr, a, B[members] / nu[a], (n, nc)), nu


def smooth(A, T, lam, omega=4.0 / 3.0):
    """(P, At, omega_hat)"""
    omega = check_omega(omega)
    A = F.canonical_csr(A)
    n = A.shape[0]
    d = diagonal(A)
    if not np.all(d > 0.0):
        raise ValueError("smoothed aggregation needs a positive diagonal; row %d" % np.flatnonzero(~(d > 0.0))[0])
    omega_hat = omega / lam
    s = omega_hat / d
    rows = np.repeat(np.arange(n), np.diff(A.indptr))
    sa = s[rows] * A.data
    vals = np.where(A.indices == rows, 1.0 - sa, -sa)
    At = F.raw_csr(A.indptr, A.indices, vals, A.shape)
    P = sp.csr_matrix(At @ T)
    P.sort_indices()
    return P, At, omega_hat


def level(A, B, lam=None, theta=0.0, omega=4.0 / 3.0, l=0):
    """one level: dict with S, the MIS(2) states, rounds and per-round history, agg, nu, T, At, P, lambda_max,
    omega_hat and the number of isolated points"""
    A = F.canonical_csr(A)
    S = strength(A, theta)
    state, rounds, history = mis2(S)
    nc = int((state == IN).sum())
    if nc == 0 or nc == A.shape[0]:
        raise ValueError("smoothed aggregation of level %d stalls (%d aggregates of %d points)" % (l, nc, A.shape[0]))
    agg, _ = aggregate(S, state)
    T, nu = tentative(agg, nc, B)
    if lam is None:
        lam = F.chebyshev_lambda_max_host(A)
    P, At, omega_hat = smooth(A, T, lam, omega)
    return {"S": S, "state": state, "rounds": rounds, "history": history, "agg": agg, "nc": nc, "nu": nu, "T": T,
            "At": At, "P": P, "lambda_max": lam, "omega_hat": omega_hat,
            "isolated": int(neighbours(S)[1].sum())}


def hierarchy(A, levels, theta=0.0, omega=4.0 / 3.0, lambdas=None):
    """(P list, level operators A_0 .. A_{levels-1}, per-level dicts of `level`)"""
    theta, omega = check_theta(theta), check_omega(omega)
    Al = F.canonical_csr(A)
    B = np.ones(Al.shape[0])
    Ps, As, info = [], [Al], []
    for l in range(levels - 1):
        d = level(Al, B, None if lambdas is None else lambdas[l], theta, omega, l)
        Ps.append(d["P"])
        info.append(d)
        Al = galerkin(Al, d["P"])
        As.append(Al)
        B = d["nu"]
    return Ps, As, info


def zero_diagonal_matrix():
    """5 x 5 path Laplacian with a_22 = 0"""
    A = sp.diags([-np.ones(4), 2.0 * np.ones(5), -np.ones(4)], [-1, 0, 1]).tolil()
    A[2, 2] = 0.0
    return F.canonical_csr(sp.csr_matrix(A))


# V(1,1) convergence factors of the oracle's cycles with the oracle's SA operators (theta 0, omega 4/3, lambda_max from
# the host Lanczos twin) on amg_oracle.cpu_problems() (right-hand side standard normal with seed 0, zero start, until
# ||r|| <= 1e-10 ||b|| or 60 cycles), measured on the CPU, rounded up to two digits with a margin of 0.02.  The device
# cycles are held to the same bounds.  The random M-matrix coarsens to one row at 3 levels, so it has no 4-level bound.
#   measured (levels 3 / 4):  poisson    gs .416/.422  jacobi .717/.718  mcgs .437/.433  cheby .427/.427
#                             variable   gs .447/.447  jacobi .708/.710  mcgs .435/.432  cheby .424/.425
#                             irregular  gs .681/.680  jacobi .824/.824  mcgs .676/.675  cheby .653/.653
#                             random     gs .099/-     jacobi .472/-     mcgs .094/-     cheby .047/-
FACTOR_BOUNDS_SA = {
    "poisson": {3: {"gs": 0.44, "jacobi": 0.74, "mcgs": 0.46, "cheby": 0.45},
                4: {"gs": 0.45, "jacobi": 0.74, "mcgs": 0.46, "cheby": 0.45}},
    "variable": {3: {"gs": 0.47, "jacobi": 0.73, "mcgs": 0.46, "cheby": 0.45},
                 4: {"gs": 0.47, "jacobi": 0.73, "mcgs": 0.46, "cheby": 0.45}},
    "irregular": {3: {"gs": 0.71, "jacobi": 0.85, "mcgs": 0.70, "cheby": 0.68},
                  4: {"gs": 0.71, "jacobi": 0.85, "mcgs": 0.70, "cheby": 0.68}},
    "random": {3: {"gs": 0.12, "jacobi": 0.50, "mcgs": 0.12, "cheby": 0.07}},
}
