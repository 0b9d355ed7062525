"""NumPy restatement of the coarsest-level block cyclic reduction (coarse.BcrCoarse, csrc/bcr.cu::bcr_solve).

The operator, with half bandwidth <= m, is cut into nb block rows of m unknowns; the last block is filled up with
identity rows.  Each reduction level keeps the even block positions and eliminates the odd ones:

    Dinv[j] = D[2j+1]^-1,  HL[j] = Dinv[j] L[2j+1],  HU[j] = Dinv[j] U[2j+1]                  (j < na // 2)
    GL[j] = L[2j] Dinv[j-1]  (j >= 1, else 0),   GU[j] = U[2j] Dinv[j]  (j < na // 2, else 0)   (j < (na + 1) // 2)
    D'[j] = D[2j] - GL[j] U[2j-1] - GU[j] L[2j+1],  L'[j] = -GL[j] L[2j-1],  U'[j] = -GU[j] U[2j+1]

until at most `tail_blocks` block rows are left; that block-tridiagonal tail is assembled densely and inverted
(`last_inv`).  The solve runs the forward updates f[2j] -= GL[j] f[2j-1] + GU[j] f[2j+1] level by level, applies
`last_inv` to the tail, and recovers the odd blocks on the way back, x[2j+1] = Dinv[j] f[2j+1] - HL[j] x[2j] -
HU[j] x[2j+2].

Everything is computed in the dtype given (float64, or np.longdouble to measure the float64 rounding error).  NumPy's
LAPACK has no extended precision, so an extended inverse is the float64 inverse polished by Newton-Schulz steps.
"""
import numpy as np
import scipy.sparse as sp


def banded_spd(n, half_bw, seed=0):
    """random symmetric positive definite matrix of exactly the given half bandwidth (strict diagonal dominance)"""
    rng = np.random.default_rng(seed)
    diags = [rng.uniform(-1.0, 0.0, n - k) for k in range(1, half_bw + 1)]
    diags[-1][rng.integers(n - half_bw)] = -1.0           # the outermost diagonal is never empty
    off = sp.diags(diags, list(range(1, half_bw + 1)), shape=(n, n))
    A = off + off.T
    d = np.asarray(abs(A).sum(axis=1)).ravel() + rng.uniform(0.05, 1.0, n)
    return sp.csr_matrix(A + sp.diags(d))


def layered_graph_matrix(layers=6, width=4400, degree=3, seed=0):
    """SPD matrix of a layered random graph: every node has `degree` random -1 couplings inside its layer and as many
    into the next one, the graph is symmetrised, and each diagonal entry is its row's absolute sum plus one.  Its half
    bandwidth (about 2 * width) stays large after reverse Cuthill-McKee."""
    rng = np.random.default_rng(seed)
    n = layers * width
    node = np.arange(n)
    layer = node // width
    rows, cols = [], []
    for shift in (0, 1):
        src = np.repeat(node[layer + shift < layers], degree)
        dst = (layer[src] + shift) * width + rng.integers(0, width, len(src))
        keep = src != dst
        rows.append(src[keep])
        cols.append(dst[keep])
    r, c = np.concatenate(rows), np.concatenate(cols)
    G = sp.csr_matrix((np.ones(len(r)), (r, c)), shape=(n, n))
    G = ((G + G.T) > 0).astype(np.float64)
    A = sp.diags(np.asarray(G.sum(axis=1)).ravel() + 1.0) - G
    return sp.csr_matrix(A)


def geometry(n, half_bw, min_block=64, tail_blocks=8):
    """the block size, block count and reduction levels BcrCoarse chooses for n unknowns of half bandwidth half_bw"""
    m = max(int(half_bw), int(min_block), 1)
    nb = (n + m - 1) // m
    nas = []
    na = nb
    while na > max(int(tail_blocks), 1):
        nas.append(na)
        na = (na + 1) // 2
    return {"m": m, "nb": nb, "n_pad": nb * m, "na": nas, "tail_na": na, "padding": nb * m - n}


def blocks(A, m, nb, dtype=np.float64):
    """(D, L, U), each [nb, m, m]: row block i of A is L[i] x[i-1] + D[i] x[i] + U[i] x[i+1]; padding rows are identity"""
    A = sp.coo_matrix(A)
    n = A.shape[0]
    r, c = A.row.astype(np.int64), A.col.astype(np.int64)
    bi, bj = r // m, c // m
    if np.any(np.abs(bj - bi) > 1):
        raise ValueError("entries outside the block-tridiagonal band")
    D, L, U = (np.zeros((nb, m, m), dtype=dtype) for _ in range(3))
    for dst, sel in ((D, bj == bi), (L, bj == bi - 1), (U, bj == bi + 1)):
        np.add.at(dst, (bi[sel], r[sel] % m, c[sel] % m), A.data[sel].astype(dtype))
    pad = np.arange(n, nb * m)
    D[pad // m, pad % m, pad % m] = 1
    return D, L, U


def inverse(A):
    """inverse of a matrix or a stack of matrices, accurate to the working precision of A's dtype"""
    X = np.linalg.inv(A.astype(np.float64)).astype(A.dtype)
    if A.dtype != np.float64:
        eye = np.eye(A.shape[-1], dtype=A.dtype)
        for _ in range(3):
            X = X @ (2 * eye - A @ X)
    return X


class BcrOracle:
    def __init__(self, A, half_bw, min_block=64, tail_blocks=8, dtype=np.float64):
        n = A.shape[0]
        g = geometry(n, half_bw, min_block, tail_blocks)
        self.n, self.geometry = n, g
        m, nb = g["m"], g["nb"]
        self.m, self.nb, self.n_pad = m, nb, g["n_pad"]
        D, L, U = blocks(A, m, nb, dtype)
        self.levels = []
        for na in g["na"]:
            nodd, nk = na // 2, (na + 1) // 2
            Dinv = inverse(D[1::2][:nodd])
            HL, HU = Dinv @ L[1::2][:nodd], Dinv @ U[1::2][:nodd]
            GL, GU = np.zeros((nk, m, m), dtype=dtype), np.zeros((nk, m, m), dtype=dtype)
            GL[1:] = L[2::2][:nk - 1] @ Dinv[:nk - 1]
            GU[:nodd] = U[0::2][:nodd] @ Dinv
            Dn = D[0::2].copy()
            Ln, Un = np.zeros_like(Dn), np.zeros_like(Dn)
            Dn[1:] -= GL[1:] @ U[1::2][:nk - 1]
            Dn[:nodd] -= GU[:nodd] @ L[1::2][:nodd]
            Ln[1:] = -(GL[1:] @ L[1::2][:nk - 1])
            Un[:nodd] = -(GU[:nodd] @ U[1::2][:nodd])
            self.levels.append({"na": na, "Dinv": Dinv, "HL": HL, "HU": HU, "GL": GL, "GU": GU})
            D, L, U = Dn, Ln, Un
        na = g["tail_na"]
        R = np.zeros((na * m, na * m), dtype=dtype)
        for p in range(na):
            R[p * m:(p + 1) * m, p * m:(p + 1) * m] = D[p]
            if p >= 1:
                R[p * m:(p + 1) * m, (p - 1) * m:p * m] = L[p]
            if p + 1 < na:
                R[p * m:(p + 1) * m, (p + 1) * m:(p + 2) * m] = U[p]
        self.tail_na = na
        self.last_inv = inverse(R)

    def factors(self):
        """(level, name, array) for every stored factor, in the order of the device's levels"""
        for s, lv in enumerate(self.levels):
            for name in ("Dinv", "HL", "HU", "GL", "GU"):
                yield s, name, lv[name]
        yield len(self.levels), "last_inv", self.last_inv

    def solve(self, b):
        """x = A^-1 b, step for step as bcr_solve: forward updates, tail product, backward recovery"""
        m, dtype = self.m, self.last_inv.dtype
        f = np.zeros(self.n_pad, dtype=dtype)
        f[:self.n] = np.asarray(b).ravel()
        fs = [f.reshape(-1, m)]
        for lv in self.levels:
            f, na = fs[-1], lv["na"]
            nodd = na // 2
            fk = f[0::2].copy()
            fk[1:] -= np.einsum("jrc,jc->jr", lv["GL"][1:], f[1::2][:len(fk) - 1])
            fk[:nodd] -= np.einsum("jrc,jc->jr", lv["GU"][:nodd], f[1::2][:nodd])
            fs.append(fk)
        x = (self.last_inv @ fs[-1].ravel()).reshape(-1, m)
        for lv, f in zip(reversed(self.levels), reversed(fs[:-1])):
            na = lv["na"]
            nodd = na // 2
            xl = np.zeros((na, m), dtype=dtype)
            xl[0::2] = x
            xo = np.einsum("jrc,jc->jr", lv["Dinv"], f[1::2][:nodd])
            xo -= np.einsum("jrc,jc->jr", lv["HL"], x[:nodd])
            nu = (na - 1) // 2                   # odd blocks that have a right neighbour: 2j + 2 < na
            xo[:nu] -= np.einsum("jrc,jc->jr", lv["HU"][:nu], x[1:nu + 1])
            xl[1::2] = xo
            x = xl
        return x.ravel()[:self.n]


def coarse_257(transfer, coefficient=None):
    """the 257^2 coarsest operator of the 1025^2 hierarchy (three levels), as SciPy's Galerkin products form it"""
    from learnmultigrid_b200 import formats as F, problems as P
    Ah = sp.csc_matrix(P.structured_laplacian_2d(1024, coefficient))
    for Q in P.structured_hierarchy_2d(1024, 3, transfer=transfer):
        Ah = sp.csr_matrix(Q.T @ Ah @ Q)
    return F.canonical_csr(Ah)


# (transfer, ordering): (m, nb, reduction levels, tail blocks, dense tail rows, padding rows).  build_coarse_solver
# keeps the natural numbering of the linear operator; the quasi-L2 one has half bandwidth 774 > 2 sqrt(n), so it is
# reordered by reverse Cuthill-McKee, which narrows the band to 770.
PRODUCTION_GEOMETRY = {
    ("linear", "natural"): (258, 257, [257, 129, 65, 33, 17, 9], 5, 1290, 257),
    ("quasi", "natural"): (774, 86, [86, 43, 22, 11], 6, 4644, 515),
    ("quasi", "rcm"): (770, 86, [86, 43, 22, 11], 6, 4620, 171),
}


def geometry_row(g):
    return g["m"], g["nb"], g["na"], g["tail_na"], g["tail_na"] * g["m"], g["padding"]


def level_gaps(A, half_bw, **kw):
    """{"level name": max|f64 - ext| / max|ext|} for every factor of the float64 reduction against the same reduction
    in np.longdouble: the rounding error of the float64 oracle itself"""
    lo, hi = BcrOracle(A, half_bw, **kw), BcrOracle(A, half_bw, dtype=np.longdouble, **kw)
    return {"%d %s" % (s, name): float(np.abs(a - b).max() / np.abs(b).max())
            for (s, name, a), (_, _, b) in zip(lo.factors(), hi.factors())}
