"""NumPy restatement of the singular coarsest solve (learnmultigrid_b200/coarse.py, singular_coarse_solver) and of a
stationary multigrid solve of a singular symmetric system with it (DESIGN.md, singular systems).

Pinned factor: k = the last row, A_pin = A with row and column k replaced by e_k,
    nu_L = e_k - A_pin^-1 Z_k a_k,       A+ = P A_pin^-1 Z_k P,      P = I - nu nu^T / (nu^T nu).
A is singular when |(A nu_L)_k| <= 1e-10 ||A||_inf ||nu_L||_inf; the pseudo-inverse is accepted when it reproduces A w
for the hashed vector w to 1e-8."""
import numpy as np
import scipy.sparse as sp

from learnmultigrid_b200 import formats as F

SINGULAR_TOL = 1e-10
VERIFY_TOL = 1e-8


def projector(nu):
    nu = np.asarray(nu, dtype=np.float64).ravel()
    return np.eye(len(nu)) - np.outer(nu, nu) / (nu @ nu)


def pinned(A, k=None):
    """dict(singular, k, nu, null_ratio, verify_ratio, pinv) for a small symmetric A (dense float64 throughout);
    pinv is the plain inverse when A is found nonsingular"""
    A = np.asarray(A.todense() if sp.issparse(A) else A, dtype=np.float64)
    n = A.shape[0]
    k = n - 1 if k is None else int(k)
    A_pin = A.copy()
    A_pin[k, :] = 0.0
    A_pin[:, k] = 0.0
    A_pin[k, k] = 1.0
    inv_pin = np.linalg.inv(A_pin)
    a_k = A[:, k].copy()
    a_k[k] = 0.0
    nu = -inv_pin @ a_k
    nu[k] = 1.0
    norm_A = np.abs(A).sum(axis=1).max()
    null_ratio = abs((A @ nu)[k]) / (norm_A * np.abs(nu).max())
    out = {"k": k, "nu": nu, "null_ratio": null_ratio, "singular": bool(null_ratio <= SINGULAR_TOL)}
    if not out["singular"]:
        out["pinv"] = np.linalg.inv(A)
        out["verify_ratio"] = None
        return out
    Zk = np.eye(n)
    Zk[k, k] = 0.0
    P = projector(nu)
    pinv = P @ inv_pin @ Zk @ P
    w = F.chebyshev_start_vector(np.arange(n, dtype=np.int64))
    Aw = A @ w
    out["pinv"] = pinv
    out["verify_ratio"] = float(np.linalg.norm(A @ (pinv @ Aw) - Aw) / np.linalg.norm(Aw))
    return out


def svd_null_vector(A):
    """unit right singular vector of the smallest singular value"""
    A = np.asarray(A.todense() if sp.issparse(A) else A, dtype=np.float64)
    return np.linalg.svd(A)[2][-1]


def coarse_solve_hook():
    """coarse_solve= for tests/helpers.py::emulate_vcycle: the pinned pseudo-inverse of the coarsest operator"""
    cache = {}

    def solve(A_nat, b):
        key = id(A_nat)
        if key not in cache:
            cache[key] = pinned(A_nat)["pinv"]
        return cache[key] @ b
    return solve


def stationary_history(A, Qs, nu, b, smoother="mcgs", cycles=20, omega=2.0 / 3.0):
    """||P b - A x_j|| for x_0 = 0 and j = 1..cycles V(1,1) cycles (emulate_vcycle with the pinned coarse solve) in
    the natural ordering of level 0; returns (history, x) with x projected"""
    from helpers import emulate_vcycle
    levels = F.build_host_hierarchy(A, Qs, smoother)
    A0 = sp.csr_matrix(A)
    nu = np.asarray(nu, dtype=np.float64).ravel()
    P = lambda v: v - (nu @ v) / (nu @ nu) * nu
    bp = P(np.asarray(b, dtype=np.float64).ravel())
    perm = levels[0]["perm"]
    to_lev = (lambda v: v) if perm is None else (lambda v: v[perm])

    def to_nat(v):
        if perm is None:
            return v
        out = np.empty_like(v)
        out[perm] = v
        return out
    x = np.zeros(A0.shape[0])
    hook = coarse_solve_hook()
    hist = [np.linalg.norm(bp - A0 @ x)]
    for _ in range(cycles):
        x = to_nat(emulate_vcycle(levels, smoother, 1, 1, omega, to_lev(x), to_lev(bp), coarse_solve=hook))
        hist.append(np.linalg.norm(bp - A0 @ x))
    return np.array(hist), P(x)


def factor(hist):
    """geometric mean reduction per cycle over the history (after the first cycle)"""
    h = np.asarray(hist, dtype=np.float64).ravel()
    return float((h[-1] / h[1]) ** (1.0 / (len(h) - 2)))


def two_squares(N):
    """two disconnected pure-Neumann squares: a two-dimensional null space"""
    from learnmultigrid_b200 import problems as P
    A = sp.csr_matrix(P.structured_laplacian_2d(N, boundary="neumann"))
    return F.canonical_csr(sp.block_diag([A, A], format="csr"))


class _PinvSolve:
    """stands in for the oracle's coarse LU: the pinned pseudo-inverse"""

    def __init__(self, A):
        self.pinv = pinned(A)["pinv"]

    def solve(self, b):
        return self.pinv @ np.ravel(b)


def oracle_history(A, Qs, b, smoother, cycles, colors=None, omega=1.0, cheby_coefficients=None):
    """||P b - A x_j||, j = 0..cycles, of V(1,1) cycles of oracle/vcycle.py (smoother "gs" = index order, "mcgs" with
    `colors`, "jacobi", "chebyshev" with one coefficient table per smoothing level) with the pinned pseudo-inverse as
    the coarsest solve, nu = ones; returns (history, projected x)"""
    from oracle.vcycle import OracleMultigrid
    from chebyshev_oracle import ChebyshevOracle
    A = sp.csr_matrix(A)
    n = A.shape[0]
    bp = np.asarray(b, dtype=np.float64).ravel()
    bp = (bp - bp.sum() / n).reshape(-1, 1)
    levels = len(Qs) + 1
    if smoother == "chebyshev":
        o = ChebyshevOracle(A, bp, Qs, cheby_coefficients=cheby_coefficients, hoist_setup=True)
    else:
        o = OracleMultigrid(A, bp, Qs, smoother=smoother, omega=omega, colors=colors, hoist_setup=True)
    o.build_hierarchy(levels)
    o._lu = _PinvSolve(o._A_levels[-1])
    x = np.zeros((n, 1))
    hist = [np.linalg.norm(bp - A @ x)]
    for _ in range(cycles):
        x = o.v_cycle(o._A_levels[0], x, bp, 1, levels)
        hist.append(np.linalg.norm(bp - A @ x))
    x = x.ravel()
    return np.array(hist), x - x.sum() / n
