"""Coarsest-level direct solvers against float64 / extended-precision references at the sizes they run at.

DenseCoarse (n <= 4096) is the cooperative Gauss-Jordan inverse (mg_dense_inverse) applied by gemv_rows; BcrCoarse is
block cyclic reduction whose factors come from the batched Gauss-Jordan and GEMM kernels and whose tail is inverted
by mg_dense_inverse.  The sizes are chosen on the switches of these kernels, derived from the device:
  * gauss_jordan_kernel runs on at most (threads per SM / 256) * SMs CTAs; above that each CTA owns several rows;
  * gemv_rows shares a row among T = 256 threads, T = 128 from sm_count * 2048 / 128 rows, T = 32 from / 32;
  * batched_gauss_jordan_kernel has 1024 threads, which loop over rows for blocks of more than 1024;
  * gemm_batched_kernel tiles 64 x 64 x 16, with partial tiles when m % 16 != 0 or m % 64 != 0;
and the 257^2 coarsest operators of the 1025^2 hierarchy run the reduction at its production geometry (odd and even
block counts, a last block that is nearly all identity padding, a 1290- or 4644-row dense tail)."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

import bcr_oracle as O
from bcr_oracle import PRODUCTION_GEOMETRY, coarse_257, geometry_row

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
MG_ERR_SINGULAR = -5                      # include/mgb200.h
E = 8                                     # bytes per double, for pointer offsets


@pytest.fixture(scope="module")
def env():
    import torch
    from learnmultigrid_b200 import _lib
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    props = torch.cuda.get_device_properties(0)
    sm = props.multi_processor_count
    want = sm * 2048                      # gemv_rows: threads that fill the device
    return {"torch": torch, "dev": torch.device("cuda", 0), "lib": _lib.load(), "_lib": _lib,
            "st": _lib.stream_handle(torch),
            "gj_grid_max": (props.max_threads_per_multi_processor // 256) * sm,
            "t128": -(-want // 128), "t32": -(-want // 32)}


def dev(env, a):
    return env["torch"].from_numpy(np.ascontiguousarray(a)).to(env["dev"])


def host(t):
    return t.cpu().numpy()


def kappa_inf(A, Ainv):
    return np.abs(A).sum(axis=1).max() * np.abs(Ainv).sum(axis=1).max()


# ---- mg_dense_inverse: cooperative Gauss-Jordan ---------------------------------------------------------------------

def dense_size(env, name):
    return {"gj+1": env["gj_grid_max"] + 1, "t128-1": env["t128"] - 1, "t128": env["t128"]}.get(name, name)


def spd_with_condition(n, kappa, seed):
    """(A, A^-1) for A = Q diag Q^T, eigenvalues from 1 down to 1 / kappa"""
    rng = np.random.default_rng(seed)
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    lam = np.geomspace(1.0, 1.0 / kappa, n)
    return (Q * lam) @ Q.T, (Q / lam) @ Q.T


def dense_inverse(env, A):
    lib, torch, _lib = env["lib"], env["torch"], env["_lib"]
    n = A.shape[0]
    dA = dev(env, A)
    inv = torch.full((n * n,), np.nan, dtype=torch.float64, device=env["dev"])
    work = torch.empty(int(lib.mg_dense_inverse_workspace(n)), dtype=torch.uint8, device=env["dev"])
    rc = lib.mg_dense_inverse(n, dA.data_ptr(), inv.data_ptr(), work.data_ptr(), env["st"])
    assert np.array_equal(host(dA), A)                           # the input is not overwritten
    return rc, host(inv).reshape(n, n)


@pytest.mark.parametrize("size", ["gj+1", 1290, "t128-1", "t128", 4096, 4644])
def test_dense_inverse_at_coarse_sizes(env, size):
    n = dense_size(env, size)
    assert n > env["gj_grid_max"]                               # every CTA owns several rows
    A, Ainv = spd_with_condition(n, 1e4, seed=n)
    perm = np.random.default_rng(n + 1).permutation(n)
    k = kappa_inf(A, Ainv)                                       # row permutations keep both infinity norms
    # rows permuted: every pivot is off the diagonal; (P A)^-1 = A^-1 P^T
    for M, Xref in ((A, Ainv), (A[perm], Ainv[:, perm])):
        rc, X = dense_inverse(env, M)
        assert rc == 0
        assert np.abs(X @ M - np.eye(n)).max() <= n * EPS * k
        assert np.abs(X - Xref).max() <= n * EPS * k * np.abs(Xref).max()
        rc, X2 = dense_inverse(env, M)
        assert rc == 0 and np.array_equal(X, X2)                # deterministic pivots and sums


def test_dense_inverse_reports_rank_deficiency_at_size(env):
    """a zero column stays exactly zero under elimination: the pivot search of every CTA finds no pivot at that
    column and all CTAs leave together"""
    n = env["t128"]
    A, _ = spd_with_condition(n, 1e2, seed=5)
    A[:, n // 3] = 0.0
    rc, _ = dense_inverse(env, A)
    assert rc == MG_ERR_SINGULAR
    assert "zero pivot" in env["lib"].mg_last_error().decode()
    rc, X = dense_inverse(env, spd_with_condition(n, 1e2, seed=6)[0])  # the device is usable afterwards
    assert rc == 0 and np.isfinite(X).all()


# ---- mg_dense_gemv: every threads-per-row route ---------------------------------------------------------------------

def gemv_threads(env, rows):
    return 32 if rows >= env["t32"] else 128 if rows >= env["t128"] else 256


@pytest.mark.parametrize("rows", [1, "t128-1", "t128", "t32-1", "t32", 12000])
def test_dense_gemv_routes(env, rows):
    rows = {"t128-1": env["t128"] - 1, "t128": env["t128"], "t32-1": env["t32"] - 1, "t32": env["t32"]}.get(rows, rows)
    T = gemv_threads(env, rows)
    lib, torch = env["lib"], env["torch"]
    rng = np.random.default_rng(rows)
    for cols in (1, 3, 4 * T - 1, 4 * T, 4 * T + 1, 2064):       # four-accumulator loop and its remainder
        M = rng.standard_normal((rows, cols))
        x = rng.standard_normal(cols)
        d_m, d_x = dev(env, M), dev(env, x)                     # held: a freed block would be handed out again
        y = torch.full((rows,), np.nan, dtype=torch.float64, device=env["dev"])
        env["_lib"].check(lib.mg_dense_gemv(rows, cols, d_m.data_ptr(), d_x.data_ptr(), y.data_ptr(), env["st"]),
                          "mg_dense_gemv")
        exact = M.astype(np.longdouble) @ x.astype(np.longdouble)
        gamma = cols * EPS / (1 - cols * EPS)
        err = np.abs(host(y).astype(np.longdouble) - exact)
        assert np.all(err <= gamma * (np.abs(M) @ np.abs(x))), (rows, cols, T, float(err.max()))


# ---- mg_dense_inverse_batched ---------------------------------------------------------------------------------------

def batched_inverse(env, mats, stride_blocks=2, offset_blocks=1):
    """inverses of mats[b] stored as BcrCoarse passes them: block b at offset_blocks + b * stride_blocks, the blocks in
    between NaN"""
    lib, torch = env["lib"], env["torch"]
    batch, m, _ = mats.shape
    mm = m * m
    src = np.full((offset_blocks + stride_blocks * batch, m, m), np.nan)
    src[offset_blocks::stride_blocks][:batch] = mats
    d_src = dev(env, src)
    out = torch.full((batch * mm,), np.nan, dtype=torch.float64, device=env["dev"])
    work = torch.empty(batch * m * 2 * m, dtype=torch.float64, device=env["dev"])
    sing = torch.zeros(1, dtype=torch.int32, device=env["dev"])
    rc = lib.mg_dense_inverse_batched(m, batch, d_src.data_ptr() + offset_blocks * mm * E, stride_blocks * mm,
                                      out.data_ptr(), mm, work.data_ptr(), sing.data_ptr(), env["st"])
    return rc, int(sing.item()), host(out).reshape(batch, m, m)


def pivoting_matrices(m, batch, seed):
    """well conditioned, rows shuffled so that the pivots are spread over the whole block"""
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((batch, m, m)) + 0.3 * m * np.eye(m)
    return np.stack([a[rng.permutation(m)] for a in A])


def block_diagonal_matrices(m, batch, seed, k=8):
    """dense k x k diagonal blocks, rows shuffled: the elimination of a column touches k rows only, so a 4096 block
    costs little while the pivot search still scans every row"""
    rng = np.random.default_rng(seed)
    out = np.zeros((batch, m, m))
    for b in range(batch):
        for i in range(0, m, k):
            j = min(i + k, m)
            out[b, i:j, i:j] = rng.standard_normal((j - i, j - i)) + 2 * k * np.eye(j - i)
        out[b] = out[b][rng.permutation(m)]
    return out


@pytest.mark.parametrize("m,batch", [(31, 4), (32, 3), (33, 2), (258, 4), (774, 3), (1023, 2), (1024, 1), (1025, 3),
                                     (1500, 2), (4096, 1)])
def test_batched_inverse(env, m, batch):
    mats = block_diagonal_matrices(m, batch, m) if m == 4096 else pivoting_matrices(m, batch, m)
    rc, sing, X = batched_inverse(env, mats)
    assert rc == 0 and sing == 0
    for b in range(batch):
        Xref = np.linalg.inv(mats[b])
        k = kappa_inf(mats[b], Xref)
        assert np.abs(X[b] @ mats[b] - np.eye(m)).max() <= m * EPS * k
        assert np.abs(X[b] - Xref).max() <= m * EPS * k * np.abs(Xref).max()


@pytest.mark.parametrize("m", [33, 1025])
def test_batched_inverse_flags_a_singular_member(env, m):
    mats = pivoting_matrices(m, 3, seed=7)
    mats[1, :, m // 2] = 0.0
    rc, sing, X = batched_inverse(env, mats)
    assert rc == 0 and sing == 1
    for b in (0, 2):                                             # the other members are still inverted
        assert np.abs(X[b] @ mats[b] - np.eye(m)).max() <= m * EPS * kappa_inf(mats[b], np.linalg.inv(mats[b]))


def test_batched_inverse_refuses_blocks_above_its_limit(env):
    from learnmultigrid_b200 import coarse
    torch, lib = env["torch"], env["lib"]
    m = coarse.BCR_MAX_BLOCK + 1
    buf = torch.zeros(1, dtype=torch.float64, device=env["dev"])
    sing = torch.zeros(1, dtype=torch.int32, device=env["dev"])
    rc = lib.mg_dense_inverse_batched(m, 1, buf.data_ptr(), m * m, buf.data_ptr(), m * m, buf.data_ptr(),
                                      sing.data_ptr(), env["st"])
    assert rc != 0
    assert "block size out of range" in lib.mg_last_error().decode()


# ---- mg_dense_gemm_batched ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("m", [1, 15, 16, 17, 63, 64, 65, 258, 774])
def test_batched_gemm(env, m):
    """C[b] = alpha A[b] B[b] + beta C[b] with the operand layouts of BcrCoarse: A every other block from block 2
    (L[2j]), B contiguous (Dinv), C from block 1 (GL[1:]); everything the kernel must not touch is NaN"""
    torch, lib = env["torch"], env["lib"]
    batch = 2 if m == 774 else 3
    mm = m * m
    rng = np.random.default_rng(m)
    A, B, C = (rng.standard_normal((batch, m, m)) for _ in range(3))
    a_store = np.full((2 + 2 * batch, m, m), np.nan)
    a_store[2::2][:batch] = A
    d_a, d_b = dev(env, a_store), dev(env, B)
    AB = np.matmul(A.astype(np.longdouble), B.astype(np.longdouble))
    absAB = np.abs(A) @ np.abs(B)
    gamma = (m + 2) * EPS / (1 - (m + 2) * EPS)
    for alpha, beta in ((1.0, 0.0), (-1.0, 1.0), (-0.5, 2.0)):
        c_store = np.full((1 + batch, m, m), np.nan)
        if beta != 0.0:
            c_store[1:] = C                                      # with beta = 0 the NaN must not leak into C
        d_c = dev(env, c_store)
        env["_lib"].check(lib.mg_dense_gemm_batched(m, batch, d_a.data_ptr() + 2 * mm * E, 2 * mm, d_b.data_ptr(), mm,
                                                    d_c.data_ptr() + mm * E, mm, alpha, beta, env["st"]),
                          "mg_dense_gemm_batched")
        got = host(d_c).reshape(1 + batch, m, m)
        assert np.isnan(got[0]).all()                            # the block before the first member is untouched
        exact = alpha * AB + (beta * C.astype(np.longdouble) if beta != 0.0 else 0.0)
        bound = gamma * (abs(alpha) * absAB + abs(beta) * np.abs(C))
        err = np.abs(got[1:].astype(np.longdouble) - exact)
        assert np.isfinite(got[1:]).all() and np.all(err <= bound), (alpha, beta, float(err.max()))


# ---- block cyclic reduction at the production geometry --------------------------------------------------------------

OPERATORS = [("linear", False), ("linear", True), ("quasi", False), ("quasi", True)]

# Rounding error of the float64 oracle on the constant-coefficient linear 257^2 operator: max|f64 - ext| / max|ext| per
# level and factor against the same reduction in 80-bit np.longdouble, from
# bcr_oracle.level_gaps(coarse_257("linear"), 258) (about ten minutes on one CPU core).  The device rounds in another
# order (Gauss-Jordan instead of LU, 16-wide tiled sums) but to the same order of magnitude, so each of its factors may
# differ from the oracle by a small multiple of this gap; a wrong term or a skipped tile differs by O(1).
CALIBRATED_GAP = {
    "0 Dinv": 2.512e-16, "0 HL": 2.930e-16, "0 HU": 2.930e-16, "0 GL": 2.930e-16, "0 GU": 2.930e-16,
    "1 Dinv": 7.126e-16, "1 HL": 1.085e-15, "1 HU": 1.051e-15, "1 GL": 1.031e-15, "1 GU": 1.063e-15,
    "2 Dinv": 1.546e-15, "2 HL": 2.191e-15, "2 HU": 1.629e-15, "2 GL": 1.733e-15, "2 GU": 1.830e-15,
    "3 Dinv": 2.617e-15, "3 HL": 3.847e-15, "3 HU": 3.800e-15, "3 GL": 3.878e-15, "3 GU": 3.967e-15,
    "4 Dinv": 5.721e-15, "4 HL": 1.076e-14, "4 HU": 1.080e-14, "4 GL": 1.085e-14, "4 GU": 1.067e-14,
    "5 Dinv": 1.315e-14, "5 HL": 3.701e-14, "5 HU": 3.134e-14, "5 GL": 3.082e-14, "5 GU": 3.740e-14,
    "6 last_inv": 6.087e-14,
}
GAP_FACTOR = 64


@pytest.fixture(scope="module")
def operators():
    from learnmultigrid_b200 import problems as P
    out = {}
    for transfer, variable in OPERATORS:
        A = coarse_257(transfer, P.variable_coefficient if variable else None)
        lu = spla.splu(sp.csc_matrix(A), permc_spec="MMD_AT_PLUS_A", diag_pivot_thresh=0.0,
                       options={"SymmetricMode": True})             # SPD: symmetric ordering, diagonal pivots
        lam_max = spla.eigsh(A, k=1, which="LA", tol=1e-3, return_eigenvectors=False)[0]
        inv_op = spla.LinearOperator(A.shape, matvec=lu.solve, dtype=np.float64)
        lam_min = 1.0 / spla.eigsh(inv_op, k=1, which="LA", tol=1e-3, return_eigenvectors=False)[0]
        out[transfer, variable] = {"A": A, "lu": lu, "kappa": lam_max / lam_min}
    return out


def upload_csr(env, A):
    return tuple(dev(env, a) for a in (A.indptr, A.indices, A.data))


def production_rhs(n):
    rng = np.random.default_rng(11)
    g = (np.arange(n) % 257 + 0.5) / 257, (np.arange(n) // 257 + 0.5) / 257
    smooth = np.sin(np.pi * g[0]) * np.sin(2 * np.pi * g[1])
    last = np.zeros(n)
    last[n - 1] = 1.0                                            # the padded last block's real row(s)
    return {"random": rng.standard_normal(n), "smooth": smooth, "last row": last}


def bcr_solve(env, bcr, b):
    torch = env["torch"]
    x = torch.full((len(b),), np.nan, dtype=torch.float64, device=env["dev"])
    bcr.solve(torch, dev(env, b), x)
    return host(x)


@pytest.mark.parametrize("transfer,variable", OPERATORS)
def test_bcr_production_geometry_and_solves(env, operators, transfer, variable):
    from learnmultigrid_b200.coarse import BcrCoarse, build_coarse_solver, half_bandwidth
    op = operators[transfer, variable]
    A = op["A"]
    n = A.shape[0]
    bw = half_bandwidth(A.indptr, A.indices)
    ip, ix, va = upload_csr(env, A)
    natural = BcrCoarse(env["torch"], env["dev"], n, ip, ix, va, bw)
    g = {"m": natural.m, "nb": natural.nb, "na": [lv["na"] for lv in natural.levels], "tail_na": natural.tail_na,
         "padding": natural.nb * natural.m - n}
    assert geometry_row(g) == PRODUCTION_GEOMETRY[transfer, "natural"]
    chosen = build_coarse_solver(env["torch"], env["dev"], n, ip, ix, va, 4096, (A.indptr, A.indices))
    assert (chosen.perm is None) == (transfer == "linear")
    if chosen.perm is not None:
        assert chosen.m * chosen.tail_na == PRODUCTION_GEOMETRY[transfer, "rcm"][4]
    nt = natural.tail_na * natural.m
    assert gemv_threads(env, nt) == (128 if transfer == "quasi" else 256)
    tol = 1e-12 * op["kappa"]
    for solver in (natural, chosen) if chosen.perm is not None else (natural,):
        for name, b in production_rhs(n).items():
            want = op["lu"].solve(b)
            x = bcr_solve(env, solver, b)
            err = np.abs(x - want).max() / np.abs(want).max()
            assert err <= tol, (name, solver.perm is not None, err, tol)


def test_bcr_factors_match_the_oracle_level_by_level(env, operators):
    from learnmultigrid_b200.coarse import BcrCoarse, half_bandwidth
    A = operators["linear", False]["A"]
    n = A.shape[0]
    bw = half_bandwidth(A.indptr, A.indices)
    bcr = BcrCoarse(env["torch"], env["dev"], n, *upload_csr(env, A), bw)
    oracle = O.BcrOracle(A, bw, tail_blocks=bcr.TAIL_BLOCKS)
    assert [lv["na"] for lv in bcr.levels] == oracle.geometry["na"] and bcr.tail_na == oracle.tail_na
    assert sorted(CALIBRATED_GAP) == sorted("%d %s" % (s, name) for s, name, _ in oracle.factors())
    for s, name, want in oracle.factors():
        got = host(bcr.last_inv if name == "last_inv" else bcr.levels[s][name]).reshape(want.shape)
        rel = np.abs(got - want).max() / np.abs(want).max()
        assert rel <= GAP_FACTOR * CALIBRATED_GAP["%d %s" % (s, name)], (s, name, rel)


# ---- block cyclic reduction: edges ----------------------------------------------------------------------------------

def check_against_oracle(env, A, half_bw, min_block, tail_blocks, perm_solver=None):
    from learnmultigrid_b200.coarse import BcrCoarse
    n = A.shape[0]
    bcr = BcrCoarse(env["torch"], env["dev"], n, *upload_csr(env, A), half_bw, min_block=min_block,
                    tail_blocks=tail_blocks)
    oracle = O.BcrOracle(A, half_bw, min_block=min_block, tail_blocks=tail_blocks)
    assert (bcr.m, bcr.nb, bcr.tail_na) == (oracle.m, oracle.nb, oracle.tail_na)
    for s, name, want in oracle.factors():
        got = host(bcr.last_inv if name == "last_inv" else bcr.levels[s][name]).reshape(want.shape)
        assert np.abs(got - want).max() <= 1e-11 * np.abs(want).max(), (s, name)
    rng = np.random.default_rng(n)
    lu = spla.splu(sp.csc_matrix(A))
    for b in (rng.standard_normal(n), np.eye(n)[n - 1]):
        want = lu.solve(b)
        np.testing.assert_allclose(bcr_solve(env, bcr, b), want, rtol=0, atol=1e-11 * np.abs(want).max())
    return bcr


def test_bcr_single_block_tail(env):
    A = O.banded_spd(700, 40, seed=1)                           # nb = 18: 18, 9, 5, 3, 2 -> one block
    bcr = check_against_oracle(env, A, 40, min_block=1, tail_blocks=1)
    assert bcr.tail_na == 1 and [lv["na"] for lv in bcr.levels] == [18, 9, 5, 3, 2]


def test_bcr_four_blocks_last_one_nearly_all_padding(env):
    m = 300
    A = O.banded_spd(3 * m + 1, m, seed=2)                      # even na at both levels: 4, 2
    bcr = check_against_oracle(env, A, m, min_block=1, tail_blocks=1)
    assert bcr.nb == 4 and [lv["na"] for lv in bcr.levels] == [4, 2]


@pytest.mark.parametrize("m,n,tail_blocks", [(1025, 5 * 1025 - 7, 1), (1500, 4 * 1500, 2)])
def test_bcr_blocks_above_1024_rows(env, m, n, tail_blocks):
    A = O.banded_spd(n, m, seed=m)
    check_against_oracle(env, A, m, min_block=1, tail_blocks=tail_blocks)


def test_bcr_reordered_path_matches_natural_order(env):
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.coarse import BcrCoarse, build_coarse_solver, half_bandwidth
    S = sp.csr_matrix(P.structured_laplacian_2d(80, P.variable_coefficient))
    n = S.shape[0]
    p = np.random.default_rng(0).permutation(n)
    Sp = sp.csr_matrix(S[p][:, p])
    Sp.sort_indices()
    shuffled = build_coarse_solver(env["torch"], env["dev"], n, *upload_csr(env, Sp), 0, (Sp.indptr, Sp.indices))
    assert shuffled.perm is not None
    natural = BcrCoarse(env["torch"], env["dev"], n, *upload_csr(env, S), half_bandwidth(S.indptr, S.indices))
    b = np.random.default_rng(1).standard_normal(n)
    x_nat = bcr_solve(env, natural, b)
    x_shuf = bcr_solve(env, shuffled, b[p])
    want = spla.spsolve(sp.csc_matrix(S), b)
    np.testing.assert_allclose(x_nat, want, rtol=0, atol=1e-11 * np.abs(want).max())
    np.testing.assert_allclose(x_shuf, x_nat[p], rtol=0, atol=1e-11 * np.abs(want).max())


def test_bcr_rejects_entries_outside_the_band(env):
    from learnmultigrid_b200 import _lib
    from learnmultigrid_b200.coarse import BcrCoarse
    A = O.banded_spd(640, 20, seed=3)
    with pytest.raises(_lib.MgError, match="outside the block-tridiagonal band"):
        BcrCoarse(env["torch"], env["dev"], 640, *upload_csr(env, A), 10, min_block=1)


def test_bcr_reports_a_singular_diagonal_block(env):
    """row 0 of block 1 keeps its couplings to block 0 but loses those inside its own block, so D[1] (inverted at the
    first level) has a zero row"""
    from learnmultigrid_b200 import _lib
    from learnmultigrid_b200.coarse import BcrCoarse
    m = 20
    A = O.banded_spd(4 * m, m, seed=4).tolil()
    for c in range(m, 2 * m):
        A[m, c] = 0.0
    A = sp.csr_matrix(A)
    A.eliminate_zeros()
    with pytest.raises(_lib.MgError, match="singular diagonal block"):
        BcrCoarse(env["torch"], env["dev"], 4 * m, *upload_csr(env, A), m, min_block=1, tail_blocks=1)


# ---- the dense coarsest level inside a V-cycle, on the T = 128 product ----------------------------------------------

def test_vcycle_with_dense_coarsest_level_on_the_t128_route(env):
    from learnmultigrid_b200 import _lib, problems as P
    from learnmultigrid_b200.engine import DeviceHierarchy
    from oracle.vcycle import OracleMultigrid
    N = 248
    A = P.structured_laplacian_2d(N)
    Qs = P.structured_hierarchy_2d(N, 3, transfer="linear")     # coarsest = 63^2 = 3969 unknowns
    nc = Qs[-1].shape[1]
    assert nc == 63 * 63 and gemv_threads(env, nc) == 128
    b = np.random.default_rng(0).standard_normal(A.shape[0])
    h = DeviceHierarchy(A, Qs, smoother="mcgs", setup="device")
    assert h.levels[-1].coarse_kind == _lib.MG_COARSE_DENSE
    o = OracleMultigrid(A, b.reshape(-1, 1), Qs, smoother="mcgs", colors=h.colors, hoist_setup=True)
    o.build_hierarchy(3)
    h.set_rhs(b)
    h.zero_x()
    p = h.make_params(nu_pre=1, nu_post=1)
    xo = np.zeros((A.shape[0], 1))
    for _ in range(2):
        h.vcycle(p)
        xo = o.v_cycle(o.matrix, xo, b.reshape(-1, 1), 1, 3)
        np.testing.assert_allclose(h.get_x(), xo, rtol=0, atol=1e-12 * np.linalg.norm(xo))


# ---- DirectSolver on a system no direct path takes -------------------------------------------------------------------

def test_direct_solver_refuses_a_wide_band_system_clearly(env):
    from learnmultigrid_b200 import _lib
    from learnmultigrid_b200.solvers.Solver import DirectSolver
    A = O.layered_graph_matrix()
    ds = DirectSolver(A, np.ones((A.shape[0], 1)))
    with pytest.raises(_lib.MgError) as err:
        ds.solve()
    assert "neither small enough for a dense inverse nor banded enough" in str(err.value)
    assert "block size out of range" not in str(err.value)
