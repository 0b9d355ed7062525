"""Coarsest-level direct solvers (replace the per-cycle SuperLU spsolve of Multigrid.py:106).

  * dense : explicit inverse by cooperative Gauss-Jordan (csrc/dense_kernels.cu), solve = one GEMV;
  * bcr   : block cyclic reduction for banded operators (csrc/bcr.cu); all dense factors formed once here with
            the batched inverse / GEMM entry points, solve = 2*levels+3 launches streaming the factors once.
"""
import ctypes
import os

import numpy as np

from . import _lib


def half_bandwidth(indptr, indices):
    n = len(indptr) - 1
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(indptr))
    return int(np.abs(indices.astype(np.int64) - rows).max()) if len(indices) else 0


class DenseCoarse:
    kind = _lib.MG_COARSE_DENSE

    def __init__(self, torch, dev, n, ip, ix, va):
        lib = _lib.load()
        st = _lib.stream_handle(torch)
        dense = torch.empty(n * n, dtype=torch.float64, device=dev)
        _lib.check(lib.mg_csr_to_dense(n, ip.data_ptr(), ix.data_ptr(), va.data_ptr(), dense.data_ptr(), st),
                   "mg_csr_to_dense")
        self.inv = torch.empty(n * n, dtype=torch.float64, device=dev)
        work = torch.empty(int(lib.mg_dense_inverse_workspace(n)), dtype=torch.uint8, device=dev)
        _lib.check(lib.mg_dense_inverse(n, dense.data_ptr(), self.inv.data_ptr(), work.data_ptr(), st),
                   "mg_dense_inverse")
        self.n = n
        self.bytes = n * n * 8
        self.launches = 1


class BcrCoarse:
    kind = _lib.MG_COARSE_BCR

    # The reduction stops at this many block rows and what is left is inverted densely (one matrix-vector product in
    # the solve instead of a chain of latency-bound levels).  The dense inverse is a Gauss-Jordan sweep over a
    # (tail m) x (2 tail m) array per pivot: with 16 blocks of the 257^2 coarsest grid that array is 272 MB -- every one
    # of the 4128 pivots streams it through DRAM, 0.3 s of the 0.43 s factorisation -- with 8 blocks it is 68 MB and
    # stays in L2.  One more reduction level costs the solve two launches and saves it three quarters of the tail
    # matrix (136 -> 34 MB).  MGB_BCR_TAIL_BLOCKS overrides.
    TAIL_BLOCKS = 8

    def __init__(self, torch, dev, n, ip, ix, va, half_bw, min_block=64, tail_blocks=None, perm=None):
        """perm (optional, host int32 array): (ip, ix, va) is P A P^T for the caller's operator A, row i of it being row
        perm[i] of A; right-hand sides are gathered and solutions scattered accordingly inside the solve."""
        if tail_blocks is None:
            tail_blocks = int(os.environ.get("MGB_BCR_TAIL_BLOCKS", self.TAIL_BLOCKS))
        import time
        lib = _lib.load()
        st = _lib.stream_handle(torch)
        f64 = torch.float64
        self.timing = {}           # seconds per phase of the factorisation (device synchronised at each mark: setup only)
        t_mark = [time.perf_counter()]

        def mark(name):
            torch.cuda.synchronize()
            now = time.perf_counter()
            self.timing[name] = self.timing.get(name, 0.0) + now - t_mark[0]
            t_mark[0] = now
        m = max(int(half_bw), min_block, 1)
        nb = (n + m - 1) // m
        n_pad = nb * m
        mm = m * m
        self.n, self.m, self.nb = n, m, nb

        def zeros(k):
            return torch.zeros(max(k, 1) * mm, dtype=f64, device=dev)

        D, L, U = zeros(nb), zeros(nb), zeros(nb)
        bad = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.check(lib.mg_bcr_blocks_from_csr(n, n_pad, m, ip.data_ptr(), ix.data_ptr(), va.data_ptr(), D.data_ptr(),
                                              L.data_ptr(), U.data_ptr(), bad.data_ptr(), st), "mg_bcr_blocks_from_csr")
        if int(bad.item()):
            raise _lib.MgError("BCR: matrix entries outside the block-tridiagonal band (half bandwidth > block size)")
        mark("blocks from CSR")
        sing = torch.zeros(1, dtype=torch.int32, device=dev)
        work = torch.empty(max(nb // 2, 1) * m * 2 * m, dtype=f64, device=dev)
        e = 8                       # bytes per double, for pointer arithmetic on data_ptr()

        def inverse(src_ptr, stride, batch):
            out = zeros(batch)
            _lib.check(lib.mg_dense_inverse_batched(m, batch, src_ptr, stride, out.data_ptr(), mm, work.data_ptr(),
                                                    sing.data_ptr(), st), "mg_dense_inverse_batched")
            return out

        def gemm(batch, a_ptr, sa, b_ptr, sb, c_ptr, sc, alpha, beta):
            # grid.z is limited to 65535 batch members per launch
            done = 0
            while done < batch:
                nb_ = min(batch - done, 65535)
                _lib.check(lib.mg_dense_gemm_batched(m, nb_, a_ptr + done * sa * e, sa, b_ptr + done * sb * e, sb,
                                                     c_ptr + done * sc * e, sc, float(alpha), float(beta), st),
                           "mg_dense_gemm_batched")
                done += nb_

        self.levels = []
        self.keep = []
        na = nb
        while na > max(int(tail_blocks), 1):
            nodd, nk = na // 2, (na + 1) // 2
            Dinv = inverse(D.data_ptr() + mm * e, 2 * mm, nodd)
            mark("block inverses (batched Gauss-Jordan)")
            HL, HU = zeros(nodd), zeros(nodd)
            gemm(nodd, Dinv.data_ptr(), mm, L.data_ptr() + mm * e, 2 * mm, HL.data_ptr(), mm, 1.0, 0.0)
            gemm(nodd, Dinv.data_ptr(), mm, U.data_ptr() + mm * e, 2 * mm, HU.data_ptr(), mm, 1.0, 0.0)
            GL, GU = zeros(nk), zeros(nk)
            # GL[j] = L[2j] Dinv[j-1]  (j >= 1);  GU[j] = U[2j] Dinv[j]  (j < nodd)
            gemm(nk - 1, L.data_ptr() + 2 * mm * e, 2 * mm, Dinv.data_ptr(), mm, GL.data_ptr() + mm * e, mm, 1.0, 0.0)
            gemm(nodd, U.data_ptr(), 2 * mm, Dinv.data_ptr(), mm, GU.data_ptr(), mm, 1.0, 0.0)
            # reduced system on the even positions
            Dn = D.view(na, mm)[0::2].contiguous().view(-1)
            Ln, Un = zeros(nk), zeros(nk)
            gemm(nk - 1, GL.data_ptr() + mm * e, mm, U.data_ptr() + mm * e, 2 * mm, Dn.data_ptr() + mm * e, mm, -1.0, 1.0)
            gemm(nodd, GU.data_ptr(), mm, L.data_ptr() + mm * e, 2 * mm, Dn.data_ptr(), mm, -1.0, 1.0)
            gemm(nk - 1, GL.data_ptr() + mm * e, mm, L.data_ptr() + mm * e, 2 * mm, Ln.data_ptr() + mm * e, mm, -1.0, 0.0)
            gemm(nodd, GU.data_ptr(), mm, U.data_ptr() + mm * e, 2 * mm, Un.data_ptr(), mm, -1.0, 0.0)
            self.levels.append({"na": na, "GL": GL, "GU": GU, "Dinv": Dinv, "HL": HL, "HU": HU})
            D, L, U = Dn, Ln, Un
            na = nk
            mark("block products (batched GEMM)")
        self.tail_na = na
        if na == 1:
            self.last_inv = inverse(D.data_ptr(), mm, 1)
        else:
            # what is left is a small block-tridiagonal system: assemble it densely and invert it once, so that the
            # solve replaces a chain of latency-bound reduction levels by one matrix-vector product
            nt = na * m
            R = torch.zeros(nt, nt, dtype=f64, device=dev)
            Dv, Lv, Uv = D.view(-1, m, m), L.view(-1, m, m), U.view(-1, m, m)
            for p in range(na):
                R[p * m:(p + 1) * m, p * m:(p + 1) * m] = Dv[p]
                if p >= 1:
                    R[p * m:(p + 1) * m, (p - 1) * m:p * m] = Lv[p]
                if p + 1 < na:
                    R[p * m:(p + 1) * m, (p + 1) * m:(p + 2) * m] = Uv[p]
            self.last_inv = torch.empty(nt * nt, dtype=f64, device=dev)
            wk = torch.empty(int(lib.mg_dense_inverse_workspace(nt)), dtype=torch.uint8, device=dev)
            _lib.check(lib.mg_dense_inverse(nt, R.data_ptr(), self.last_inv.data_ptr(), wk.data_ptr(), st),
                       "mg_dense_inverse (BCR tail)")
            del R, wk
        mark("dense inverse of the tail")
        if int(sing.item()):
            raise _lib.MgError("BCR: singular diagonal block in the coarsest operator")
        self.f = torch.zeros(n_pad, dtype=f64, device=dev)
        self.x = torch.zeros(n_pad, dtype=f64, device=dev)
        h = _lib.mg_bcr()
        h.n, h.n_pad, h.m, h.nb = n, n_pad, m, nb
        h.nlevels = len(self.levels)
        if h.nlevels > 32:
            raise _lib.MgError("BCR: too many reduction levels")
        for s, lv in enumerate(self.levels):
            h.d_GL[s], h.d_GU[s] = lv["GL"].data_ptr(), lv["GU"].data_ptr()
            h.d_Dinv[s], h.d_HL[s], h.d_HU[s] = lv["Dinv"].data_ptr(), lv["HL"].data_ptr(), lv["HU"].data_ptr()
            h.na[s] = lv["na"]
        h.d_last_inv = self.last_inv.data_ptr()
        h.d_f, h.d_x = self.f.data_ptr(), self.x.data_ptr()
        h.tail_na = self.tail_na
        self.tail = torch.zeros(max(self.tail_na, 1) * m, dtype=f64, device=dev)
        h.d_tail = self.tail.data_ptr()
        self.perm = None
        if perm is not None:
            self.perm = torch.from_numpy(np.ascontiguousarray(perm, dtype=np.int32)).to(dev)
            h.d_perm = self.perm.data_ptr()
        self.handle = h
        self.bytes = (sum((2 * ((lv["na"] + 1) // 2) + 3 * (lv["na"] // 2)) * mm * 8 for lv in self.levels)
                      + self.tail_na * self.tail_na * mm * 8)
        self.launches = 2 * len(self.levels) + 3
        self.torch, self.dev = torch, dev
        self.dist = None

    def make_dist(self, rank, world, min_blocks=32):
        """mg_bcr_dist: split the reduction levels with at least `min_blocks` block rows, and the dense tail, over the
        ranks; each split step is followed by an all-gather (index lists into the padded work vectors)."""
        torch, dev = self.torch, self.dev
        m = self.m
        d = _lib.mg_bcr_dist()
        self._dist_keep = []

        def offsets(k):
            return [(k * r) // world for r in range(world + 1)]

        def gather_xfer(pos_of_rank):
            """all-gather site: rank q contributes the entries pos_of_rank[q] (int64 numpy positions)"""
            idx = [torch.from_numpy(np.ascontiguousarray(p, dtype=np.int32)).to(dev) for p in pos_of_rank]
            x = _lib.mg_xfer()
            for q in range(world):
                if q == rank:
                    continue
                k = x.npeers
                x.npeers += 1
                x.peer[k] = q
                x.d_send_idx[k] = idx[rank].data_ptr() if idx[rank].numel() else None
                x.send_cnt[k] = idx[rank].numel()
                x.d_recv_idx[k] = idx[q].data_ptr() if idx[q].numel() else None
                x.recv_cnt[k] = idx[q].numel()
            self._dist_keep.append((idx, x))
            return ctypes.pointer(x)

        ar = np.arange(m, dtype=np.int64)
        for s, lv in enumerate(self.levels):
            na = lv["na"]
            nk, nodd = (na + 1) // 2, na // 2
            if world > 1 and nk >= min_blocks:
                o = offsets(nk)
                d.fwd_j0[s], d.fwd_j1[s] = o[rank], o[rank + 1]
                d.fwd_xfer[s] = gather_xfer([(((2 * np.arange(o[q], o[q + 1], dtype=np.int64)) << s) * m)[:, None]
                                             + ar[None, :] for q in range(world)])
            if world > 1 and nodd >= min_blocks:
                o = offsets(nodd)
                d.bwd_j0[s], d.bwd_j1[s] = o[rank], o[rank + 1]
                d.bwd_xfer[s] = gather_xfer([(((2 * np.arange(o[q], o[q + 1], dtype=np.int64) + 1) << s) * m)[:, None]
                                             + ar[None, :] for q in range(world)])
        S = len(self.levels)
        nt = max(self.tail_na, 1) * m
        if world > 1 and self.tail_na > 1:
            o = offsets(nt)
            d.tail_i0, d.tail_i1 = o[rank], o[rank + 1]
            rows = [np.arange(o[q], o[q + 1], dtype=np.int64) for q in range(world)]
            d.tail_xfer = gather_xfer([((i // m) << S) * m + i % m for i in rows])
        self.dist = d
        return d

    def solve(self, torch, rhs, out):
        _lib.check(_lib.load().mg_bcr_solve(ctypes.byref(self.handle), rhs.data_ptr(), out.data_ptr(),
                                            _lib.stream_handle(torch)), "mg_bcr_solve")


BCR_MAX_FACTOR_BYTES = 24 << 30     # refuse factorisations beyond this (5 n m doubles)
BCR_MAX_BLOCK = 4096                # largest block the batched inverse takes (kGjMaxM in csrc/bcr.cu)


def bcr_fits(n, half_bw):
    """whether BcrCoarse takes n unknowns of half bandwidth half_bw (with its default min_block of 64): at least four
    block rows, blocks the batched inverse can invert, and factors within BCR_MAX_FACTOR_BYTES"""
    m = max(int(half_bw), 64)
    return m <= BCR_MAX_BLOCK and (n + m - 1) // m >= 4 and 5 * n * m * 8 <= BCR_MAX_FACTOR_BYTES


def rcm_ordering(indptr, indices, n):
    """reverse Cuthill-McKee ordering of the symmetrised pattern (host, setup time): perm[i] = old row of new row i"""
    import scipy.sparse as sp
    from scipy.sparse.csgraph import reverse_cuthill_mckee
    pat = sp.csr_matrix((np.ones(len(indices), dtype=np.int8), indices, indptr), shape=(n, n))
    return np.array(reverse_cuthill_mckee(sp.csr_matrix(pat + pat.T), symmetric_mode=True), dtype=np.int32, copy=True)


def permuted_half_bandwidth(indptr, indices, perm):
    n = len(indptr) - 1
    iperm = np.empty(n, dtype=np.int64)
    iperm[perm] = np.arange(n, dtype=np.int64)
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(indptr))
    return int(np.abs(iperm[indices] - iperm[rows]).max()) if len(indices) else 0


def bcr_ordering(n, indptr, indices):
    """(half bandwidth, perm) for block cyclic reduction of the n x n pattern (indptr, indices) on the host: perm is
    None to keep the numbering, else the reverse Cuthill-McKee permutation.  Raises MgError when neither numbering
    fits bcr_fits."""
    bw = half_bandwidth(indptr, indices)
    # a structured grid in natural order has half bandwidth ~ sqrt(n): keep it (no permutation in the solve)
    if bcr_fits(n, bw) and bw * bw <= 4 * n:
        return bw, None
    perm = rcm_ordering(indptr, indices, n)
    bw_p = permuted_half_bandwidth(indptr, indices, perm)
    if bw_p >= bw and bcr_fits(n, bw):
        return bw, None
    if not bcr_fits(n, bw_p):
        raise _lib.MgError("direct solve: %d unknowns with half bandwidth %d (%d after reverse Cuthill-McKee) are neither "
                           "small enough for a dense inverse nor banded enough for block cyclic reduction"
                           % (n, bw, bw_p))
    return bw_p, perm


def build_coarse_solver(torch, dev, n, ip, ix, va, dense_max, host_pattern=None, singular=False, label="coarsest level"):
    """Direct solver for an operator given as device CSR (ip, ix, va) -- the coarsest level of a hierarchy
    (Multigrid.py:106) or the system of DirectSolver (Solver.py:56-59):
      * n <= dense_max: explicit inverse;
      * banded as it is numbered (structured grids in natural order): block cyclic reduction;
      * anything else: reverse Cuthill-McKee first (unstructured meshes, shuffled numberings), then block cyclic
        reduction on P A P^T with the permutation applied inside the solve.
    singular=True: the operator may be symmetric with a one-dimensional null space (singular_coarse_solver); `label`
    names it in the errors."""
    if singular:
        return singular_coarse_solver(torch, dev, n, ip, ix, va, dense_max, host_pattern, label)
    if n <= dense_max:
        return DenseCoarse(torch, dev, n, ip, ix, va)
    if host_pattern is None:
        host_pattern = (ip.cpu().numpy(), ix.cpu().numpy())
    bw, perm = bcr_ordering(n, *host_pattern)
    return _bcr_solver(torch, dev, n, ip, ix, va, bw, perm)


def _bcr_solver(torch, dev, n, ip, ix, va, bw, perm):
    if perm is None:
        return BcrCoarse(torch, dev, n, ip, ix, va, bw)
    # P A P^T on the device: rows gathered by perm, columns relabelled by its inverse (entry order inside a row is
    # irrelevant to the block extraction)
    from .setup_device import DevCSR, DeviceSetup
    S = DeviceSetup(torch, dev)
    dperm = torch.from_numpy(perm).to(dev)
    iperm = S.empty(n, torch.int32)
    _lib.check(S.lib.mg_invert_permutation(n, dperm.data_ptr(), iperm.data_ptr(), S.st()), "mg_invert_permutation")
    Ap = S.permute(DevCSR((n, n), ip, ix, va), dperm, iperm)
    return BcrCoarse(torch, dev, n, Ap.indptr, Ap.indices, Ap.values, bw, perm=perm)


# A coarsest operator is taken as singular when the derived null vector nu_L leaves a residual in the pinned row of at most
# this much relative to ||A||_inf ||nu_L||_inf, and the pseudo-inverse is accepted when ||A A+ A w - A w|| <= VERIFY_TOL ||A w||.
SINGULAR_TOL = 1e-10
VERIFY_TOL = 1e-8


def apply_coarse(solver, rhs, out):
    """out = the solver's inverse (pseudo-inverse of a singular operator) applied to rhs (device vectors; rhs of a
    singular block cyclic reduction is overwritten with Z_k P rhs)"""
    torch = solver.torch
    lib = _lib.load()
    st = _lib.stream_handle(torch)
    if solver.kind == _lib.MG_COARSE_DENSE:
        _lib.check(lib.mg_dense_gemv(solver.n, solver.n, solver.inv.data_ptr(), rhs.data_ptr(), out.data_ptr(), st),
                   "mg_dense_gemv")
        return
    if solver.null is not None:
        project_out(solver, rhs, solver.null_pin)
    solver.solve(torch, rhs, out)
    if solver.null is not None:
        project_out(solver, out, -1)


def project_out(solver, v, pin):
    """v <- v - (nu^T v / nu^T nu) nu with the solver's null vector, then v[pin] = 0 if pin >= 0 (mg_project_out)"""
    torch = solver.torch
    lib = _lib.load()
    _lib.check(lib.mg_project_out(solver.n, solver.null.data_ptr(), solver.null_inv_nn, int(pin), v.data_ptr(),
                                  solver.null_work.data_ptr(), None, _lib.stream_handle(torch)), "mg_project_out")


def singular_coarse_solver(torch, dev, n, ip, ix, va, dense_max, host_pattern, label):
    """Direct solver of a symmetric operator A that may have a one-dimensional null space (DESIGN.md, singular systems).
    In the solver's own ordering (after reverse Cuthill-McKee where block cyclic reduction uses it) k is the last row and
    A_pin is A with row and column k replaced by e_k; the band, and with it the block structure, is unchanged.
      nu_L = e_k - A_pin^-1 Z_k a_k            (a_k: column k of A; Z_k zeroes entry k)
    is a null vector of A if A has one with a non-zero entry k.  A is taken as singular when
    |(A nu_L)_k| <= SINGULAR_TOL ||A||_inf ||nu_L||_inf, and then solved with
      A+ = P A_pin^-1 Z_k P,    P = I - nu_L nu_L^T / (nu_L^T nu_L)
    (the minimum-norm solution for right-hand sides in range(A) = nu_L-perp, the least-squares one for others): dense,
    as the explicit matrix mg_dense_gemv applies; by block cyclic reduction, as the projections around the solve
    (cycle.cu, mg_project_out).  A pseudo-inverse that does not reproduce A w for the hashed vector w to VERIFY_TOL
    (a null space of more than one vector) raises MgError.  Otherwise A is factored as it is.  The solver carries
    null_info = {"singular", "pin", "null_ratio", "verify_ratio"} and, when singular, null / null_inv_nn / null_pin."""
    import scipy.sparse as sp
    from . import formats as F
    hip, hix = (ip.cpu().numpy(), ix.cpu().numpy()) if host_pattern is None else host_pattern
    A = sp.csr_matrix((va.cpu().numpy(), np.asarray(hix), np.asarray(hip)), shape=(n, n))
    norm_A = float(abs(A).sum(axis=1).max()) if A.nnz else 0.0
    if n <= dense_max:
        bw, perm = 0, None
    else:
        bw, perm = bcr_ordering(n, hip, hix)
    k = n - 1 if perm is None else int(perm[n - 1])          # the pinned row in the level's ordering
    keep = np.ones(n)
    keep[k] = 0.0
    Z = sp.diags(keep)
    A_pin = sp.csr_matrix(Z @ A @ Z + sp.csr_matrix(([1.0], ([k], [k])), shape=(n, n)))
    A_pin.sort_indices()
    dip, dix, dva = (torch.from_numpy(np.ascontiguousarray(a, dtype=t)).to(dev) for a, t in
                     ((A_pin.indptr, np.int32), (A_pin.indices, np.int32), (A_pin.data, np.float64)))
    solver = DenseCoarse(torch, dev, n, dip, dix, dva) if n <= dense_max else _bcr_solver(
        torch, dev, n, dip, dix, dva, bw, perm)
    solver.torch = torch
    solver.null = None
    a_k = np.asarray(A[:, [k]].todense()).ravel() * keep
    y = torch.empty(n, dtype=torch.float64, device=dev)
    apply_coarse(solver, torch.from_numpy(-a_k).to(dev), y)
    nu = y.cpu().numpy()
    nu[k] = 1.0
    null_ratio = abs(float((A @ nu)[k])) / max(norm_A * float(np.abs(nu).max()), np.finfo(float).tiny)
    info = {"singular": bool(null_ratio <= SINGULAR_TOL), "pin": k, "null_ratio": null_ratio, "verify_ratio": None}
    if not info["singular"]:
        # taken as nonsingular: factored as it is, and the factor checked the same way (a rank-deficient operator whose
        # null vectors all vanish at k would pass the rule; its factor does not reproduce A w)
        del solver
        solver = build_coarse_solver(torch, dev, n, ip, ix, va, dense_max, (hip, hix))
        solver.torch = torch
        solver.null = None
        info["verify_ratio"] = _verify(solver, A, label, "the factor taken as nonsingular")
        solver.null_info = info
        return solver
    nn = float(nu @ nu)
    d_nu = torch.from_numpy(nu).to(dev)
    if solver.kind == _lib.MG_COARSE_DENSE:
        # A+ = P M P with M = A_pin^-1 Z_k (column k of the inverse dropped); rank-one updates on the device
        M = solver.inv.view(n, n)
        M[:, k] = 0.0
        Mnu = M @ d_nu
        nuM = d_nu @ M
        c = float(d_nu @ Mnu)
        M -= torch.outer(d_nu, nuM) / nn
        M -= torch.outer(Mnu, d_nu) / nn
        M += torch.outer(d_nu, d_nu) * (c / (nn * nn))
    solver.null = d_nu
    solver.null_inv_nn = 1.0 / nn
    solver.null_pin = k
    solver.null_work = torch.zeros(int(_lib.load().mg_project_workspace_size(n)), dtype=torch.float64, device=dev)
    info["verify_ratio"] = _verify(solver, A, label, "the pseudo-inverse pinned at row %d" % k)
    solver.null_info = info
    return solver


def _verify(solver, A, label, what):
    """||A X A w - A w|| / ||A w|| for the solver's X and the hashed vector w; MgError above VERIFY_TOL"""
    from . import formats as F
    torch = solver.torch
    n = A.shape[0]
    w = F.chebyshev_start_vector(np.arange(n, dtype=np.int64))
    Aw = A @ w
    x = torch.empty(n, dtype=torch.float64, device=solver.dev if hasattr(solver, "dev") else solver.inv.device)
    apply_coarse(solver, torch.from_numpy(Aw).to(x.device), x)
    ratio = float(np.linalg.norm(A @ x.cpu().numpy() - Aw)) / max(float(np.linalg.norm(Aw)), np.finfo(float).tiny)
    if not ratio <= VERIFY_TOL:
        raise _lib.MgError("%s: %s reproduces A w only to %.3e relative (limit %.0e): the null space has more than "
                           "one vector" % (label, what, ratio, VERIFY_TOL))
    return ratio
