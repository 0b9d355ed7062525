"""Device-side hierarchy setup: Galerkin products by two-pass SpGEMM, transposes, colour-blocked permutation and
SELL-32 build, all through the setup entry points of libmgb200 (csrc/setup_kernels.cu).  PyTorch only provides
the device buffers.  The host path (formats.build_host_hierarchy) produces the same data with SciPy/NumPy and is
what the GPU tests compare this against.
"""
import ctypes
import os

import numpy as np
import scipy.sparse as sp

from . import _lib
from . import formats as F


class DevCSR:
    """CSR matrix in device memory (int32 indptr / indices, float64 values)."""

    def __init__(self, shape, indptr, indices, values):
        self.shape = (int(shape[0]), int(shape[1]))
        self.indptr, self.indices, self.values = indptr, indices, values
        self.nnz = int(indices.numel())

    def ptrs(self):
        return self.indptr.data_ptr(), self.indices.data_ptr(), self.values.data_ptr()


class ColorList(list):
    """Per-level colour arrays of a hierarchy.  Colours computed on the device stay there (the setup only needs them
    there: permutation, flags); an entry is downloaded the first time somebody asks for it on the host (tests, the
    oracle's colour argument, the partition plans) and is a NumPy int32 array from then on."""

    def _host(self, k):
        v = list.__getitem__(self, k)
        if v is not None and not isinstance(v, np.ndarray):
            v = v.cpu().numpy()
            list.__setitem__(self, k, v)
        return v

    def __getitem__(self, k):
        if isinstance(k, slice):
            return [self._host(i) for i in range(*k.indices(len(self)))]
        return self._host(k if k >= 0 else k + len(self))

    def __iter__(self):
        return (self._host(i) for i in range(len(self)))

    def device(self, k):
        """entry k as it is stored (device tensor or host array), without a download"""
        return list.__getitem__(self, k)


class DeviceSetup:
    def __init__(self, torch, device):
        self.torch = torch
        self.dev = device
        self.lib = _lib.load()
        self._temp = None
        self._total = torch.zeros(1, dtype=torch.int64, device=device)
        self._flag = torch.zeros(1, dtype=torch.int32, device=device)

    # ---- helpers ----------------------------------------------------------------------------------------
    def st(self):
        return _lib.stream_handle(self.torch)

    def empty(self, n, dtype):
        return self.torch.empty(max(int(n), 0), dtype=dtype, device=self.dev)

    def temp(self, nbytes):
        if self._temp is None or self._temp.numel() < nbytes:
            self._temp = None
            self._temp = self.torch.empty(int(nbytes), dtype=self.torch.uint8, device=self.dev)
        return self._temp

    def upload(self, A):
        A = F.canonical_csr(A)
        t = self.torch
        return DevCSR(A.shape, t.from_numpy(A.indptr).to(self.dev), t.from_numpy(A.indices).to(self.dev),
                      t.from_numpy(A.data).to(self.dev))

    def download(self, A):
        M = F.raw_csr(A.indptr.cpu().numpy(), A.indices.cpu().numpy(), A.values.cpu().numpy(), A.shape)
        return M

    def scan(self, counts, n):
        """int32 row pointer (n+1) from int32 counts; returns (indptr tensor, total)"""
        t = self.torch
        out = self.empty(n + 1, t.int32)
        nb = int(self.lib.mg_scan_workspace_size(max(n, 1)))
        tmp = self.temp(nb)
        _lib.check(self.lib.mg_exclusive_scan_i32(n, counts.data_ptr(), out.data_ptr(), self._total.data_ptr(),
                                                  tmp.data_ptr(), nb, self.st()), "mg_exclusive_scan_i32")
        return out, int(self._total.item())

    def argsort_i32(self, keys, bits):
        """stable argsort of non-negative int32 keys on their low `bits` bits (LSD radix sort)"""
        t = self.torch
        n = keys.numel()
        ks, perm, iota = self.empty(n, t.int32), self.empty(n, t.int32), self.empty(n, t.int32)
        nb = int(self.lib.mg_sort_workspace_size(max(n, 1)))
        tmp = self.temp(nb)
        _lib.check(self.lib.mg_stable_argsort_i32(n, keys.data_ptr(), ks.data_ptr(), perm.data_ptr(), iota.data_ptr(),
                                                  int(bits), tmp.data_ptr(), nb, self.st()), "mg_stable_argsort_i32")
        return perm

    def row_col_order(self, rows, cols, n_rows, n_cols):
        """stable sort order of (row, col) pairs: by column, then stably by row"""
        bits_c = max(1, int(np.ceil(np.log2(max(n_cols, 2)))))
        bits_r = max(1, int(np.ceil(np.log2(max(n_rows, 2)))))
        if cols is None:
            return self.argsort_i32(rows, bits_r)
        o1 = self.argsort_i32(cols, bits_c)
        o2 = self.argsort_i32(rows[o1.long()].contiguous(), bits_r)
        return o1[o2.long()].contiguous()

    # ---- kernels -------------------------------------------------------------------------------------------
    def transpose(self, A):
        t = self.torch
        nr, nc = A.shape
        ip = self.empty(nc + 1, t.int32)
        ix = self.empty(A.nnz, t.int32)
        va = self.empty(A.nnz, t.float64)
        work = self.temp(int(self.lib.mg_csr_transpose_workspace(max(A.nnz, 1))))
        _lib.check(self.lib.mg_csr_transpose(nr, nc, A.nnz, *A.ptrs(), ip.data_ptr(), ix.data_ptr(), va.data_ptr(),
                                             work.data_ptr(), self.st()), "mg_csr_transpose")
        return DevCSR((nc, nr), ip, ix, va)

    @staticmethod
    def _group_for(avg_b_row, log_t, numeric):
        g = 4 if avg_b_row <= 4 else 8 if avg_b_row <= 12 else 16 if avg_b_row <= 24 else 32
        while g < 32 and (256 // g) * (1 << log_t) * (12 if numeric else 4) > 200 * 1024:
            g *= 2
        if (256 // g) * (1 << log_t) * (12 if numeric else 4) > 200 * 1024:
            raise _lib.MgError("SpGEMM row too long for the shared-memory hash table (2^%d slots)" % log_t)
        return g

    def spgemm(self, A, B):
        """C = A @ B: sorted columns, values accumulated in SciPy's csr_matmat order, exact zeros pruned."""
        t = self.torch
        if A.shape[1] != B.shape[0]:
            raise ValueError("dimension mismatch")
        n = A.shape[0]
        avg = B.nnz / max(B.shape[0], 1)
        counts = self.empty(n, t.int32)
        # the symbolic pass clears and counts a whole table per row: start from the size twice the average number of
        # products per row asks for (at least 2^5, at most 2^7 as before) and grow on overflow
        est = 2.0 * (A.nnz / max(n, 1)) * avg
        log_t = min(7, max(5, int(np.ceil(np.log2(max(2.0 * est, 2.0))))))
        while True:
            g = self._group_for(avg, log_t, False)
            self._flag.zero_()
            _lib.check(self.lib.mg_spgemm_symbolic(n, A.indptr.data_ptr(), A.indices.data_ptr(), B.indptr.data_ptr(),
                                                   B.indices.data_ptr(), g, log_t, counts.data_ptr(),
                                                   self._flag.data_ptr(), self.st()), "mg_spgemm_symbolic")
            if int(self._flag.item()) == 0:
                break
            log_t += 1
            if log_t > 14:
                raise _lib.MgError("SpGEMM symbolic pass: row exceeds 2^14 distinct columns")
        max_row = int(counts.max().item()) if n else 0
        cptr, total = self.scan(counts, n)
        cidx = self.empty(total, t.int32)
        cval = self.empty(total, t.float64)
        log_n = max(4, int(np.ceil(np.log2(max(2 * max_row, 2)))))
        g = self._group_for(avg, log_n, True)
        nzc = self.empty(n, t.int32)
        self._flag.zero_()
        _lib.check(self.lib.mg_spgemm_numeric(n, *A.ptrs(), *B.ptrs(), g, log_n, cptr.data_ptr(), cidx.data_ptr(),
                                              cval.data_ptr(), nzc.data_ptr(), self._flag.data_ptr(), self.st()),
                   "mg_spgemm_numeric")
        if int(self._flag.item()) != 0:
            raise _lib.MgError("SpGEMM numeric pass overflowed its hash table")
        optr, ototal = self.scan(nzc, n)
        if ototal == total:
            return DevCSR((n, B.shape[1]), cptr, cidx, cval)
        oidx = self.empty(ototal, t.int32)
        oval = self.empty(ototal, t.float64)
        _lib.check(self.lib.mg_csr_compact_nonzeros(n, cptr.data_ptr(), cidx.data_ptr(), cval.data_ptr(),
                                                    optr.data_ptr(), oidx.data_ptr(), oval.data_ptr(), self.st()),
                   "mg_csr_compact_nonzeros")
        return DevCSR((n, B.shape[1]), optr, oidx, oval)

    def galerkin(self, A, Q, QT, keep_pattern=None):
        """A_c = Q^T A Q exactly as SciPy evaluates csr_matrix(i.T @ A @ i) (Multigrid.py:97-98):
        T = A^T Q, C = Q^T T, A_c = C^T.  keep_pattern (a list): the pattern of A^T is appended to it -- the first-fit
        colouring of the level walks it and need not transpose A again."""
        AT = self.transpose(A)
        if keep_pattern is not None:
            keep_pattern.append((AT.indptr, AT.indices))
        T = self.spgemm(AT, Q)
        del AT
        self.last_product_nnz = T.nnz              # nnz(A^T Q): the intermediate product of SURVEY 8(d)'s byte formula
        C = self.spgemm(QT, T)
        del T
        return self.transpose(C)

    def permute(self, A, perm, col_iperm):
        t = self.torch
        if perm is None and col_iperm is None:
            return A
        n = A.shape[0]
        if perm is None:
            optr = A.indptr
        else:
            lens = self.empty(n, t.int32)
            _lib.check(self.lib.mg_csr_row_lengths(n, A.indptr.data_ptr(), perm.data_ptr(), lens.data_ptr(), self.st()),
                       "mg_csr_row_lengths")
            optr, total = self.scan(lens, n)
            assert total == A.nnz
        oidx = self.empty(A.nnz, t.int32)
        oval = self.empty(A.nnz, t.float64)
        _lib.check(self.lib.mg_csr_permute(n, *A.ptrs(), _lib.ptr(perm), _lib.ptr(col_iperm), optr.data_ptr(),
                                           oidx.data_ptr(), oval.data_ptr(), self.st()), "mg_csr_permute")
        return DevCSR(A.shape, optr, oidx, oval)

    def to_sell(self, A):
        from .engine import DeviceSell
        t = self.torch
        n = A.shape[0]
        nsl = (n + 31) // 32
        slen = self.empty(nsl, t.int32)
        sptr = self.empty(nsl + 1, t.int64)
        nb = int(self.lib.mg_scan_workspace_size(max(nsl, 1)))
        tmp = self.temp(nb)
        total = ctypes.c_int64(0)
        maxlen = ctypes.c_int64(0)
        unilen = ctypes.c_int64(0)
        _lib.check(self.lib.mg_sell_layout(n, A.indptr.data_ptr(), slen.data_ptr(), sptr.data_ptr(),
                                           ctypes.byref(total), ctypes.byref(maxlen), ctypes.byref(unilen),
                                           tmp.data_ptr(), nb, self.st()), "mg_sell_layout")
        cols = self.empty(total.value, t.int32)
        vals = self.empty(total.value, t.float64)
        _lib.check(self.lib.mg_sell_fill(n, *A.ptrs(), sptr.data_ptr(), cols.data_ptr(), vals.data_ptr(), self.st()),
                   "mg_sell_fill")
        return DeviceSell.from_device(A.shape, A.nnz, sptr, cols, vals, maxlen.value, unilen.value)

    def dinv(self, A, perm):
        out = self.empty(A.shape[0], self.torch.float64)
        _lib.check(self.lib.mg_extract_dinv(A.shape[0], *A.ptrs(), _lib.ptr(perm), out.data_ptr(), self.st()),
                   "mg_extract_dinv")
        return out

    def first_fit_colors(self, A, max_rounds=400000, t_pattern=None, host=True):
        """The colours of formats.greedy_colors computed on the device (csrc/color_kernels.cu: dependency rounds on the
        patterns of A and A^T); returns a host int32 array, or the device tensor with host=False.  t_pattern: (indptr,
        indices) of A^T on the device if the caller has them (the Galerkin product forms A^T anyway).  Raises MgError
        (UNSUPPORTED) when the dependency chains are too long for the round-based algorithm -- the caller then uses the
        host helper."""
        t = self.torch
        n = A.shape[0]
        if t_pattern is None:
            AT = self.transpose(A)
            t_pattern = (AT.indptr, AT.indices)
        colors = self.empty(n, t.int32)
        nb = int(self.lib.mg_color_workspace_size(n))
        work = self.temp(nb)
        rounds = ctypes.c_int64(0)
        _lib.check(self.lib.mg_color_first_fit(n, A.indptr.data_ptr(), A.indices.data_ptr(), t_pattern[0].data_ptr(),
                                               t_pattern[1].data_ptr(), colors.data_ptr(), work.data_ptr(), nb,
                                               int(max_rounds), ctypes.byref(rounds), self.st()), "mg_color_first_fit")
        self.last_color_rounds = int(rounds.value)
        return colors.cpu().numpy() if host else colors

    def coloring_flags(self, A, colors_host, row0=0):
        """mg_level.flags of a level from its operator in natural ordering (rows row0.. of the global matrix when A is
        a row block with global column ids) and the GLOBAL colour array: MG_LEVEL_PROPER_COLORING if no row couples to
        another row of its colour, MG_LEVEL_NONZERO_DIAG if every row has a non-zero diagonal."""
        t = self.torch
        col = self._colors_on_device(colors_host)
        self._flag.zero_()
        _lib.check(self.lib.mg_csr_coloring_flags(A.shape[0], int(row0), *A.ptrs(), col.data_ptr(),
                                                  self._flag.data_ptr(), self.st()), "mg_csr_coloring_flags")
        bad = int(self._flag.item())
        return ((0 if bad & 1 else _lib.MG_LEVEL_PROPER_COLORING) | (0 if bad & 2 else _lib.MG_LEVEL_NONZERO_DIAG))

    def _colors_on_device(self, colors):
        """int32 colour array as a device tensor (host arrays are uploaded, device tensors taken as they are)"""
        t = self.torch
        if isinstance(colors, t.Tensor):
            return colors if colors.dtype == t.int32 else colors.to(t.int32)
        return t.from_numpy(np.ascontiguousarray(colors, dtype=np.int32)).to(self.dev)

    def color_perm(self, colors_host):
        """device perm (new -> old, stable by colour), inverse perm, host colour offsets; the colours may be a host
        array or a device tensor"""
        t = self.torch
        n = len(colors_host)
        keys = self._colors_on_device(colors_host)
        ncol = int(keys.max().item()) + 1 if n else 0
        ks = self.empty(n, t.int32)
        perm = self.empty(n, t.int32)
        iota = self.empty(n, t.int32)
        nb = int(self.lib.mg_sort_workspace_size(max(n, 1)))
        tmp = self.temp(nb)
        bits = max(1, int(np.ceil(np.log2(max(ncol, 2)))))
        _lib.check(self.lib.mg_stable_argsort_i32(n, keys.data_ptr(), ks.data_ptr(), perm.data_ptr(), iota.data_ptr(),
                                                  bits, tmp.data_ptr(), nb, self.st()), "mg_stable_argsort_i32")
        iperm = self.empty(n, t.int32)
        _lib.check(self.lib.mg_invert_permutation(n, perm.data_ptr(), iperm.data_ptr(), self.st()),
                   "mg_invert_permutation")
        cptr = np.zeros(ncol + 1, dtype=np.int64)
        if n:
            np.cumsum(t.bincount(keys.long(), minlength=ncol).cpu().numpy(), out=cptr[1:])
        return perm, iperm, cptr


def build_natural(S, A, Q_list, tm=None, t_patterns=None):
    """Upload A and the transfer operators and form the Galerkin hierarchy in natural ordering on the device.
    Returns (A_host0, A_nat, Q_nat, QT_nat).  t_patterns (a list): receives the pattern of A_l^T of every level that
    has a coarser one (level_colors walks them)."""
    L = len(Q_list) + 1
    if isinstance(A, DevCSR):                              # already on the device (assembly_device / neural2d)
        A_host0 = None
        A_nat = [A]
    else:
        A_host0 = F.solver_csr(A)                          # Solver.py:18 stores csc_matrix(matrix)
        if tm:
            tm.mark("host format conversion")
        A_nat = [S.upload(A_host0)]
    Q_nat, QT_nat = [], []
    for l in range(L - 1):
        Q = Q_list[l] if isinstance(Q_list[l], DevCSR) else S.upload(Q_list[l])
        if Q.shape[0] != A_nat[l].shape[0]:
            raise ValueError("Q_%d has %d rows, level operator has %d" % (l, Q.shape[0], A_nat[l].shape[0]))
        if tm:
            tm.mark("upload")
        QT = S.transpose(Q)
        Q_nat.append(Q)
        QT_nat.append(QT)
        if tm:
            tm.mark("transpose Q")
        A_nat.append(S.galerkin(A_nat[l], Q, QT, t_patterns))
        if tm:
            dt = tm.mark("Galerkin SpGEMM")
            # SURVEY 8(d), SpGEMM row: read A, Q, Q^T once, write and read the intermediate product, write A_c
            csr = lambda nnz, n: 12 * nnz + 4 * (n + 1)
            a, ac = A_nat[l], A_nat[l + 1]
            nbytes = (csr(a.nnz, a.shape[0]) + csr(Q.nnz, Q.shape[0]) + csr(QT.nnz, QT.shape[0])
                      + 2 * csr(S.last_product_nnz, a.shape[0]) + csr(ac.nnz, ac.shape[0]))
            tm.galerkin_levels.append({"level": l, "rows": a.shape[0], "nnz_A": a.nnz, "nnz_Q": Q.nnz,
                                       "nnz_AQ": S.last_product_nnz, "coarse_rows": ac.shape[0], "nnz_Ac": ac.nnz,
                                       "ms": round(dt * 1e3, 3), "algorithmic_bytes": nbytes,
                                       "gb_per_s": round(nbytes / dt / 1e9, 1) if dt > 0 else None})
    return A_host0, A_nat, Q_nat, QT_nat


def level_colors(S, smoother, colors, A_host0, A_nat, t_patterns=None):
    """Per level: colour array (or None) for multicolour Gauss-Seidel; the coarsest level is never coloured.  Returns a
    ColorList: colours found on the device stay there until somebody reads them on the host."""
    L = len(A_nat)
    out = ColorList()
    for l in range(L):
        if smoother == "mcgs" and l < L - 1:
            if colors is not None and colors[l] is not None:
                col = np.ascontiguousarray(colors[l], dtype=np.int32)
            else:
                col = None
                # first-fit on the device by dependency rounds (csrc/color_kernels.cu: the colours of the serial
                # helper, entry for entry; 8193^2: 0.78 s for the whole hierarchy instead of 2.3 s, profiles/
                # r02_bench_device_colours.json); small levels and long dependency chains take the serial helper
                if os.environ.get("MGB_DEVICE_COLORS", "1") == "1" and A_nat[l].shape[0] >= 50000:
                    try:
                        col = S.first_fit_colors(A_nat[l], host=False,
                                                 t_pattern=t_patterns[l] if t_patterns and l < len(t_patterns) else None)
                    except _lib.MgError:
                        col = None                                       # chains too long: serial helper below
                if col is None:
                    pat = A_host0 if (l == 0 and A_host0 is not None) else F.raw_csr(
                        A_nat[l].indptr.cpu().numpy(), A_nat[l].indices.cpu().numpy(), np.zeros(A_nat[l].nnz),
                        A_nat[l].shape)
                    col = F.greedy_colors(pat)[0]
            out.append(col)
        else:
            out.append(None)
    return out


def build_replicated_level(h, S, l, L, A_host0, A_nat, Q_nat, QT_nat, perms, iperms, cptrs, dense_coarse_max):
    """One level held in full on this GPU (colour-blocked ordering, SELL-32)."""
    from .engine import Level
    torch, dev = h.torch, h.device
    lev = Level()
    lev.n = A_nat[l].shape[0]
    lev.perm = perms[l]
    lev.color_ptr = cptrs[l]
    lev.nnz_A = A_nat[l].nnz
    if l < L - 1:
        Ap = S.permute(A_nat[l], perms[l], iperms[l])
        lev.A = S.to_sell(Ap)
        del Ap
        lev.dinv = S.dinv(A_nat[l], perms[l])
        Qp = S.permute(Q_nat[l], perms[l], iperms[l + 1])
        lev.Q = S.to_sell(Qp)
        del Qp
        QTp = S.permute(QT_nat[l], perms[l + 1], iperms[l])
        lev.QT = S.to_sell(QTp)
        del QTp
        lev.nnz_Q = Q_nat[l].nnz
        if h.smoother == "lexgs":
            lev.csr = (A_nat[l].indptr, A_nat[l].indices, A_nat[l].values)
            pat = A_host0 if (l == 0 and A_host0 is not None) else S.download(A_nat[l])
            lp, lr = F.lex_levels(pat)
            lev.lex_ptr = torch.from_numpy(lp).to(dev)
            lev.lex_rows = torch.from_numpy(lr).to(dev)
            lev.lex_nlevels = len(lp) - 1
    else:
        h._coarsest_from_device_csr(lev, A_nat[l], dense_coarse_max)
    return lev


class PhaseTimer:
    """wall-clock seconds per setup phase (the device is synchronised at every mark: setup only)"""

    def __init__(self, torch):
        import time
        self.torch, self.time = torch, time
        self.t = time.perf_counter()
        self.phases = {}
        self.galerkin_levels = []      # per level: time and SURVEY 8(d) bytes of the Galerkin product

    def mark(self, name):
        self.torch.cuda.synchronize()
        now = self.time.perf_counter()
        dt = now - self.t
        self.phases[name] = self.phases.get(name, 0.0) + dt
        self.t = now
        return dt


def setup_device(h, A, Q_list, colors, dense_coarse_max):
    """Populate `h.levels` of a DeviceHierarchy with device-built data (same contents as the host path)."""
    torch, dev = h.torch, h.device
    S = DeviceSetup(torch, dev)
    h._setup = S
    L = h.nlevels
    tm = PhaseTimer(torch)
    t_patterns = [] if h.smoother == "mcgs" and colors is None else None
    A_host0, A_nat, Q_nat, QT_nat = build_natural(S, A, Q_list, tm, t_patterns)
    # orderings
    h.colors = level_colors(S, h.smoother, colors, A_host0, A_nat, t_patterns)
    del t_patterns
    tm.mark("colouring")
    if h.smoother == "chebyshev":
        h._chebyshev_setup(S, A_nat)
        tm.mark("Chebyshev bounds (Lanczos)")
    perms, iperms, cptrs = [], [], []
    for l in range(L):
        if h.colors.device(l) is not None:
            p, ip, cp = S.color_perm(h.colors.device(l))
        else:
            p = ip = cp = None
        perms.append(p)
        iperms.append(ip)
        cptrs.append(cp)
    tm.mark("colour permutations")
    h.levels = []
    for l in range(L):
        h.levels.append(build_replicated_level(h, S, l, L, A_host0, A_nat, Q_nat, QT_nat, perms, iperms, cptrs,
                                               dense_coarse_max))
        tm.mark("coarsest factorisation" if l == L - 1 else "permute + SELL build")
    for k, v in (getattr(getattr(h.levels[-1], "coarse", None), "timing", None) or {}).items():
        tm.phases["coarsest: " + k] = v          # the split of "coarsest factorisation"
    h.setup_timing = tm.phases
    h.setup_galerkin = tm.galerkin_levels
    h.host_A = None
    h.host_Q = None
    if h.keep_host:
        h._dev_A_nat = A_nat
        h._dev_Q_nat = Q_nat
    S._temp = None
    torch.cuda.synchronize()


def download_level_matrix(h, l):
    A = getattr(h, "_dev_A_nat", None)
    if A is None:
        raise _lib.MgError("level matrices were not kept (keep_host=False)")
    return h._setup.download(A[l])


def chebyshev_lambda_max(S, A, steps=F.CHEBY_LANCZOS_STEPS):
    """Estimate of lambda_max(D^-1 A) for the Chebyshev smoother: `steps` Lanczos steps on D^-1/2 A D^-1/2 on the
    device (mg_spmv_csr, mg_dot, mg_axpby; the diagonal scalings are element-wise products), the tridiagonal
    eigenproblem with NumPy.  A is the level's operator in NATURAL order (DevCSR); the start vector is a hash of the
    global row index (formats.chebyshev_start_vector), so every rank and every ordering gets the same bits.  The
    operations are those of formats.chebyshev_lambda_max_host."""
    torch, lib, dev = S.torch, S.lib, S.dev
    n = A.shape[0]
    st = S.st()
    dinv = S.dinv(A, None)
    if not bool(torch.all(dinv > 0.0).item()):
        raise ValueError("the Chebyshev smoother needs a positive diagonal")
    s = torch.sqrt(dinv)
    ws = torch.empty(1 << 16, dtype=torch.float64, device=dev)
    out = torch.empty(1, dtype=torch.float64, device=dev)

    def dot(x, y):
        _lib.check(lib.mg_dot(n, x.data_ptr(), y.data_ptr(), ws.data_ptr(), out.data_ptr(), st), "mg_dot")
        return float(out.item())

    def axpby(a, x, b, y, o):
        _lib.check(lib.mg_axpby(n, float(a), x.data_ptr(), float(b), _lib.ptr(y), o.data_ptr(), st), "mg_axpby")

    v = F.chebyshev_start_vector(torch.arange(n, dtype=torch.int64, device=dev))
    axpby(1.0 / np.sqrt(dot(v, v)), v, 0.0, None, v)
    v_prev = torch.empty_like(v)
    u = torch.empty_like(v)
    w = torch.empty_like(v)
    alphas, betas = [], []
    beta = 0.0
    for k in range(int(steps)):
        torch.mul(s, v, out=u)
        _lib.check(lib.mg_spmv_csr(n, *A.ptrs(), u.data_ptr(), w.data_ptr(), st), "mg_spmv_csr")
        torch.mul(s, w, out=w)
        a = dot(w, v)
        axpby(1.0, w, -a, v, w)
        if k > 0:
            axpby(1.0, w, -beta, v_prev, w)
        alphas.append(a)
        beta = float(np.sqrt(dot(w, w)))
        if k == steps - 1 or F.lanczos_breakdown(beta, alphas):
            break
        betas.append(beta)
        v_prev, v = v, v_prev
        axpby(1.0 / beta, w, 0.0, None, v)
    return F.lanczos_tridiagonal_max(alphas, betas)
