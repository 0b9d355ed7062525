"""Device multigrid hierarchy and V-cycle engine (host side of libmgb200).

`DeviceHierarchy` owns, per level, the operator A_l, the transfer operators Q_l / Q_l^T (SELL-32, fp64 values,
int32 columns), the level vectors and the smoother data, all resident in HBM, and replays one captured CUDA
graph per V-cycle.  It is what `learnmultigrid_b200.solvers.Multigrid` drives; the arithmetic it performs is
the reference's `Multigrid.v_cycle` (learn_multigrid/solvers/Multigrid.py:77-124) with the Galerkin product
(:97-98) and the coarse factorisation (:106) hoisted out of the cycle.

Orderings.  For multicolour Gauss-Seidel every level is stored colour-blocked (rows of colour 0 first, ...;
natural order inside a colour; matrix columns and the transfer operators relabelled accordingly; entries keep
their natural order inside every row), so that each colour's sweep streams one contiguous slab of the matrix
and reads/writes x contiguously.  Vectors are permuted once on the way in and out.
"""
import ctypes
import os

import numpy as np
import scipy.sparse as sp

from . import _lib
from . import formats as F
from . import setup_device as SD
from .coarse import build_coarse_solver

DENSE_COARSE_MAX = 4096


class DeviceSell:
    """SELL-32 matrix in device memory."""

    def __init__(self, torch, A_csr, device, sell=None):
        slice_ptr, cols, vals = F.csr_to_sell(A_csr) if sell is None else sell
        self.shape = A_csr.shape
        self.nnz = int(A_csr.nnz)
        self.padded = int(slice_ptr[-1])
        self.slice_ptr = torch.from_numpy(slice_ptr).to(device)
        self.cols = torch.from_numpy(cols).to(device)
        self.vals = torch.from_numpy(vals).to(device)
        d = np.diff(slice_ptr) // 32
        self.max_len = int(d.max()) if len(d) else 0
        self.uniform_len = self.max_len if len(d) and int(d.min()) == self.max_len else 0
        self.struct = _lib.mg_sell(self.shape[0], self.shape[1], (self.shape[0] + 31) // 32,
                                   self.slice_ptr.data_ptr(), self.cols.data_ptr(), self.vals.data_ptr(),
                                   self.max_len, self.uniform_len)
        self._attach_value_dict()
        self._attach_slice_offsets()
        self._attach_patterns()

    VALUE_DICT_MIN_ROWS = 1 << 16      # smaller matrices are latency-bound launches: a dictionary buys nothing there

    def _attach_value_dict(self):
        """Value dictionary (csrc/valdict.cu): if the matrix holds at most 256 distinct values and its rows have at
        most 8 entries, keep one byte per entry next to the values; the streaming kernels then read that byte and look
        the double up in a 2 KB table.  MGB_VALUE_DICT=0 switches it off."""
        self.val_idx = self.val_table = None
        self.distinct_values = None
        floor = int(os.environ.get("MGB_VALUE_DICT_MIN_ROWS", self.VALUE_DICT_MIN_ROWS))
        if (os.environ.get("MGB_VALUE_DICT", "1") == "0" or not 1 <= self.max_len <= 8 or self.shape[0] < floor
                or self.vals.numel() == 0):
            return
        import torch
        lib = _lib.load()
        dev = self.vals.device
        idx = torch.empty(self.vals.numel(), dtype=torch.uint8, device=dev)
        table = torch.zeros(256, dtype=torch.float64, device=dev)
        work = torch.empty(int(lib.mg_value_dict_workspace()), dtype=torch.uint8, device=dev)
        cnt = ctypes.c_int(0)
        _lib.check(lib.mg_value_dict_build(self.vals.numel(), self.vals.data_ptr(), idx.data_ptr(), table.data_ptr(),
                                           work.data_ptr(), ctypes.byref(cnt), _lib.stream_handle(torch)),
                   "mg_value_dict_build")
        if cnt.value > 0:
            self.distinct_values = int(cnt.value)
            self.val_idx, self.val_table = idx, table
            self.struct.d_val_idx = idx.data_ptr()
            self.struct.d_val_table = table.data_ptr()

    IMPLIED_MIN_ROWS = 1 << 19      # the kernels' floor (mg_set_implied_min_rows): smaller matrices never use a table

    def _attach_slice_offsets(self):
        """Implied columns (sell_core.cuh): the per-slice column offsets of a uniform matrix with <= 8 entries per row
        (mg_sell_slice_offsets), deduplicated: a structured level has a handful of distinct offset records, so a slice
        keeps two bytes (the id of its record, 0xffff = not regular) and the records sit in a table, most frequent
        first.  Kept when at least half of the slices are regular (structured stencil levels: ~99 %; unstructured
        numberings: none).  MGB_IMPLIED_COLUMNS=0 switches it off."""
        self.slice_rec = self.rec_table = self.rec_vals = None
        self.regular_slices = 0
        self._spec_keep = None
        floor = int(os.environ.get("MGB_IMPLIED_MIN_ROWS", self.IMPLIED_MIN_ROWS))
        if (os.environ.get("MGB_IMPLIED_COLUMNS", "1") == "0" or not 1 <= self.uniform_len <= 8
                or self.shape[0] < max(floor // 2, 1)):
            return
        import torch
        nsl = (self.shape[0] + 31) // 32
        dev = self.cols.device
        off = torch.empty(nsl * 8, dtype=torch.int32, device=dev)
        cnt = torch.zeros(1, dtype=torch.int64, device=dev)
        _lib.check(_lib.load().mg_sell_slice_offsets(ctypes.byref(self.struct), off.data_ptr(), cnt.data_ptr(),
                                                     _lib.stream_handle(torch)), "mg_sell_slice_offsets")
        self.regular_slices = int(cnt.item())
        if 2 * self.regular_slices < nsl:
            return
        # Deduplicated records (formats.slice_records).  Implied values (sell_core.cuh, IMPV): with a value dictionary the
        # records also carry the values where the 32 rows of a slice hold the same value per entry -- on a
        # constant-coefficient stencil level that is every slice without a boundary node -- and a slice that is regular
        # in its columns only then counts as irregular; kept when that loses at most a tenth of the regular slices
        # (variable coefficients have no dictionary to begin with).  MGB_IMPLIED_VALUES=0: columns only.
        with_values = self.val_idx is not None and os.environ.get("MGB_IMPLIED_VALUES", "1") != "0"
        ids, self.rec_table, self.rec_vals, self.regular_slices = F.slice_records(
            torch, off.view(nsl, 8), self.val_idx if with_values else None, self.val_table if with_values else None,
            self.uniform_len)
        self.slice_rec = ids
        self.struct.d_slice_rec = ids.data_ptr()
        self.struct.d_rec_table = self.rec_table.data_ptr()
        self.struct.nrec = int(self.rec_table.shape[0])
        if self.rec_vals is not None:
            self.struct.d_rec_vals = self.rec_vals.data_ptr()
        self.set_spec_blocks([0, self.shape[0]])

    PATTERN_SAMPLE = 4096        # slices looked at first: a matrix whose sample shares few patterns is skipped

    def _attach_patterns(self):
        """Implied transfer columns (sell_core.cuh, sell_pattern_kernel): for a rectangular uniform matrix with <= 8
        entries per row -- a transfer operator, whose columns live in the other level's numbering -- a record id and a
        base column (the slice's first stored column) per slice; the records (formats.pattern_records) hold the columns
        relative to the base and the values of the slice's 32 rows.  They sit in the fields of the implied columns,
        which a transfer operator does not use, flagged by nrec < 0; the bases follow the patterns in d_rec_table
        (include/mgb200.h).  Kept when at least half of the slices have a record (structured hierarchies: 98-99.99 %);
        an evenly spaced sample of slices is deduplicated first, so that matrices whose slices share nothing
        (unstructured numberings, the Galerkin levels of variable coefficients) cost only that.
        MGB_IMPLIED_TRANSFERS=0 switches it off."""
        self.pat_rec = self.pat_table = self.pat_vals = None
        self.pattern_slices = 0
        floor = int(os.environ.get("MGB_IMPLIED_MIN_ROWS", self.IMPLIED_MIN_ROWS))
        L = self.uniform_len
        if (os.environ.get("MGB_IMPLIED_TRANSFERS", "1") == "0" or self.slice_rec is not None
                or self.shape[0] == self.shape[1] or not 1 <= L <= 8 or self.shape[0] < max(floor, 1)):
            return
        import torch
        nsl = (self.shape[0] + 31) // 32
        if nsl > 2 * self.PATTERN_SAMPLE:
            pick = torch.linspace(0, nsl - 2, self.PATTERN_SAMPLE, device=self.cols.device).long()
            sc = self.cols.view(nsl, 32 * L)[pick].reshape(-1)
            sv = self.vals.view(nsl, 32 * L)[pick].reshape(-1)
            *_, nreg = F.pattern_records(torch, sc, sv, self.PATTERN_SAMPLE * 32, L)
            if 2 * nreg < self.PATTERN_SAMPLE:
                return
        base, ids, delta, pvals, nreg = F.pattern_records(torch, self.cols, self.vals, self.shape[0], L)
        if 2 * nreg < nsl:
            return
        self.pat_rec, self.pat_vals = ids, pvals
        self.pat_table = torch.cat([delta.reshape(-1), base])           # patterns, then the base of every slice
        self.pattern_slices = nreg
        s = self.struct
        s.d_slice_rec, s.d_rec_table, s.d_rec_vals = ids.data_ptr(), self.pat_table.data_ptr(), pvals.data_ptr()
        s.nrec = -int(delta.shape[0])
        self.set_pattern_blocks([0, self.shape[0]])

    def set_pattern_blocks(self, row_ptr):
        """Tell the launcher which pattern the slices of each row block [row_ptr[k], row_ptr[k+1]) mostly use (the
        colour blocks of the level the rows belong to) and how many of them do: where that is most, a launch gathers
        with it before the slice's own id has arrived (mg_sell.h_spec_*; the kernel knows 8 blocks, later rows count to
        the eighth)."""
        if self.pat_rec is None:
            return
        import torch
        row_ptr = [int(v) for v in row_ptr]
        if len(row_ptr) > 9:
            row_ptr = row_ptr[:8] + row_ptr[-1:]
        nb = len(row_ptr) - 1
        rows = (ctypes.c_int64 * (nb + 1))(*row_ptr)
        rec = (ctypes.c_int32 * (9 * max(nb, 1)))()
        for k in range(nb):
            ids = self.pat_rec[row_ptr[k] // 32:max((row_ptr[k + 1] + 31) // 32, row_ptr[k] // 32 + 1)]
            n = ids.numel()
            ids = ids[ids >= 0]
            cnt = torch.bincount(ids.long(), minlength=1) if ids.numel() else torch.zeros(1, dtype=torch.int64)
            rec[9 * k] = int(cnt.argmax().item())
            rec[9 * k + 1] = int(1000 * int(cnt.max().item()) // max(n, 1))
        self._spec_keep = (rows, rec)
        self.struct.n_spec = nb
        self.struct.h_spec_row = ctypes.cast(rows, ctypes.POINTER(ctypes.c_int64))
        self.struct.h_spec_rec = ctypes.cast(rec, ctypes.POINTER(ctypes.c_int32))

    @property
    def slice_off(self):
        """per-slice offset records [nslices][8] rebuilt from ids + table (tests; None without implied columns)"""
        if self.slice_rec is None:
            return None
        import torch
        out = torch.zeros(self.slice_rec.numel(), 8, dtype=torch.int32, device=self.slice_rec.device)
        reg = self.slice_rec >= 0
        out[reg] = self.rec_table[self.slice_rec[reg].long()]
        out[~reg, 0] = _lib.SLICE_IRREGULAR
        return out.reshape(-1)

    def set_spec_blocks(self, row_ptr):
        """Tell the launcher which offset record the slices of each row block [row_ptr[k], row_ptr[k+1]) mostly use
        (the colour blocks: the ranges the cycle launches over), so that a launch can carry that record by value and
        gather with it before the slice's own id has arrived (mg_sell.h_spec_*)."""
        if self.slice_rec is None:
            return
        import torch
        row_ptr = [int(v) for v in row_ptr]
        nb = len(row_ptr) - 1
        table = self.rec_table.cpu().numpy()
        vals_table = None if self.rec_vals is None else self.rec_vals.cpu().numpy()
        rows = (ctypes.c_int64 * (nb + 1))(*row_ptr)
        rec = (ctypes.c_int32 * (9 * max(nb, 1)))()
        vals = (ctypes.c_double * (8 * max(nb, 1)))()
        for k in range(nb):
            s0, s1 = row_ptr[k] // 32, max((row_ptr[k + 1] + 31) // 32, row_ptr[k] // 32 + 1)
            ids = self.slice_rec[s0:s1]
            ids = ids[ids >= 0]
            best = int(torch.bincount(ids.long(), minlength=1).argmax().item()) if ids.numel() else 0
            rec[9 * k] = best
            for j in range(8):
                rec[9 * k + 1 + j] = int(table[best, j])
                if vals_table is not None:
                    vals[8 * k + j] = float(vals_table[best, j])
        self._spec_keep = (rows, rec, vals)
        self.struct.n_spec = nb
        self.struct.h_spec_row = ctypes.cast(rows, ctypes.POINTER(ctypes.c_int64))
        self.struct.h_spec_rec = ctypes.cast(rec, ctypes.POINTER(ctypes.c_int32))
        if vals_table is not None:
            self.struct.h_spec_vals = ctypes.cast(vals, ctypes.POINTER(ctypes.c_double))

    @classmethod
    def from_device(cls, shape, nnz, slice_ptr, cols, vals, max_len=0, uniform_len=0):
        self = cls.__new__(cls)
        self.shape = tuple(shape)
        self.nnz = int(nnz)
        self.padded = int(cols.numel())
        self.slice_ptr, self.cols, self.vals = slice_ptr, cols, vals
        self.max_len = int(max_len)
        self.uniform_len = int(uniform_len)
        self.struct = _lib.mg_sell(shape[0], shape[1], (shape[0] + 31) // 32,
                                   slice_ptr.data_ptr(), cols.data_ptr(), vals.data_ptr(), self.max_len,
                                   self.uniform_len)
        self._attach_value_dict()
        self._attach_slice_offsets()
        self._attach_patterns()
        return self

    def bytes(self):
        return self.padded * 12 + self.slice_ptr.numel() * 8

    def stream_bytes(self):
        """bytes one pass over the matrix actually reads: values, and columns or -- for regular slices of a matrix with
        implied columns (large launches) -- 4 bytes of offset per slice and entry index; with slice patterns the id
        and base column of every slice and the columns and values of the slices without a record"""
        nsl = (self.shape[0] + 31) // 32
        if self.pat_rec is not None and _lib.load().mg_set_implied_transfers(-1):
            # slice patterns (as the library is switched now): an id and a base column per slice; slices without a
            # record read their columns and values (8 B each)
            return (nsl - self.pattern_slices) * 32 * self.uniform_len * 12 + 6 * nsl
        vbytes = 1 if (self.val_idx is not None and os.environ.get("MGB_VALUE_DICT", "1") != "0") else 8
        if self.slice_rec is None or self.shape[0] < self.IMPLIED_MIN_ROWS or nsl == 0:
            return self.padded * (4 + vbytes) + (0 if self.uniform_len else self.slice_ptr.numel() * 8)
        per_slice = 32 * self.uniform_len
        irregular = nsl - self.regular_slices
        if self.rec_vals is not None and os.environ.get("MGB_IMPLIED_VALUES", "1") != "0" and vbytes == 1:
            return irregular * per_slice * (4 + vbytes) + 2 * nsl          # implied values: regular slices read their id
        return self.padded * vbytes + irregular * per_slice * 4 + 2 * nsl


class Level:
    pass


def algorithmic_bytes_csr(nnz, n):
    """S(nnz, n) of SURVEY.md 8(d): 8 B value + 4 B column per entry, 4 B row pointer per row."""
    return 12 * nnz + 4 * (n + 1)


class DeviceHierarchy:
    """Prebuilt multigrid hierarchy on one GPU.

    A        : fine operator (anything SciPy accepts), n0 x n0
    Q_list   : transfer operators [Q_0 (n0 x n1), Q_1, ...]; levels = len(Q_list) + 1
    smoother : "jacobi" | "mcgs" (multicolour Gauss-Seidel) | "lexgs" (exact index-order Gauss-Seidel)
               | "chebyshev" (Chebyshev polynomial in D^-1 A; natural order, no colouring, like "jacobi")
    colors   : optional list of per-level colour arrays for "mcgs" (default: first-fit greedy colouring)
    cheby_degree : degree of the Chebyshev polynomial (steps per smoothing sweep)
    cheby_bounds : None (default: [0.3, 1.1] x a 10-step Lanczos estimate of lambda_max(D^-1 A) per level) or one
                   (lo, hi) pair per smoothing level (levels - 1 of them)
    setup    : "device" (SpGEMM / transposes / SELL build by CUDA kernels) or "host" (NumPy/SciPy cross-check)
    """

    def __init__(self, A, Q_list, smoother="jacobi", colors=None, device=None, setup="device",
                 dense_coarse_max=DENSE_COARSE_MAX, keep_host=True, cheby_degree=2, cheby_bounds=None):
        torch = _lib.require_cuda()
        self.torch = torch
        self.lib = _lib.load()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if smoother not in ("jacobi", "mcgs", "lexgs", "chebyshev"):
            raise ValueError("unknown smoother %r" % (smoother,))
        self.smoother = smoother
        self.nlevels = len(Q_list) + 1
        if self.nlevels < 2:
            raise ValueError("need at least one transfer operator (levels >= 2)")
        self._chebyshev_args(cheby_degree, cheby_bounds)
        self.keep_host = keep_host
        self._graphs = {}
        self._keep = []          # tensors / ctypes buffers that must outlive the level structs
        self.setup_kind = setup
        if setup == "host":
            self._setup_host(A, Q_list, colors, dense_coarse_max)
        elif setup == "device":
            SD.setup_device(self, A, Q_list, colors, dense_coarse_max)
        else:
            raise ValueError("setup must be 'device' or 'host'")
        self._finish_structs()

    # ------------------------------------------------------------------------------------------------
    def _chebyshev_args(self, degree, bounds):
        """validate the Chebyshev options (ValueError) before anything is built"""
        self.cheby_degree = self.cheby_bounds = self.cheby_coefficients = self.cheby_lambda = None
        self._cheby_key = None
        if self.smoother != "chebyshev":
            return
        if bounds is not None:
            bounds = [tuple(float(v) for v in b) for b in bounds]
            if len(bounds) != self.nlevels - 1 or any(len(b) != 2 for b in bounds):
                raise ValueError("cheby_bounds needs one (lo, hi) pair per smoothing level (%d)" % (self.nlevels - 1))
        F.chebyshev_check(degree, bounds)
        self.cheby_degree = int(degree)
        self.cheby_bounds = bounds

    def _chebyshev_setup(self, S, A_nat):
        """Bounds and coefficient tables of the Chebyshev smoother, from the levels' operators in natural order (DevCSR,
        the GLOBAL operators on a partitioned hierarchy: every rank computes the same bits).  Given bounds are kept;
        otherwise [0.3, 1.1] x the Lanczos estimate of lambda_max(D^-1 A_l) (setup_device.chebyshev_lambda_max)."""
        if self.cheby_bounds is None:
            self.cheby_lambda = [SD.chebyshev_lambda_max(S, A_nat[l]) for l in range(self.nlevels - 1)]
            lo, hi = F.CHEBY_INTERVAL
            self.cheby_bounds = [(lo * lam, hi * lam) for lam in self.cheby_lambda]
        self.cheby_coefficients = [F.chebyshev_coefficients(lo, hi, self.cheby_degree) for lo, hi in self.cheby_bounds]
        # part of every graph key: a table the captured launches were not made with never replays them
        self._cheby_key = tuple(c.tobytes() for c in self.cheby_coefficients)

    def _setup_host(self, A, Q_list, colors, dense_coarse_max):
        """Hierarchy build with SciPy/NumPy on the host (formats.build_host_hierarchy), then upload."""
        torch, dev = self.torch, self.device
        L = self.nlevels
        host = F.build_host_hierarchy(A, Q_list, self.smoother, colors, with_sell=True)
        if self.smoother == "chebyshev":
            S = SD.DeviceSetup(torch, dev)
            up = [SD.DevCSR(d["A_nat"].shape, *(torch.from_numpy(np.ascontiguousarray(a, dtype=t)).to(dev) for a, t in
                                                  ((d["A_nat"].indptr, np.int32), (d["A_nat"].indices, np.int32),
                                                   (d["A_nat"].data, np.float64)))) for d in host[:-1]]
            self._chebyshev_setup(S, up)
            del up
        self.host_A = [d["A_nat"] for d in host] if self.keep_host else None
        self.host_Q = [d.get("Q_nat") for d in host[:-1]] if self.keep_host else None
        self.colors = [d["colors"] for d in host]
        self.levels = []
        for l, d in enumerate(host):
            lev = Level()
            lev.n = d["n"]
            lev.perm = None if d["perm"] is None else torch.from_numpy(d["perm"]).to(dev)
            lev.color_ptr = d["color_ptr"]
            lev.nnz_A = d["nnz_A"]
            if l < L - 1:
                lev.A = DeviceSell(torch, d["A"], dev, d["A_sell"])
                lev.dinv = torch.from_numpy(d["dinv"]).to(dev)
                lev.Q = DeviceSell(torch, d["Q"], dev, d["Q_sell"])
                lev.QT = DeviceSell(torch, d["QT"], dev, d["QT_sell"])
                lev.nnz_Q = d["nnz_Q"]
                if self.smoother == "lexgs":
                    An = d["A_nat"]
                    lev.csr = tuple(torch.from_numpy(a).to(dev) for a in (An.indptr, An.indices, An.data))
                    lev.lex_ptr = torch.from_numpy(d["lex_ptr"]).to(dev)
                    lev.lex_rows = torch.from_numpy(d["lex_rows"]).to(dev)
                    lev.lex_nlevels = len(d["lex_ptr"]) - 1
            else:
                self._setup_coarsest(lev, d["A_nat"], dense_coarse_max)
            self.levels.append(lev)

    def _setup_coarsest(self, lev, A_csr, dense_coarse_max):
        """Coarsest level from a host CSR: upload, then dense inverse or block cyclic reduction (coarse.py)."""
        torch, dev = self.torch, self.device
        ip = torch.from_numpy(A_csr.indptr).to(dev)
        ix = torch.from_numpy(A_csr.indices).to(dev)
        va = torch.from_numpy(A_csr.data).to(dev)
        self._coarsest(lev, A_csr.shape[0], ip, ix, va, dense_coarse_max, (A_csr.indptr, A_csr.indices))

    def _coarsest_from_device_csr(self, lev, A_dev, dense_coarse_max):
        self._coarsest(lev, A_dev.shape[0], A_dev.indptr, A_dev.indices, A_dev.values, dense_coarse_max, None)

    def _coarsest(self, lev, n, ip, ix, va, dense_coarse_max, host_pattern):
        solver = build_coarse_solver(self.torch, self.device, n, ip, ix, va, dense_coarse_max, host_pattern)
        lev.coarse = solver
        lev.coarse_kind = solver.kind
        lev.coarse_bytes = solver.bytes
        if solver.kind == _lib.MG_COARSE_DENSE:
            lev.coarse_inv = solver.inv
        else:
            lev.coarse_bcr = ctypes.cast(ctypes.pointer(solver.handle), ctypes.c_void_p)

    # ------------------------------------------------------------------------------------------------
    def _finish_structs(self):
        torch, dev = self.torch, self.device
        L = self.nlevels
        import time
        t0 = time.perf_counter()
        for lev in self.levels:
            n = getattr(lev, "n_vec", lev.n)          # partitioned levels: owned entries + halo
            lev.x = torch.zeros(n, dtype=torch.float64, device=dev)
            lev.b = torch.zeros(n, dtype=torch.float64, device=dev)
            lev.r = torch.zeros(n, dtype=torch.float64, device=dev)
            lev.tmp = torch.zeros(n, dtype=torch.float64, device=dev)
        n0 = self.levels[0].n
        self.n = n0
        self._stage = torch.zeros(n0, dtype=torch.float64, device=dev)       # natural-order staging
        # the pinned host staging buffer (8 n0 bytes of page-locked memory: 0.2-0.3 s at 67 M unknowns) is allocated
        # by the first transfer that needs it -- a hierarchy fed with device-resident or pinned vectors never does
        self._pinned_buf = None
        torch.cuda.synchronize()
        if getattr(self, "setup_timing", None) is not None:
            self.setup_timing["level vectors"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        self._inspect_levels()
        torch.cuda.synchronize()
        if getattr(self, "setup_timing", None) is not None:
            self.setup_timing["inspect (diagonal, colouring flags)"] = time.perf_counter() - t0
        self._norm_ws = torch.zeros(int(self.lib.mg_norm_workspace_size(n0)) + 4096, dtype=torch.float64, device=dev)
        self._norm_out = torch.zeros(1, dtype=torch.float64, device=dev)
        self._norm_host = torch.zeros(1, dtype=torch.float64).pin_memory()
        arr = (_lib.mg_level * L)()
        for l, lev in enumerate(self.levels):
            s = arr[l]
            s.n = lev.n
            s.d_x, s.d_b, s.d_r, s.d_tmp = (t.data_ptr() for t in (lev.x, lev.b, lev.r, lev.tmp))
            if getattr(lev, "dist_struct", None) is not None:
                s.dist = ctypes.pointer(lev.dist_struct)
            if l < L - 1:
                s.A, s.Q, s.QT = lev.A.struct, lev.Q.struct, lev.QT.struct
                s.d_dinv = lev.dinv.data_ptr()
                if lev.color_ptr is not None:
                    cp = (ctypes.c_int64 * len(lev.color_ptr))(*[int(v) for v in lev.color_ptr])
                    self._keep.append(cp)
                    s.ncolors = len(lev.color_ptr) - 1
                    s.h_color_ptr = ctypes.cast(cp, ctypes.POINTER(ctypes.c_int64))
                    s.flags = int(getattr(lev, "flags", 0))
                    if getattr(lev, "diag", None) is not None:
                        s.d_diag = lev.diag.data_ptr()
                if self.cheby_coefficients is not None:
                    tab = np.ascontiguousarray(self.cheby_coefficients[l], dtype=np.float64).reshape(-1)
                    ct = (ctypes.c_double * len(tab))(*[float(v) for v in tab])
                    self._keep.append(ct)
                    s.cheb_degree = self.cheby_degree
                    s.h_cheb_coef = ctypes.cast(ct, ctypes.POINTER(ctypes.c_double))
                if getattr(lev, "csr", None) is not None and getattr(lev, "lex_ptr", None) is not None:
                    s.d_csr_indptr, s.d_csr_indices, s.d_csr_values = (t.data_ptr() for t in lev.csr)
                    s.d_lex_level_ptr = lev.lex_ptr.data_ptr()
                    s.d_lex_level_rows = lev.lex_rows.data_ptr()
                    s.lex_nlevels = lev.lex_nlevels
            else:
                s.coarse_kind = lev.coarse_kind
                if lev.coarse_kind == _lib.MG_COARSE_DENSE:
                    s.d_coarse_inv = lev.coarse_inv.data_ptr()
                else:
                    s.coarse_bcr = lev.coarse_bcr
                    if getattr(lev, "coarse_bcr_dist", None) is not None:
                        s.coarse_bcr_dist = ctypes.pointer(lev.coarse_bcr_dist)
        self._level_structs = arr

    def _inspect_levels(self):
        """What the cycle may assume about every coloured level (mg_level.flags / d_diag, csrc/cycle.cu
        g_cycle_fusion): the diagonal as the Gauss-Seidel kernel finds it, whether the colouring is proper and whether
        every row has a non-zero diagonal.  Levels whose flags were already set by the builder (partitioned levels:
        the facts must hold for the GLOBAL operator, distributed.py) only get their diagonal here."""
        torch, dev = self.torch, self.device
        for lev, nxt in zip(self.levels[:-1], self.levels[1:]):
            if getattr(lev, "QT", None) is not None and getattr(nxt, "color_ptr", None) is not None:
                lev.QT.set_pattern_blocks(nxt.color_ptr)
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        st = _lib.stream_handle(torch)
        for lev in self.levels:
            if getattr(lev, "A", None) is None or lev.color_ptr is None:
                continue
            lev.diag = torch.empty(lev.n, dtype=torch.float64, device=dev)
            lev.A.set_spec_blocks(lev.color_ptr)          # launches run over colour blocks: one offset record each
            if getattr(lev, "Q", None) is not None:
                lev.Q.set_pattern_blocks(lev.color_ptr)       # Q's rows are this level's, Q^T's the next level's
            have = getattr(lev, "flags", None) is not None
            cp = torch.tensor([int(v) for v in lev.color_ptr], dtype=torch.int64, device=dev)
            flag.zero_()
            _lib.check(self.lib.mg_level_inspect(ctypes.byref(lev.A.struct), 0 if have else len(lev.color_ptr) - 1,
                                                 cp.data_ptr(), lev.diag.data_ptr(), flag.data_ptr(), st),
                       "mg_level_inspect")
            if not have:
                bad = int(flag.item())
                lev.flags = ((0 if bad & 1 else _lib.MG_LEVEL_PROPER_COLORING)
                             | (0 if bad & 2 else _lib.MG_LEVEL_NONZERO_DIAG))

    # ------------------------------------------------------------------------------------------------
    # vectors in and out (host NumPy <-> permuted device vectors)
    @property
    def _pinned(self):
        if self._pinned_buf is None:
            import time
            t0 = time.perf_counter()
            self._pinned_buf = self.torch.empty(self.n, dtype=self.torch.float64, pin_memory=True)
            self.pinned_alloc_s = time.perf_counter() - t0
        return self._pinned_buf

    def _to_level0(self, host_vec, dst):
        torch = self.torch
        # the pinned staging buffer is reused by every transfer: wait until the previous H2D copy has read it
        evt = getattr(self, "_pin_evt", None)
        if evt is not None:
            evt.synchronize()
        self._to_level0_enqueue(host_vec, dst)
        if evt is None:
            evt = self._pin_evt = torch.cuda.Event()
        evt.record(torch.cuda.current_stream())

    def _to_level0_enqueue(self, host_vec, dst):
        torch = self.torch
        if isinstance(host_vec, torch.Tensor):
            src = host_vec.reshape(-1)
            if src.dtype != torch.float64 or src.numel() != self.n:
                raise ValueError("tensor input must be float64 with %d entries" % self.n)
            if not src.is_pinned() and not src.is_cuda:
                self._pinned.copy_(src)
                src = self._pinned
        else:
            v = np.ascontiguousarray(np.asarray(host_vec, dtype=np.float64).reshape(-1))
            if v.size != self.n:
                raise ValueError("vector has %d entries, operator has %d rows" % (v.size, self.n))
            self._pinned.copy_(torch.from_numpy(v))
            src = self._pinned
        lev = self.levels[0]
        if lev.perm is None:
            dst[:self.n].copy_(src, non_blocking=True)
        else:
            self._stage.copy_(src, non_blocking=True)
            _lib.check(self.lib.mg_gather(self.n, lev.perm.data_ptr(), self._stage.data_ptr(), dst.data_ptr(),
                                          _lib.stream_handle(torch)), "mg_gather")

    def _from_level0(self, src, view=False):
        """device level-0 vector -> host (n,1) array in natural ordering.  view=True returns a view of the
        engine's pinned buffer (valid until the next transfer) instead of a fresh copy."""
        torch = self.torch
        lev = self.levels[0]
        if lev.perm is None:
            self._pinned.copy_(src[:self.n], non_blocking=True)
        else:
            _lib.check(self.lib.mg_scatter(self.n, lev.perm.data_ptr(), src.data_ptr(), self._stage.data_ptr(),
                                           _lib.stream_handle(torch)), "mg_scatter")
            self._pinned.copy_(self._stage, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        out = self._pinned.numpy()
        return out.reshape(-1, 1) if view else out.copy().reshape(-1, 1)

    def set_rhs(self, b):
        self._to_level0(b, self.levels[0].b)

    def set_x(self, x):
        self._to_level0(x, self.levels[0].x)

    def zero_x(self):
        self.levels[0].x.zero_()

    def get_x(self, view=False):
        return self._from_level0(self.levels[0].x, view)

    # ------------------------------------------------------------------------------------------------
    def residual_norm(self):
        """||b - A x||_2 on level 0, fused residual + norm (Multigrid.py:62-63), one D2H of 8 bytes."""
        torch = self.torch
        lev = self.levels[0]
        st = _lib.stream_handle(torch)
        _lib.check(self.lib.mg_sell_residual_norm2(ctypes.byref(lev.A.struct), lev.x.data_ptr(), lev.b.data_ptr(),
                                                   self._norm_ws.data_ptr(), self._norm_out.data_ptr(), st),
                   "mg_sell_residual_norm2")
        self._norm_host.copy_(self._norm_out, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(np.sqrt(self._norm_host.item()))

    def last_norm(self):
        """||b - A x||_2 left on the device by vcycle(with_norm=True): one D2H of 8 bytes."""
        torch = self.torch
        self._norm_host.copy_(self._norm_out, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(np.sqrt(self._norm_host.item()))

    def residual_vector(self):
        lev = self.levels[0]
        _lib.check(self.lib.mg_sell_residual(ctypes.byref(lev.A.struct), lev.x.data_ptr(), lev.b.data_ptr(),
                                             lev.r.data_ptr(), _lib.stream_handle(self.torch)), "mg_sell_residual")
        return self._from_level0(lev.r)

    def make_params(self, nu_pre=1, nu_post=None, omega=1.0, zero_guess_skip=True, reverse_post=False, x0_zero=False):
        """x0_zero: the cycle starts from a zero iterate on level 0 WITHOUT reading (or needing) the contents of x --
        a preconditioner application z = M^-1 r."""
        sm = {"jacobi": _lib.MG_SMOOTH_JACOBI, "mcgs": _lib.MG_SMOOTH_MCGS, "lexgs": _lib.MG_SMOOTH_LEXGS,
              "chebyshev": _lib.MG_SMOOTH_CHEBY}[self.smoother]
        return _lib.mg_cycle_params(sm, int(nu_pre), int(nu_pre if nu_post is None else nu_post), float(omega),
                                    1 if zero_guess_skip else 0, 1 if reverse_post else 0, 1 if x0_zero else 0, 0)

    def _enqueue_cycle(self, L, params, with_norm, stream):
        if with_norm:
            return self.lib.mg_vcycle_norm(self._level_structs, L, ctypes.byref(params), self._norm_ws.data_ptr(),
                                           self._norm_out.data_ptr(), stream)
        return self.lib.mg_vcycle(self._level_structs, L, ctypes.byref(params), stream)

    def vcycle(self, params, nlevels=None, use_graph=True, with_norm=False):
        """One V-cycle on the level-0 vectors (x updated in place).  The launch sequence is captured into a CUDA
        graph the first time a parameter set is used and replayed afterwards.
        with_norm: the cycle also leaves ||b - A x||^2 of the NEW iterate on the device (mg_vcycle_norm: the last
        colour sweep sums its own rows' share from registers); read it with last_norm()."""
        torch = self.torch
        L = self.nlevels if nlevels is None else int(nlevels)
        st = _lib.stream_handle(torch)
        if not use_graph or self.smoother == "lexgs":      # cooperative launches are not captured
            _lib.check(self._enqueue_cycle(L, params, with_norm, st), "mg_vcycle")
            self.last_launches = int(self.lib.mg_last_launch_count())
            return
        key = (L, params.smoother, params.nu_pre, params.nu_post, params.omega, params.zero_guess_skip,
               params.reverse_post, params.x0_zero, bool(with_norm), self._cheby_key)
        g = self._graphs.get(key)
        if g is None:
            cap = torch.cuda.Stream(device=self.device)
            cap.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(cap):
                h = cap.cuda_stream
                _lib.check(self.lib.mg_graph_begin(h), "mg_graph_begin")
                rc = self._enqueue_cycle(L, params, with_norm, h)
                launches = int(self.lib.mg_last_launch_count())
                out = ctypes.c_void_p()
                rc2 = self.lib.mg_graph_end(h, ctypes.byref(out))
                _lib.check(rc, "mg_vcycle (capture)")
                _lib.check(rc2, "mg_graph_end")
            torch.cuda.current_stream().wait_stream(cap)
            g = (out, launches)
            self._graphs[key] = g
        _lib.check(self.lib.mg_graph_launch(g[0], st), "mg_graph_launch")
        self.last_launches = g[1]

    # ------------------------------------------------------------------------------------------------
    def _comm_ptr(self):
        """the communicator of a partitioned hierarchy (distributed.py overrides), or None"""
        return None

    def pcg(self, rhs, params, error=1e-8, max_iterations=1000, view=False):
        """Conjugate gradients preconditioned by one V-cycle per iteration (BASELINE.json configs[4]), entirely in
        the level-0 ordering of this hierarchy and entirely on the device (mg_pcg_start / mg_pcg_iterate): the residual
        LIVES in the level's right-hand-side buffer and z = M^-1 r in its iterate, so nothing is copied or permuted per
        iteration; the scalars stay on the device, p.Ap comes out of the SpMV and r.r out of the update of x and r; an
        iteration is one CUDA graph, after which the host reads 8 bytes (the convergence test).  params=None: plain CG.
        Statement order = solvers/CG.py (the reference's CG.py:12-50 plus the preconditioner).  Works on a partitioned
        hierarchy too (every rank makes the same call; dots are summed over the ranks in rank order).
        Returns (solution (n,1) natural order -- this rank's block when partitioned --, history list, iterations);
        self.last_pcg_timing holds the wall-clock split transfer in / iterations / transfer out."""
        import time
        torch, lib = self.torch, self.lib
        lev = self.levels[0]
        n = self.n
        st = _lib.stream_handle(torch)
        comm = self._comm_ptr()
        if getattr(self, "_cg", None) is None:
            n_vec = getattr(lev, "n_vec", n)
            x = torch.zeros(n, dtype=torch.float64, device=self.device)
            p = torch.zeros(n_vec, dtype=torch.float64, device=self.device)
            Ap = torch.zeros(n, dtype=torch.float64, device=self.device)
            sc = torch.zeros(8, dtype=torch.float64, device=self.device)
            slots = torch.zeros(_lib.MG_MAX_RANKS, dtype=torch.float64, device=self.device)
            self._cg = (x, p, Ap, sc, slots)
            self._cg_struct = _lib.mg_pcg(x.data_ptr(), p.data_ptr(), Ap.data_ptr(), sc.data_ptr(),
                                          self._norm_ws.data_ptr(), slots.data_ptr())
            self._cg_graphs = {}
        x, p, Ap, sc, _ = self._cg
        pcg = ctypes.byref(self._cg_struct)
        pp = None if params is None else ctypes.byref(params)

        def read_rr():
            self._norm_host.copy_(sc[4:5], non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return float(np.sqrt(self._norm_host.item()))

        def iterate(first):
            key = (first, None if params is None else (params.smoother, params.nu_pre, params.nu_post, params.omega,
                                                       params.zero_guess_skip, params.reverse_post, self._cheby_key))
            g = self._cg_graphs.get(key)
            if g is None:
                if self.smoother == "lexgs" and params is not None:      # cooperative launches are not captured
                    _lib.check(lib.mg_pcg_iterate(comm, self._level_structs, self.nlevels, pp, pcg, first, st),
                               "mg_pcg_iterate")
                    return
                cap = torch.cuda.Stream(device=self.device)
                cap.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(cap):
                    h = cap.cuda_stream
                    _lib.check(lib.mg_graph_begin(h), "mg_graph_begin")
                    rc = lib.mg_pcg_iterate(comm, self._level_structs, self.nlevels, pp, pcg, first, h)
                    out = ctypes.c_void_p()
                    rc2 = lib.mg_graph_end(h, ctypes.byref(out))
                    _lib.check(rc, "mg_pcg_iterate (capture)")
                    _lib.check(rc2, "mg_graph_end")
                torch.cuda.current_stream().wait_stream(cap)
                g = self._cg_graphs[key] = out
                self._graphs[("pcg",) + key] = (out, 0)        # destroyed with the other graphs
            _lib.check(lib.mg_graph_launch(g, st), "mg_graph_launch")

        t0 = time.perf_counter()
        self.set_rhs(rhs)                      # r = b - A*0 = b
        torch.cuda.current_stream().synchronize()
        t1 = time.perf_counter()
        _lib.check(lib.mg_pcg_start(comm, self._level_structs, pcg, st), "mg_pcg_start")
        track = [read_rr()]
        its = 0
        for k in range(max_iterations):
            its += 1
            iterate(1 if k == 0 else 0)
            res = read_rr()
            track.append(res)
            if res <= error:
                break
        t2 = time.perf_counter()
        sol = self._from_level0(x, view)
        t3 = time.perf_counter()
        self.last_pcg_timing = {"transfer_in_s": t1 - t0, "iterations_s": t2 - t1, "transfer_out_s": t3 - t2,
                                "iterations": its}
        return sol, track, its

    def gmres(self, rhs, params, error=1e-8, max_iterations=1000, restart=30, x0=None, view=False):
        """Restarted GMRES(restart), right-preconditioned by one V-cycle from zero per Arnoldi step (params=None: no
        preconditioner), entirely in the level-0 ordering of this hierarchy and on the device (mg_gmres_start /
        mg_gmres_iterate / mg_gmres_finish): classical Gram-Schmidt in one pass, Givens rotations, the scalars on the
        device; a step is one CUDA graph (per step index and parameter set; index-order Gauss-Seidel runs uncaptured)
        after which the host reads 8 bytes.  Valid for nonsymmetric operators and preconditioners, unlike pcg.
        Works on a partitioned hierarchy too (every rank makes the same call; dots are summed over the ranks in rank
        order).

        error is absolute, as in pcg.  The history is ||b - A x0||, then the GMRES estimate |g_{j+1}| of the residual
        after every step.  At every restart, and when the estimate reaches `error`, x is updated and the true residual
        recomputed; while it is above `error` and steps remain, the solve restarts from there.  max_iterations counts
        Arnoldi steps over all restarts; when it runs out, x is the iterate of the last completed step.
        Returns (solution (n,1) natural order -- this rank's block when partitioned --, history list, steps, true
        residual of the solution); self.last_gmres_timing holds the wall-clock split transfer in / iterations /
        transfer out (orthogonalisation: None, the steps run as graphs; tools/bench_gmres.py times its kernels)."""
        import time
        torch, lib = self.torch, self.lib
        restart = int(restart)
        if restart < 1:
            raise ValueError("restart must be >= 1 (got %d)" % restart)
        lev = self.levels[0]
        n = self.n
        st = _lib.stream_handle(torch)
        comm = self._comm_ptr()
        ws = getattr(self, "_gm", None)
        if ws is None or ws["restart"] != restart:
            self._gm = None
            for key in [k for k in self._graphs if k[0] == "gmres"]:
                lib.mg_graph_destroy(self._graphs.pop(key)[0])
            ws = self._gm = self._gmres_workspace(restart, n, getattr(lev, "n_vec", n))
        G = ctypes.byref(ws["struct"])
        pp = None if params is None else ctypes.byref(params)
        sc = ws["scalars"]

        def read_r2():
            self._norm_host.copy_(sc[0:1], non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return float(np.sqrt(self._norm_host.item()))

        pkey = None if params is None else (params.smoother, params.nu_pre, params.nu_post, params.omega,
                                            params.zero_guess_skip, params.reverse_post, self._cheby_key)

        def iterate(j):
            key = ("gmres", j, pkey)
            g = self._graphs.get(key)
            if g is None:
                if self.smoother == "lexgs" and params is not None:      # cooperative launches are not captured
                    _lib.check(lib.mg_gmres_iterate(comm, self._level_structs, self.nlevels, pp, G, j, st),
                               "mg_gmres_iterate")
                    return
                cap = torch.cuda.Stream(device=self.device)
                cap.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(cap):
                    h = cap.cuda_stream
                    _lib.check(lib.mg_graph_begin(h), "mg_graph_begin")
                    rc = lib.mg_gmres_iterate(comm, self._level_structs, self.nlevels, pp, G, j, h)
                    out = ctypes.c_void_p()
                    rc2 = lib.mg_graph_end(h, ctypes.byref(out))
                    _lib.check(rc, "mg_gmres_iterate (capture)")
                    _lib.check(rc2, "mg_graph_end")
                torch.cuda.current_stream().wait_stream(cap)
                g = self._graphs[key] = (out, 0)
            _lib.check(lib.mg_graph_launch(g[0], st), "mg_graph_launch")

        t0 = time.perf_counter()
        self.set_rhs(rhs)
        x = ws["x"]
        if x0 is None:
            x.zero_()
        else:
            self._to_level0(x0, x)
        torch.cuda.current_stream().synchronize()
        t1 = time.perf_counter()
        its = 0
        track = []
        while True:
            _lib.check(lib.mg_gmres_start(comm, self._level_structs, G, st), "mg_gmres_start")    # true residual
            res = read_r2()
            if not track:
                track.append(res)
            if res <= error or its >= max_iterations:
                break
            k = 0
            while k < restart and its < max_iterations:
                iterate(k)
                its += 1
                k += 1
                est = read_r2()
                track.append(est)
                if est <= error:
                    break
            _lib.check(lib.mg_gmres_finish(self._level_structs, pp, G, k, st), "mg_gmres_finish")
        t2 = time.perf_counter()
        sol = self._from_level0(x, view)
        t3 = time.perf_counter()
        self.last_gmres_timing = {"transfer_in_s": t1 - t0, "iterations_s": t2 - t1, "orthogonalisation_s": None,
                                  "transfer_out_s": t3 - t2, "iterations": its}
        return sol, track, its, res

    def gmres_residual_vector(self):
        """b - A x of the last gmres solution, (n,1) natural order (this rank's block when partitioned: the halo of x
        is current, the last mg_gmres_start exchanged it)"""
        lev = self.levels[0]
        _lib.check(self.lib.mg_sell_residual(ctypes.byref(lev.A.struct), self._gm["x"].data_ptr(), lev.b.data_ptr(),
                                             lev.r.data_ptr(), _lib.stream_handle(self.torch)), "mg_sell_residual")
        return self._from_level0(lev.r)

    def _gmres_workspace(self, restart, n, n_vec):
        """device buffers of mg_gmres for one restart length; ValueError when the two bases do not fit"""
        torch, lib, dev = self.torch, self.lib, self.device
        ld = (n_vec + 31) // 32 * 32
        m = restart + 1
        parts = max(int(lib.mg_norm_workspace_size(n)), int(lib.mg_krylov_partials(n, m)))
        small = 4 * m + m * restart + 8 + parts + _lib.MG_MAX_RANKS * m
        need = 8 * (2 * m * ld + ld + small)
        free, _ = torch.cuda.mem_get_info(dev)
        free += torch.cuda.memory_reserved(dev) - torch.cuda.memory_allocated(dev)     # cached by torch, reusable
        if need > free:
            raise ValueError("GMRES(%d) needs %d bytes of device memory for its bases (2 x %d vectors of %d entries), "
                             "%d are free" % (restart, need, m, ld, free))
        f64 = dict(dtype=torch.float64, device=dev)
        ws = {"restart": restart, "x": torch.zeros(ld, **f64), "V": torch.zeros(m * ld, **f64),
              "Z": torch.zeros(m * ld, **f64), "H": torch.zeros(m * restart, **f64), "g": torch.zeros(m, **f64),
              "cs": torch.zeros(m, **f64), "sn": torch.zeros(m, **f64), "y": torch.zeros(m, **f64),
              "scalars": torch.zeros(8, **f64), "partials": torch.zeros(parts, **f64),
              "slots": torch.zeros(_lib.MG_MAX_RANKS * m, **f64)}
        ws["struct"] = _lib.mg_gmres(*(ws[k].data_ptr() for k in ("x", "V", "Z")), ld, restart, 0,
                                     *(ws[k].data_ptr() for k in ("H", "g", "cs", "sn", "y", "scalars", "partials",
                                                                  "slots")))
        return ws

    def __del__(self):
        try:
            for g, _ in self._graphs.values():
                self.lib.mg_graph_destroy(g)
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------------
    def cycle_bytes(self, nu_pre, nu_post):
        """Algorithmic bytes of one outer iteration (residual+norm, then one V(nu_pre,nu_post) cycle), exactly
        the formula of SURVEY.md 8(d), from the ACTUAL nnz of the built hierarchy."""
        S = algorithmic_bytes_csr
        lv = self.levels
        total = S(lv[0].nnz_A, lv[0].n) + 16 * lv[0].n
        per_level = []
        for l in range(self.nlevels - 1):
            n, nc = lv[l].n, lv[l + 1].n
            a, q = lv[l].nnz_A, lv[l].nnz_Q
            b = (nu_pre + nu_post + 1) * (S(a, n) + 24 * n)           # sweeps + in-cycle residual
            b += S(q, nc) + 8 * n + 8 * nc                            # restriction
            b += S(q, n) + 8 * nc + 16 * n                            # prolongation + correction
            per_level.append(b)
            total += b
        coarse = lv[-1].coarse_bytes + 16 * lv[-1].n
        total += coarse
        return {"total": total, "outer": S(lv[0].nnz_A, lv[0].n) + 16 * lv[0].n, "levels": per_level,
                "coarse": coarse}

    def cycle_bytes_moved(self, nu_pre, nu_post):
        """Bytes THIS GPU has to move per outer iteration (V-cycle + norm of its result) the way the cycle is actually
        run -- the model behind roofline.cycle.moved_frac in bench.py, next to the CSR yardstick of cycle_bytes():
        matrix streams as stored (values; columns, or 4 B of offset per slice and entry where columns are implied),
        every vector entry an operation reads or writes counted once per operation (gathers: the distinct entries,
        bounded by the rows read), and the passes the multicolour cycle leaves out (cycle.cu g_cycle_fusion)."""
        fusion = os.environ.get("MGB_CYCLE_FUSION", "1") != "0"
        total = 0.0
        lv = self.levels
        for l in range(self.nlevels - 1):
            L_ = lv[l]
            n = L_.n
            nc = getattr(lv[l + 1], "n", 0)
            SA, SQ, SQT = L_.A.stream_bytes(), L_.Q.stream_bytes(), L_.QT.stream_bytes()
            lenA = max(L_.A.max_len, 1)
            lenQ = max(L_.Q.max_len, 1)

            def rows_pass(R, write_vec, read_b=True):      # matrix share + b + output + distinct x entries gathered
                return SA * R / max(n, 1) + (8 * R if read_b else 0) + 8 * R * write_vec + 8 * min(n, lenA * R)
            mc = self.smoother == "mcgs" and L_.color_ptr is not None
            cheb = self.smoother == "chebyshev"
            fused = mc and fusion and int(getattr(L_, "flags", 0)) & 1
            skip_prolong = fused and int(getattr(L_, "flags", 0)) & 2 and nu_post > 0
            if cheb:
                # step k: matrix, b, x gathers, x_out, plus x_i and dinv_i, d written, and d read after step 0
                deg = self.cheby_degree
                sweep = deg * (rows_pass(n, 1) + 16 * n + 8 * n) + (deg - 1) * 8 * n
                last = first = 0
            elif mc:
                sizes = np.diff(np.asarray(L_.color_ptr, dtype=np.int64))
                sweep = sum(SA * c / max(n, 1) + 16 * c + 8 * min(n - c, (lenA - 1) * c) for c in sizes)
                last, first = int(sizes[-1]), int(sizes[0])
            else:
                sweep = rows_pass(n, 1) + (8 * n if self.smoother == "jacobi" else 0)
                last = first = 0
            b = (nu_pre + nu_post) * sweep
            if l > 0 and nu_pre > 0:
                if cheb:                                       # step 0 on zeros: dinv, b, d, x; no matrix
                    b += 32 * n - (rows_pass(n, 1) + 24 * n)
                elif mc and fusion and getattr(L_, "diag", None) is not None:
                    b += 8 * n + 16 * first - (SA * first / max(n, 1) + 16 * first + 8 * min(n - first, (lenA - 1) * first))
                else:
                    b += 8 * n                                 # zero fill
            r_rows = n - last if (fused and nu_pre > 0) else n
            b += rows_pass(r_rows, 1) + (8 * last if (fused and nu_pre > 0) else 0)         # residual
            b += SQT + 8 * nc + 8 * n                                                      # restriction
            p_rows = n - first if skip_prolong else n
            b += SQ * p_rows / max(n, 1) + 16 * p_rows + 8 * min(nc, lenQ * p_rows)        # prolongation
            if l == 0:                                                                     # norm of the new iterate
                nr = n - last if (fused and nu_post > 0) else n
                b += rows_pass(nr, 0)
            total += b
        total += lv[-1].coarse_bytes + 16 * lv[-1].n
        return {"total": total, "model": "bytes this GPU streams per step as run: stored matrix bytes (implied columns "
                                         "counted as 4 B per slice and entry), vector entries once per operation, "
                                         "skipped passes left out"}

    def level_matrix(self, l):
        """A_l in natural ordering as a SciPy CSR (for pattern / value parity checks)."""
        if self.host_A is not None and self.host_A[l] is not None:
            return self.host_A[l]
        return SD.download_level_matrix(self, l)
