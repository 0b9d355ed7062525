"""Classical algebraic multigrid setup on the device (csrc/amg_kernels.cu): transfer operators from the matrix alone.

Per level, on the level operator A (canonical CSR, fp64, device memory):
  strength     S_i = {j != i : -a_ij > 0 and -a_ij >= theta * max_{k != i}(-a_ik)}   (S as CSR with the values a_ij,
               S^T by the setup transpose)
  split        PMIS (De Sterck, Yang, Heys 2006) with the deterministic weights w_i = |S^T_i| + r_i, r_i the integer hash
               of the global row index in [0, 1) (formats.chebyshev_start_vector + 0.5), ties broken by the index;
               then one promotion pass (an F point with a non-empty S_i and no C point in it becomes C)
  interpolate  C points numbered in ascending fine index; direct interpolation with positive couplings lumped into the
               diagonal: Q[i, cmap[j]] = -(sn_all / sn_str) / (a_ii + sp_all) * a_ij for j in S_i n C
  A_c = Q^T A Q by the setup's Galerkin product, and the next level.
Q is the prolongation and Q^T the restriction, as for every other transfer operator of the engine.  Everything stays
in device memory; the host reads one flag per PMIS round.  tests/amg_oracle.py restates the definition in NumPy and
the GPU tests hold the two to the same bits.  DESIGN.md §4.10 has the definition, the kernels and measurements.
"""
import ctypes
import time

import numpy as np

from . import _lib
from . import formats as F
from . import setup_device as SD

C_POINT, F_POINT = 1, 2


def check_theta(theta):
    theta = float(theta)
    if not 0.0 <= theta < 1.0:
        raise ValueError("the strength threshold theta must be in [0, 1), got %r" % (theta,))
    return theta


def pmis_weights_host(st_counts):
    """w_i = |S^T_i| + r_i on the host (NumPy): the weights the device builder forms with torch"""
    n = len(st_counts)
    return np.asarray(st_counts, dtype=np.float64) + (F.chebyshev_start_vector(np.arange(n, dtype=np.int64)) + 0.5)


def complexities(rows, nnz):
    """(grid complexity sum n_l / n_0, operator complexity sum nnz_l / nnz_0)"""
    return float(sum(rows)) / rows[0], float(sum(nnz)) / nnz[0]


class AmgBuilder:
    """device kernels of the classical AMG setup, one method per step"""

    def __init__(self, torch=None, device=None):
        self.torch = torch = _lib.require_cuda() if torch is None else torch
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else device
        self.lib = _lib.load()
        self.S = SD.DeviceSetup(torch, self.dev)
        self.stats = []
        self.trace = []

    def st(self):
        return _lib.stream_handle(self.torch)

    def upload(self, A):
        return self.S.upload(A)

    def download(self, M):
        return self.S.download(M)

    # strength of connection: (S, S^T) as device CSR, values a_ij
    def strength(self, A, theta=0.25):
        theta = check_theta(theta)
        t, S = self.torch, self.S
        n = A.shape[0]
        count = S.empty(n, t.int32)
        _lib.check(self.lib.mg_amg_strength_count(n, *A.ptrs(), theta, count.data_ptr(), self.st()),
                   "mg_amg_strength_count")
        sptr, nnz = S.scan(count, n)
        sidx, sval = S.empty(nnz, t.int32), S.empty(nnz, t.float64)
        _lib.check(self.lib.mg_amg_strength_fill(n, *A.ptrs(), theta, sptr.data_ptr(), sidx.data_ptr(),
                                                 sval.data_ptr(), self.st()), "mg_amg_strength_fill")
        Sm = SD.DevCSR((n, n), sptr, sidx, sval)
        return Sm, S.transpose(Sm)

    def weights(self, ST):
        """w_i = |S^T_i| + r_i (float64 device tensor); the same operations as pmis_weights_host"""
        t = self.torch
        n = ST.shape[0]
        cnt = (ST.indptr[1:] - ST.indptr[:-1]).to(t.float64)
        return cnt + (F.chebyshev_start_vector(t.arange(n, dtype=t.int64, device=self.dev)) + 0.5)

    # PMIS + promotion: final C/F states (int32, 1 = C, 2 = F); the states before promotion, the number of rounds and
    # of promoted points are left in last_pmis_state, last_rounds, last_promoted
    def split(self, S, ST):
        t, D = self.torch, self.S
        n = S.shape[0]
        w = self.weights(ST)
        state = D.empty(n, t.int32)
        work = D.empty(n + 1, t.int32)
        rounds = self.lib.mg_amg_pmis(n, S.indptr.data_ptr(), S.indices.data_ptr(), ST.indptr.data_ptr(),
                                      ST.indices.data_ptr(), w.data_ptr(), state.data_ptr(), work.data_ptr(), self.st())
        if rounds < 0:
            _lib.check(rounds, "mg_amg_pmis")
        final = D.empty(n, t.int32)
        promoted = self.lib.mg_amg_promote(n, S.indptr.data_ptr(), S.indices.data_ptr(), state.data_ptr(),
                                           final.data_ptr(), work.data_ptr(), self.st())
        if promoted < 0:
            _lib.check(promoted, "mg_amg_promote")
        self.last_pmis_state = state
        self.last_rounds = int(rounds)
        self.last_promoted = int(promoted)
        return final

    # coarse numbering + direct interpolation: (Q as device CSR n x n_c, cmap)
    def interpolate(self, A, S, state):
        t, D = self.torch, self.S
        n = A.shape[0]
        scan, nc = D.scan((state == C_POINT).to(t.int32), n)
        cmap, clist = D.empty(n, t.int32), D.empty(nc, t.int32)
        _lib.check(self.lib.mg_nn_compact(n, state.data_ptr(), scan.data_ptr(), cmap.data_ptr(), clist.data_ptr(),
                                          self.st()), "mg_nn_compact")
        count = D.empty(n, t.int32)
        _lib.check(self.lib.mg_amg_interp_count(n, S.indptr.data_ptr(), S.indices.data_ptr(), state.data_ptr(),
                                                count.data_ptr(), self.st()), "mg_amg_interp_count")
        qptr, nnz = D.scan(count, n)
        qidx, qval = D.empty(nnz, t.int32), D.empty(nnz, t.float64)
        work = D.empty(1, t.int32)
        bad = ctypes.c_int64(-1)
        _lib.check(self.lib.mg_amg_interp_fill(n, *A.ptrs(), *S.ptrs(), state.data_ptr(), cmap.data_ptr(),
                                               qptr.data_ptr(), qidx.data_ptr(), qval.data_ptr(), work.data_ptr(),
                                               ctypes.byref(bad), self.st()), "mg_amg_interp_fill")
        return SD.DevCSR((n, nc), qptr, qidx, qval), cmap

    def define_hierarchy(self, A, levels, theta=0.25, keep_intermediates=False):
        """A: SciPy matrix (taken as canonical CSR) or DevCSR.  Returns [Q_0, ..., Q_{levels-2}] as device CSR.
        self.stats: one dict per level (the coarsest included) with rows, nnz and, for every level that is coarsened,
        C points, PMIS rounds, promoted points and the setup split in ms; self.complexities(): grid and operator
        complexity.  Raises ValueError if a level cannot be coarsened (no C point, or every point C)."""
        theta = check_theta(theta)
        if levels < 2:
            raise ValueError("levels must be >= 2")
        Al = A if isinstance(A, SD.DevCSR) else self.upload(A)
        Qs, self.stats, self.trace = [], [], []
        clock, mark = time.perf_counter, self.mark
        for l in range(levels - 1):
            n = Al.shape[0]
            t0 = clock()
            S, ST = self.strength(Al, theta)
            t0, ms_s = mark(t0)
            state = self.split(S, ST)
            t0, ms_p = mark(t0)
            nc = int((state == C_POINT).sum().item())
            if nc == 0 or nc == n:
                raise ValueError("AMG coarsening of level %d (%d rows) %s; no transfer operator is built for it"
                                 % (l, n, "selects no C point" if nc == 0 else "keeps every point as a C point"))
            t0 = clock()
            Q, cmap = self.interpolate(Al, S, state)
            t0, ms_i = mark(t0)
            Ac = self.S.galerkin(Al, Q, self.S.transpose(Q))
            t0, ms_g = mark(t0)
            self.stats.append({"level": l, "rows": n, "nnz": Al.nnz, "c_points": nc, "pmis_rounds": self.last_rounds,
                               "promoted": self.last_promoted, "strong_nnz": S.nnz, "nnz_Q": Q.nnz,
                               "strength_ms": ms_s, "pmis_ms": ms_p, "interpolation_ms": ms_i, "galerkin_ms": ms_g})
            if keep_intermediates:
                self.trace.append({"A": Al, "S": S, "ST": ST, "pmis_state": self.last_pmis_state, "state": state,
                                   "cmap": cmap, "Q": Q})
            Qs.append(Q)
            Al = Ac
        self.stats.append({"level": levels - 1, "rows": Al.shape[0], "nnz": Al.nnz})
        if keep_intermediates:
            self.trace.append({"A": Al})
        return Qs

    def mark(self, t0):
        """(now, ms since t0) after the device has finished the work enqueued so far: the setup split's clock"""
        self.torch.cuda.synchronize()
        now = time.perf_counter()
        return now, round((now - t0) * 1e3, 3)

    def complexities(self, levels=None):
        st = self.stats[:levels]
        return complexities([s["rows"] for s in st], [s["nnz"] for s in st])
