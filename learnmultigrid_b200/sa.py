"""Smoothed aggregation setup on the device (csrc/sa_kernels.cu): transfer operators from the matrix alone.

Per level, on the level operator A (canonical CSR, fp64, device memory) and the near-null-space vector B (B = 1 on the
fine level):
  strength   S_i = {j != i : a_ij != 0 and a_ij * a_ij >= theta^2 * (|a_ii| * |a_jj|)}   (S as CSR with the values
             a_ij, S^T by the setup transpose); N_i = S_i u S^T_i, a point with an empty N_i is isolated
  MIS(2)     the tuple algorithm of Bell, Dalton and Olson (2012) on keys (state, r_i, i), r_i the integer hash of the
             row index (formats.chebyshev_start_vector + 0.5); isolated points start OUT
  aggregate  roots (IN points) numbered in ascending fine index; pass 1 joins a point to the root among its neighbours,
             pass 2 a point still unassigned to the aggregate of its pass-1 neighbour of largest (r_j, j)
  tentative  nu_a = sqrt(sum_{i in a} B_i * B_i), T[i, agg(i)] = B_i / nu_agg(i); the next level's B is nu
  smooth     P = (I - (omega / lambda_max) D^-1 A) T, lambda_max the device Lanczos estimate of lambda_max(D^-1 A)
             (setup_device.chebyshev_lambda_max), the product by the setup's SpGEMM
  A_c = P^T A P by the setup's Galerkin product, and the next level.
Isolated points are never aggregated (their T rows are empty): they are left to the smoother.  Everything stays in
device memory; the host reads one flag per MIS(2) round.  tests/sa_oracle.py restates the definition in NumPy and the
GPU tests hold the two to the same bits.  DESIGN.md §4.11 has the definition, the kernels and measurements.
"""
import ctypes
import time

from . import _lib
from . import setup_device as SD
from .amg import AmgBuilder, check_theta

MIS_OUT, MIS_UNDECIDED, MIS_IN = 0, 1, 2


def check_omega(omega):
    omega = float(omega)
    if not 0.0 < omega < 2.0:
        raise ValueError("the prolongation smoothing weight omega must be in (0, 2), got %r" % (omega,))
    return omega


class SaBuilder(AmgBuilder):
    """device kernels of the smoothed aggregation setup, one method per step (upload, download, the setup clock and the
    complexities are AmgBuilder's)"""

    def diagonal(self, A):
        d = self.S.empty(A.shape[0], self.torch.float64)
        _lib.check(self.lib.mg_sa_diagonal(A.shape[0], *A.ptrs(), d.data_ptr(), self.st()), "mg_sa_diagonal")
        return d

    # symmetric strength of connection: (S, S^T) as device CSR, values a_ij; diag from diagonal()
    def strength(self, A, theta=0.0, diag=None):
        theta = check_theta(theta)
        t, D = self.torch, self.S
        n = A.shape[0]
        diag = self.diagonal(A) if diag is None else diag
        count = D.empty(n, t.int32)
        _lib.check(self.lib.mg_sa_strength_count(n, *A.ptrs(), diag.data_ptr(), theta, count.data_ptr(), self.st()),
                   "mg_sa_strength_count")
        sptr, nnz = D.scan(count, n)
        sidx, sval = D.empty(nnz, t.int32), D.empty(nnz, t.float64)
        _lib.check(self.lib.mg_sa_strength_fill(n, *A.ptrs(), diag.data_ptr(), theta, sptr.data_ptr(),
                                                sidx.data_ptr(), sval.data_ptr(), self.st()), "mg_sa_strength_fill")
        Sm = SD.DevCSR((n, n), sptr, sidx, sval)
        return Sm, D.transpose(Sm)

    # MIS(2): final states (int32, 0 = OUT, 1 = undecided, 2 = IN); the number of rounds is left in last_rounds
    def mis2(self, S, ST):
        t, D = self.torch, self.S
        n = S.shape[0]
        state = D.empty(n, t.int32)
        work = D.empty(n + 1, t.int32)
        keys = D.empty(2 * n, t.int64)
        rounds = self.lib.mg_sa_mis2(n, S.indptr.data_ptr(), S.indices.data_ptr(), ST.indptr.data_ptr(),
                                     ST.indices.data_ptr(), state.data_ptr(), work.data_ptr(), keys.data_ptr(),
                                     self.st())
        if rounds < 0:
            _lib.check(rounds, "mg_sa_mis2")
        self.last_rounds = int(rounds)
        return state

    # roots numbered in ascending fine index, then the two aggregation passes: (agg: aggregate per point, -1 for an
    # isolated point; number of aggregates).  A point with two roots among its neighbours or a non-isolated point left
    # unassigned raises MgError naming it
    def aggregate(self, S, ST, state):
        t, D = self.torch, self.S
        n = S.shape[0]
        root = (state == MIS_IN).to(t.int32)
        scan, nc = D.scan(root, n)
        cmap, clist = D.empty(n, t.int32), D.empty(nc, t.int32)
        _lib.check(self.lib.mg_nn_compact(n, root.data_ptr(), scan.data_ptr(), cmap.data_ptr(), clist.data_ptr(),
                                          self.st()), "mg_nn_compact")
        agg, work = D.empty(n, t.int32), D.empty(n + 2, t.int32)
        bad = ctypes.c_int64(-1)
        _lib.check(self.lib.mg_sa_aggregate(n, S.indptr.data_ptr(), S.indices.data_ptr(), ST.indptr.data_ptr(),
                                            ST.indices.data_ptr(), state.data_ptr(), cmap.data_ptr(), agg.data_ptr(),
                                            work.data_ptr(), ctypes.byref(bad), self.st()), "mg_sa_aggregate")
        return agg, nc

    # tentative prolongator: (T as device CSR n x n_c, nu)
    def tentative(self, agg, nc, B):
        t, D = self.torch, self.S
        n = agg.numel()
        tptr, nnz = D.scan((agg >= 0).to(t.int32), n)
        tidx, tval = D.empty(nnz, t.int32), D.empty(nnz, t.float64)
        fill = self.lib.mg_sa_tentative_fill
        _lib.check(fill(n, agg.data_ptr(), tptr.data_ptr(), B.data_ptr(), None, tidx.data_ptr(), tval.data_ptr(),
                        self.st()), "mg_sa_tentative_fill")
        T = SD.DevCSR((n, nc), tptr, tidx, tval)
        TT = D.transpose(T)                        # members of every aggregate in ascending index, values B_i
        nu = D.empty(nc, t.float64)
        _lib.check(self.lib.mg_sa_aggregate_norm(nc, TT.indptr.data_ptr(), TT.values.data_ptr(), nu.data_ptr(),
                                                 self.st()), "mg_sa_aggregate_norm")
        _lib.check(fill(n, agg.data_ptr(), tptr.data_ptr(), B.data_ptr(), nu.data_ptr(), tidx.data_ptr(),
                        tval.data_ptr(), self.st()), "mg_sa_tentative_fill")
        return T, nu

    # prolongation smoothing: (P = At T, At = I - omega_hat D^-1 A on A's pattern, lambda_max, omega_hat)
    def smooth(self, A, T, omega=4.0 / 3.0, diag=None):
        omega = check_omega(omega)
        t = self.torch
        diag = self.diagonal(A) if diag is None else diag
        bad = t.nonzero(diag <= 0.0)
        if bad.numel():
            raise ValueError("smoothed aggregation needs a positive diagonal; a_ii = %r in row %d"
                             % (float(diag[bad[0, 0]].item()), int(bad[0, 0].item())))
        lam = SD.chebyshev_lambda_max(self.S, A)
        omega_hat = omega / lam
        vals = self.S.empty(A.nnz, t.float64)
        _lib.check(self.lib.mg_sa_smooth_scale(A.shape[0], *A.ptrs(), diag.data_ptr(), omega_hat, vals.data_ptr(),
                                               self.st()), "mg_sa_smooth_scale")
        At = SD.DevCSR(A.shape, A.indptr, A.indices, vals)
        return self.S.spgemm(At, T), At, lam, omega_hat

    def define_hierarchy(self, A, levels, theta=0.0, omega=4.0 / 3.0, keep_intermediates=False):
        """A: SciPy matrix (taken as canonical CSR) or DevCSR.  Returns [P_0, ..., P_{levels-2}] as device CSR.
        self.stats: one dict per level (the coarsest included) with rows, nnz and, for every level that is coarsened,
        aggregates, MIS(2) rounds, isolated points, nnz_Q, lambda_max, omega_eff and the setup split in ms;
        self.complexities(): grid and operator complexity.  Raises ValueError if a level cannot be coarsened (no
        aggregate, or one aggregate per point) or has a non-positive diagonal."""
        theta, omega = check_theta(theta), check_omega(omega)
        if levels < 2:
            raise ValueError("levels must be >= 2")
        t = self.torch
        Al = A if isinstance(A, SD.DevCSR) else self.upload(A)
        B = t.ones(Al.shape[0], dtype=t.float64, device=self.dev)
        Ps, self.stats, self.trace = [], [], []
        clock, mark = time.perf_counter, self.mark
        for l in range(levels - 1):
            n = Al.shape[0]
            t0 = clock()
            diag = self.diagonal(Al)
            S, ST = self.strength(Al, theta, diag)
            t0, ms_s = mark(t0)
            state = self.mis2(S, ST)
            t0, ms_m = mark(t0)
            nc = int((state == MIS_IN).sum().item())
            if nc == 0 or nc == n:
                raise ValueError("smoothed aggregation of level %d (%d rows) %s; no transfer operator is built for it"
                                 % (l, n, "finds no aggregate" if nc == 0 else "keeps every point as an aggregate"))
            agg, _ = self.aggregate(S, ST, state)
            T, nu = self.tentative(agg, nc, B)
            t0, ms_a = mark(t0)
            try:
                P, At, lam, omega_hat = self.smooth(Al, T, omega, diag)
            except ValueError as e:
                raise ValueError("level %d: %s" % (l, e)) from None
            t0, ms_p = mark(t0)
            Ac = self.S.galerkin(Al, P, self.S.transpose(P))
            t0, ms_g = mark(t0)
            isolated = int(((S.indptr[1:] == S.indptr[:-1]) & (ST.indptr[1:] == ST.indptr[:-1])).sum().item())
            self.stats.append({"level": l, "rows": n, "nnz": Al.nnz, "aggregates": nc, "mis2_rounds": self.last_rounds,
                               "isolated": isolated, "strong_nnz": S.nnz, "nnz_Q": P.nnz, "lambda_max": lam,
                               "omega_eff": omega_hat, "strength_ms": ms_s, "mis2_ms": ms_m, "aggregation_ms": ms_a,
                               "smoothing_ms": ms_p, "galerkin_ms": ms_g})
            if keep_intermediates:
                self.trace.append({"A": Al, "S": S, "ST": ST, "state": state, "agg": agg, "nu": nu, "T": T, "At": At,
                                   "P": P})
            Ps.append(P)
            Al, B = Ac, nu
        self.stats.append({"level": levels - 1, "rows": Al.shape[0], "nnz": Al.nnz})
        if keep_intermediates:
            self.trace.append({"A": Al})
        return Ps
