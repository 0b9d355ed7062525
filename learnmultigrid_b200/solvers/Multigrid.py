"""Multigrid drivers with the reference's interface (learn_multigrid/solvers/Multigrid.py) on the B200 engine.

    Multigrid(matrix, rhs)                    Multigrid.py:26-161
    GeometricMG(matrix, rhs)                  Multigrid.py:164-173
    SemiGeometricMG(matrix, rhs, l2_proj)     Multigrid.py:176-197
    AlgebraicMG(matrix, rhs, theta=0.25)      extension: classical AMG transfer operators built from the matrix
    SmoothedAggregationMG(matrix, rhs, theta=0.0, omega=4/3)
                                              extension: smoothed aggregation transfer operators built from the matrix

`solve()` keeps the reference's outer loop statement by statement (Multigrid.py:36-75): residual, 2-norm,
the first-iteration sqrt(n) quirk (:64-66), history, ABSOLUTE tolerance test, one V-cycle.  The V-cycle itself
(:77-124) runs on the device from a hierarchy that is built ONCE (the reference rebuilds Q^T A Q and refactorises
the coarsest operator in every cycle, :97-98,106).

Differences, all explicit:
  * `smoother` is honoured.  The committed reference ignores it and always calls PyAMG's index-order
    Gauss-Seidel (:88,121).  Here "GaussSeidel" selects multicolour Gauss-Seidel (`gs_order="multicolor"`,
    default) or the exact index-order sweep (`gs_order="lexicographic"`, bit-for-bit the reference's smoother);
    "Jacobi" selects damped Jacobi with `omega` (Jacobi.py:35 is omega=1, which does not smooth; default 2/3).
    "Chebyshev" (extension) selects the Chebyshev polynomial smoother in D^-1 A: `cheby_degree` steps per sweep
    (default 2) over [0.3, 1.1] x a Lanczos estimate of lambda_max(D^-1 A) per level, or over `cheby_bounds`
    (one (lo, hi) pair per smoothing level).  It needs no colouring and is symmetric, so it also preconditions CG.
  * `l2_proj` may be a list [Q_0, Q_1, ...] giving a transfer operator for every level.  Levels without one
    use the reference's 1D linear interpolator (Multigrid.interpolator, :126-147), as the reference does
    below the first level (:188-197).
  * `initial_guess` is copied to the device, not mutated in place.
"""
import sys

import numpy as np
import scipy.sparse as sp
from scipy.sparse import csr_matrix

from .. import _lib
from .. import formats as F
from ..engine import DeviceHierarchy
from .Solver import IterativeSolver
from .Jacobi import Jacobi
from .CG import CG
from .GaussSeidel import GaussSeidel


class Multigrid(IterativeSolver):

    def __init__(self, matrix, rhs):
        super().__init__(matrix, rhs)
        self.label = "Multigrid"
        self._hier = None
        self._hier_key = None
        self._interp_cache = {}
        self.verbose = False
        self.setup = "device"
        self.fabric = None           # set by distribute(): run the V-cycle row-partitioned over several GPUs
        self.dist_options = {}

    def distribute(self, fabric=None, **options):
        """Row-partition the fine levels over the ranks of `fabric` (default: the torch.distributed world, one
        process per GPU) -- no reference counterpart, see learnmultigrid_b200/distributed.py.  Every rank must
        construct the solver with the same global (matrix, rhs, transfers) and make the same calls."""
        if fabric is None:
            from ..distributed import TorchFabric
            fabric = TorchFabric()
        self.fabric = fabric
        self.dist_options = dict(options)
        self._hier = None
        return self

    # ------------------------------------------------------------------------------------------------
    def solve(self, levels=2, smoother="Jacobi", smooth_steps=1, max_iterations=100, error=1e-08,
              initial_guess=None, cycle="V", first_call=False, *, omega=2.0 / 3.0, gs_order="multicolor",
              colors=None, use_graph=True, cheby_degree=2, cheby_bounds=None):
        if initial_guess is None:
            self.solution = np.zeros(shape=(self.get_dimension(), 1))
        else:
            self.solution = initial_guess
        cycle_method = self.cycle_to_method(cycle)
        if not callable(cycle_method):
            print("Cycle type unknown, exit...")
            sys.exit(0)                                            # Multigrid.py:55-57
        h = self._hierarchy(levels, smoother, gs_order, colors, first_call,
                            **self._cheby_kw(smoother, cheby_degree, cheby_bounds))
        params = h.make_params(nu_pre=smooth_steps, nu_post=smooth_steps, omega=omega)
        h.set_rhs(self.rhs)
        if initial_guess is None:
            h.zero_x()
        else:
            h.set_x(self.solution)
        track_res = np.ndarray(shape=(0, 1), dtype=float)
        # :62-63 residual + norm.  Only the first one is a pass of its own: every cycle that is followed by another
        # iteration also leaves the norm of its new iterate (the last colour sweep sums its rows' share from
        # registers, engine.vcycle(with_norm=True) / mg_vcycle_norm)
        res = h.residual_norm() if max_iterations > 0 else None
        for it in range(0, max_iterations):
            self.iterations += 1
            self.residual = res
            if self.iterations <= 1:                               # :64-66
                self.residual = float(np.sqrt(float(self.get_dimension())))
                self._residual_is_ones = True
            else:
                self._residual_is_ones = False
            track_res = np.vstack((track_res, self.residual))
            if self.verbose:
                print("It: ", self.iterations, self.residual)
            if self.residual <= error:
                break
            more = it + 1 < max_iterations
            if self.fabric is not None and hasattr(h, "comm"):
                h.vcycle(params, use_graph=use_graph, norm_after=more)             # :73
            else:
                h.vcycle(params, use_graph=use_graph, with_norm=more)              # :73
            if more:
                res = h.last_norm()
        if self.fabric is not None and hasattr(h, "check"):
            h.check()          # an exchange site that timed out leaves a wrong iterate behind: raise, do not return it
        if self.fabric is not None and getattr(self, "local_solution", False) and hasattr(h, "get_x_local"):
            self.solution = h.get_x_local(view=getattr(self, "pinned_io", False))     # this rank's row block only
        else:
            self.solution = h.get_x(view=getattr(self, "pinned_io", False))
        self.track_res = track_res
        self._residual_dirty = True

    def get_residual_vector(self):
        if getattr(self, "_residual_dirty", False) and self._hier is not None:
            if getattr(self, "_residual_is_ones", False):
                self.residual_vector = np.ones(shape=self.solution.shape)      # :65
            else:
                self.residual_vector = self._hier.residual_vector()
            self._residual_dirty = False
        return self.residual_vector

    # ------------------------------------------------------------------------------------------------
    def v_cycle(self, A, u0, rhs, smoother, smooth_steps, error, levels, first_call=False, *, omega=2.0 / 3.0,
                gs_order="multicolor", colors=None, cheby_degree=2, cheby_bounds=None):
        """One V-cycle for (A, rhs) starting from u0; returns the new iterate as an (n,1) array
        (Multigrid.py:77-124).  The hierarchy is cached as long as the same matrix object is passed."""
        if A is self.matrix:
            h = self._hierarchy(levels, smoother, gs_order, colors, first_call,
                                **self._cheby_kw(smoother, cheby_degree, cheby_bounds))
        else:
            h = self._build(A, levels, smoother, gs_order, colors, first_call,
                            **self._cheby_kw(smoother, cheby_degree, cheby_bounds))
        params = h.make_params(nu_pre=smooth_steps, nu_post=smooth_steps, omega=omega)
        h.set_rhs(rhs)
        h.set_x(u0)
        h.vcycle(params)
        return h.get_x()

    def interpolator(self, dimension, _):
        """Dense 1D linear interpolation, same values as Multigrid.py:126-147 (memoised per dimension)."""
        key = int(dimension)
        if key not in self._interp_cache:
            self._interp_cache[key] = F.geometric_interpolator_csr(key).toarray()
        return self._interp_cache[key]

    def smoother_to_method(self, smoother):
        switcher = {
            "GaussSeidel": GaussSeidel,
            "Jacobi": Jacobi,
            "CG": CG,
        }
        return switcher.get(smoother, "Invalid smoother")

    def cycle_to_method(self, cycle):
        switcher = {
            "V": self.v_cycle,
        }
        return switcher.get(cycle, "Invalid smoother")

    # ------------------------------------------------------------------------------------------------
    def _transfer_list(self, levels, first_call):
        """[Q_0 ... Q_{levels-2}] in CSR; geometric 1D interpolation where none is supplied."""
        given = self._given_transfers() if first_call else []
        qs = []
        n = self.matrix.shape[0]
        for l in range(levels - 1):
            if l < len(given):
                q = given[l] if hasattr(given[l], "ptrs") else F.canonical_csr(given[l])      # DevCSR: already on the device
            else:
                q = F.geometric_interpolator_csr(n)
            if q.shape[0] != n:
                raise ValueError("transfer operator %d has %d rows but the level has %d unknowns"
                                 % (l, q.shape[0], n))
            qs.append(q)
            n = q.shape[1]
        return qs

    def _given_transfers(self):
        return []

    @staticmethod
    def _cheby_kw(smoother, degree, bounds):
        """the Chebyshev options as keywords of _hierarchy / _build (none for the other smoothers)"""
        return {"cheby_degree": degree, "cheby_bounds": bounds} if smoother == "Chebyshev" else {}

    @staticmethod
    def _smoother_kind(smoother, gs_order):
        if smoother == "Jacobi":
            return "jacobi"
        if smoother == "Chebyshev":
            return "chebyshev"
        if smoother == "GaussSeidel":
            if gs_order == "multicolor":
                return "mcgs"
            if gs_order == "lexicographic":
                return "lexgs"
            raise ValueError("gs_order must be 'multicolor' or 'lexicographic'")
        # the reference fails with "'str' object is not callable" for an unknown name (Multigrid.py:79-80)
        raise TypeError("'str' object is not callable (unknown smoother %r)" % (smoother,))

    def _build(self, A, levels, smoother, gs_order, colors, first_call, cheby_degree=2, cheby_bounds=None):
        if levels < 2:
            raise ValueError("levels must be >= 2 (the reference recurses without bound for levels=1, "
                             "Multigrid.py:78,102)")
        kind = self._smoother_kind(smoother, gs_order)
        cheby = {}
        if kind == "chebyshev":
            F.chebyshev_check(cheby_degree, cheby_bounds)
            cheby = {"cheby_degree": cheby_degree, "cheby_bounds": cheby_bounds}
        save = self.matrix
        try:
            self.matrix = A
            qs = self._transfer_list(levels, first_call)
        finally:
            self.matrix = save
        # the hierarchy re-derives CSR from what the Solver holds (csc_matrix(matrix), Solver.py:18); when the caller's
        # own object is canonical CSR that round trip is the identity and is skipped (seconds at 10^8 entries)
        src = getattr(self, "_matrix_src", None)
        if (A is save and src is not None and sp.isspmatrix_csr(src) and src.dtype == np.float64
                and src.has_canonical_format):
            A = src
        if self.fabric is not None and self.fabric.world > 1:
            from ..distributed import DistributedHierarchy
            return DistributedHierarchy(A, qs, self.fabric, smoother=kind, colors=colors, **cheby, **self.dist_options)
        return DeviceHierarchy(A, qs, smoother=kind, colors=colors, setup=self.setup, **cheby)

    def _hierarchy(self, levels, smoother, gs_order, colors, first_call, cheby_degree=2, cheby_bounds=None):
        cb = None if cheby_bounds is None else tuple(tuple(float(v) for v in b) for b in cheby_bounds)
        key = (levels, smoother, gs_order, bool(first_call), id(self.matrix), None if colors is None else id(colors),
               cheby_degree if smoother == "Chebyshev" else None, cb if smoother == "Chebyshev" else None)
        if self._hier is None or self._hier_key != key:
            self._hier = self._build(self.matrix, levels, smoother, gs_order, colors, first_call,
                                     **self._cheby_kw(smoother, cheby_degree, cheby_bounds))
            self._hier_key = key
        return self._hier

    def get_hierarchy(self):
        """The device hierarchy of the last solve (level matrices, colourings, byte counts)."""
        return self._hier

    def as_preconditioner(self, levels=2, smoother="GaussSeidel", smooth_steps=1, omega=2.0 / 3.0,
                          gs_order="multicolor", first_call=True, symmetric=True, colors=None, cheby_degree=2,
                          cheby_bounds=None):
        """z = M^-1 r by one V-cycle from a zero guess, on natural-order device vectors (for solvers.CG).
        symmetric=True runs the multicolour post-smoothing in reverse colour order, so that M is symmetric for a
        symmetric A (Galerkin coarse operators, restriction = Q^T); damped Jacobi and the Chebyshev polynomial are
        symmetric as they are."""
        h = self._hierarchy(levels, smoother, gs_order, colors, first_call,
                            **self._cheby_kw(smoother, cheby_degree, cheby_bounds))
        params = h.make_params(nu_pre=smooth_steps, nu_post=smooth_steps, omega=omega,
                               reverse_post=bool(symmetric) and smoother == "GaussSeidel")
        lib, torch = h.lib, h.torch
        lev = h.levels[0]

        def apply(r, z):
            st = _lib.stream_handle(torch)
            if lev.perm is None:
                lev.b.copy_(r)
            else:
                _lib.check(lib.mg_gather(h.n, lev.perm.data_ptr(), r.data_ptr(), lev.b.data_ptr(), st), "mg_gather")
            lev.x.zero_()
            h.vcycle(params)
            if lev.perm is None:
                z.copy_(lev.x)
            else:
                _lib.check(lib.mg_scatter(h.n, lev.perm.data_ptr(), lev.x.data_ptr(), z.data_ptr(), st), "mg_scatter")
        apply.hierarchy = h            # solvers.CG runs the whole iteration inside the hierarchy when it sees these
        apply.params = params
        apply.matrix = self.matrix
        apply.matrix_src = getattr(self, "_matrix_src", None)
        return apply


class GeometricMG(Multigrid):

    def __init__(self, matrix, rhs):
        super().__init__(matrix, rhs)
        self.label = "GeometricMG"

    def interpolator(self, dimension, _):
        return super().interpolator(dimension, _)


class SemiGeometricMG(Multigrid):

    def __init__(self, matrix, rhs, l2_proj):
        super().__init__(matrix, rhs)
        self.label = "SemiGeometricMG"
        if isinstance(l2_proj, (list, tuple)):
            # one operator per level (extension); operators already on the device (DevCSR) stay there
            self.l_hierarchy = [q if hasattr(q, "ptrs") else csr_matrix(q) for q in l2_proj]
        else:
            self.l_hierarchy = [csr_matrix(l2_proj)]               # Multigrid.py:182
        self.l2_proj = self.l_hierarchy[0]

    def solve(self, levels=2, smoother="Jacobi", smooth_steps=1, max_iterations=100, error=1e-08,
              initial_guess=None, cycle="V", first_call=True, **kw):
        super().solve(levels, smoother, smooth_steps, max_iterations, error, initial_guess, cycle, first_call, **kw)

    def interpolator(self, dimension, first_call):
        if first_call:
            return self.l2_proj
        return super().interpolator(dimension, first_call)

    def _given_transfers(self):
        return self.l_hierarchy


class AlgebraicMG(Multigrid):
    """AlgebraicMG(matrix, rhs, theta=0.25) -- classical AMG (extension; no reference counterpart in the engine): the
    transfer operators come from the matrix alone, built on the device by learnmultigrid_b200/amg.py (strength of
    connection on negative couplings with threshold `theta`, PMIS C/F splitting, direct interpolation), one level at a
    time.  This is the multigrid the reference's 2D scripts compare against with PyAMG's ruge_stuben_solver; the
    splitting is PMIS, not Ruge-Stueben's serial first pass, so the coarse grids differ from PyAMG's.

    The operators are built on demand for the matrix a hierarchy is built for (solve, v_cycle, as_preconditioner,
    distribute) and cached by matrix object; the operators for fewer levels are a prefix of those for more levels.
    `define_hierarchy(levels)` builds them explicitly, `l_hierarchy` holds them (device CSR) and `amg_stats` their
    per-level statistics and complexities.  A level that cannot be coarsened raises ValueError."""

    def __init__(self, matrix, rhs, theta=0.25):
        super().__init__(matrix, rhs)
        from ..amg import check_theta
        self.label = "AlgebraicMG"
        self.theta = check_theta(theta)
        self.l_hierarchy = []
        self.amg_stats = None
        self._amg_cache = {}            # "own" / "other" -> (matrix object, [Q_0, ...], per-level stats)
        self._builder = None

    def _ab(self):
        if self._builder is None:
            from ..amg import AmgBuilder
            self._builder = AmgBuilder()
        return self._builder

    def _define_transfers(self, source, levels):
        """the builder's transfer operators for `source` and the parameters amg_stats reports with them"""
        return self._ab().define_hierarchy(source, levels, self.theta), {"theta": self.theta}

    def _amg_source(self, A):
        """the level-0 operator as the hierarchy will hold it (the caller's canonical CSR, or CSR of the stored CSC)"""
        if hasattr(A, "ptrs"):
            return A
        src = getattr(self, "_matrix_src", None)
        if (A is self._own_matrix() and src is not None and sp.isspmatrix_csr(src) and src.dtype == np.float64
                and src.has_canonical_format):
            return F.canonical_csr(src)
        return F.solver_csr(A)

    def _own_matrix(self):
        return getattr(self, "_solver_matrix", self.matrix)

    def _amg_transfers(self, A, levels):
        """[Q_0 ... Q_{levels-2}] for operator A, from the cache or built.  The cache holds the operators of the solver's
        own matrix and of the last other operator a V-cycle was asked for (v_cycle(A, ...)), each with the matrix
        object it was built for; l_hierarchy and amg_stats always describe the solver's own matrix."""
        from ..amg import complexities
        if levels < 2:
            raise ValueError("levels must be >= 2")
        own = A is self._own_matrix()
        slot = "own" if own else "other"
        c = self._amg_cache.get(slot)
        if c is None or c[0] is not A or len(c[1]) < levels - 1:
            qs, head = self._define_transfers(self._amg_source(A), levels)
            c = self._amg_cache[slot] = (A, qs, [dict(s) for s in self._ab().stats], head)
        qs = list(c[1][:levels - 1])
        if own:
            stats = [dict(s) for s in c[2][:levels]]
            stats[-1] = {"level": levels - 1, "rows": stats[-1]["rows"], "nnz": stats[-1]["nnz"]}
            gc, oc = complexities([s["rows"] for s in stats], [s["nnz"] for s in stats])
            self.amg_stats = dict(c[3], levels=stats, grid_complexity=gc, operator_complexity=oc)
            self.l_hierarchy = qs
        return qs

    def define_hierarchy(self, levels=2):
        return self._amg_transfers(self.matrix, levels)

    def _transfer_list(self, levels, first_call):
        return self._amg_transfers(self.matrix, levels)

    def _build(self, A, levels, smoother, gs_order, colors, first_call, **kw):
        self._solver_matrix = self.matrix           # _build swaps self.matrix for the operator it is given
        try:
            return super()._build(A, levels, smoother, gs_order, colors, first_call, **kw)
        finally:
            del self._solver_matrix


class SmoothedAggregationMG(AlgebraicMG):
    """SmoothedAggregationMG(matrix, rhs, theta=0.0, omega=4/3) -- smoothed aggregation AMG (extension): the transfer
    operators come from the matrix alone, built on the device by learnmultigrid_b200/sa.py (symmetric strength of
    connection with threshold `theta`, MIS(2) aggregation, the tentative prolongator of the constant vector and one
    Jacobi smoothing step with weight `omega / lambda_max(D^-1 A)`), one level at a time.  This is the solver PyAMG calls
    smoothed_aggregation_solver; the aggregation is parallel (MIS(2)), not PyAMG's serial standard aggregation, so the
    aggregates differ from PyAMG's.

    Caching, the prefix property, l_hierarchy, amg_stats (which also carries omega) and every smoother, PCG and
    distribute() work as for AlgebraicMG.  A level that cannot be coarsened, or has a non-positive diagonal, raises
    ValueError."""

    def __init__(self, matrix, rhs, theta=0.0, omega=4.0 / 3.0):
        super().__init__(matrix, rhs, theta)
        from ..sa import check_omega
        self.label = "SmoothedAggregationMG"
        self.omega = check_omega(omega)

    def _ab(self):
        if self._builder is None:
            from ..sa import SaBuilder
            self._builder = SaBuilder()
        return self._builder

    def _define_transfers(self, source, levels):
        return (self._ab().define_hierarchy(source, levels, self.theta, self.omega),
                {"theta": self.theta, "omega": self.omega})


class NeuralMG(Multigrid):
    """NeuralMG(matrix, rhs, model, M, std, mean) -- the 1D NN multigrid of Multigrid.py:200-370.

    `transfer_op(M)` builds the transfer operator of one level from its mass matrix exactly as the reference does:
    seven mass entries per interior coarse node (`prepare_nn_input`, :313-334), `model.predict` on the normalised
    features, `construct_B` (:336-370: entries [2], [4:7], [8] of each prediction, boundary rows from the
    partition-of-unity constraint rowsum(B) = rowsum(M)), Q = B / rowsum(B).  The reference re-predicts Q and
    recomputes Q^T A Q, Q^T M Q on every level of every cycle (:262-275); here the hierarchy is built once per solve
    and the V-cycle (:246-301, the same statement order as Multigrid.v_cycle) runs on the device.  The reference's
    smoother is PyAMG's index-order Gauss-Seidel whatever `smoother` says (:257,299): pass gs_order="lexicographic"
    to reproduce its histories, the default is multicolour Gauss-Seidel / damped Jacobi as for the other classes."""

    def __init__(self, matrix, rhs, model, M, std, mean):
        super().__init__(matrix, rhs)
        self.label = "NeuralMG"
        self.model = model
        self.M = M
        self.std = std
        self.mean = mean
        self.l_hierarchy = []

    @staticmethod
    def _dense(M):
        return np.asarray(M.todense() if sp.issparse(M) else M, dtype=np.float64)

    def prepare_nn_input(self, mass):
        """(n_c - 2, 7): [M[i,i-1], M[i,i], M[i,i+1], M[i+1,i+1], M[i+1,i+2], M[i+2,i+2], M[i+2,i+3]] for odd i"""
        M = sp.csr_matrix(mass)
        dim = M.shape[0]
        i = np.arange(1, dim - 2, 2)
        rows = np.stack([i, i, i, i + 1, i + 1, i + 2, i + 2], axis=1)
        cols = np.stack([i - 1, i, i + 1, i + 1, i + 2, i + 2, i + 3], axis=1)
        return np.asarray(M[rows.ravel(), cols.ravel()]).reshape(-1, 7)[:int((dim - 1) / 2) - 1]

    def construct_B(self, data_M, M):
        dim = M.shape[0]
        nc = int((dim - 1) / 2) + 1
        res = np.asarray(self.model.predict(data_M), dtype=np.float64)
        k = np.arange(res.shape[0])
        r = np.concatenate([2 * k + 2, 2 * k + 1, 2 * k + 2, 2 * k + 3, 2 * k + 2])
        c = np.concatenate([k, k + 1, k + 1, k + 1, k + 2])
        v = np.concatenate([res[:, 2], res[:, 4], res[:, 5], res[:, 6], res[:, 8]])
        B = sp.lil_matrix(sp.csr_matrix((v, (r, c)), shape=(dim, nc)))      # every (row, col) is written once
        Ms = sp.csr_matrix(M)
        diff = np.asarray(Ms.sum(axis=1)).ravel() - np.asarray(B.sum(axis=1)).ravel()
        B[0, 0], B[1, 0] = diff[0], diff[1]
        B[dim - 2, nc - 1], B[dim - 1, nc - 1] = diff[-2], diff[-1]
        B = sp.csr_matrix(B)
        row_sums = np.asarray(B.sum(axis=1)).ravel()
        Q = sp.csr_matrix(sp.diags(1.0 / row_sums) @ B)
        Q.sort_indices()
        return Q

    def transfer_op(self, M):
        """Q of one level (Multigrid.py:306-311); dense ndarray for a dense M (like the reference), CSR otherwise"""
        data_M = (self.prepare_nn_input(M) - self.mean) / self.std
        Q = self.construct_B(data_M, M)
        return Q.toarray() if not sp.issparse(M) else Q

    def define_hierarchy(self, levels=2):
        """the transfer operators of all levels, M coarsened by Q^T M Q between them (:269-275)"""
        M = sp.csr_matrix(self.M)
        qs = []
        for _ in range(levels - 1):
            Q = sp.csr_matrix(self.transfer_op(M))
            qs.append(Q)
            M = sp.csr_matrix(Q.T @ M @ Q)
        self.l_hierarchy = qs

    def solve(self, levels=2, smoother="Jacobi", smooth_steps=1, max_iterations=100, error=1e-08,
              initial_guess=None, cycle="V", first_call=True, **kw):
        if len(self.l_hierarchy) != levels - 1:
            self.define_hierarchy(levels)
        super().solve(levels, smoother, smooth_steps, max_iterations, error, initial_guess, cycle, True, **kw)

    def v_cycle(self, A, M, u0, rhs, smoother, smooth_steps, error, levels, first_call=False, **kw):
        """One V-cycle with the reference's argument list (Multigrid.py:246: the level's mass matrix M comes second).
        The transfer operators are predicted from M for all levels at once (define_hierarchy) and kept while the same
        M object and level count are passed; the cycle itself is Multigrid.v_cycle on the device."""
        if M is not self.M or len(self.l_hierarchy) != levels - 1:
            self.M = M
            self.define_hierarchy(levels)
            self._hier = None
        return super().v_cycle(A, u0, rhs, smoother, smooth_steps, error, levels, True, **kw)

    def _given_transfers(self):
        return self.l_hierarchy


class NeuralMG_2D(Multigrid):
    """NeuralMG_2D(matrix, rhs, model, M, std, mean) -- Multigrid.py:373-765.  `define_hierarchy(levels)` builds the
    transfer operators from the mass matrix M with the predictor `model` (anything with `.predict(X) -> (len(X), 31)`,
    the Keras interface the reference uses, or `.predict_device`), on the device (learnmultigrid_b200/neural2d.py).

    Differences, all explicit: the reference stores the hierarchy in `l_hierarchy` but its `solve` never uses it
    (no `interpolator` override: it falls through to the 1D geometric interpolator, SURVEY 2 row 4); here `solve`
    runs the V-cycle with `l_hierarchy`.  `fill_B` returns B as a SciPy CSR matrix instead of a dense n x n_C array.
    Coarse nodes with 7..12 neighbours get the reference's extra patch variants (:631-663; rows appended behind the
    regular patches); more than 12 is an MgError (the reference fails there too)."""

    def __init__(self, matrix, rhs, model, M, std, mean):
        super().__init__(matrix, rhs)
        self.label = "NeuralMG"
        self.model = model
        self.M = M
        self.std = std
        self.mean = mean
        self.l_hierarchy = []
        self._builder = None

    def _nb(self):
        if self._builder is None:
            from ..neural2d import NeuralBuilder
            self._builder = NeuralBuilder()
        return self._builder

    @staticmethod
    def diff(first, second):
        second = set(second)
        return [item for item in first if item not in second]

    @staticmethod
    def scaling_vnodes(_neighs):
        switcher = {2: [6, 1], 3: [3, 2], 4: [2, 3], 5: [1.5, 4]}
        return switcher.get(_neighs, "Invalid month")

    @staticmethod
    def map_coarse(_C):
        return dict(zip(_C, range(len(_C))))

    @staticmethod
    def get_conn(mat):
        """dense 0/1 adjacency of the positive off-diagonal entries (Multigrid.py:391-398); unlike the reference's
        `mat[:]`, which is a view for some SciPy formats, the argument is left untouched"""
        Mh = sp.csr_matrix(mat, copy=True)
        Mh.setdiag(0)
        Mh.eliminate_zeros()
        out = Mh.toarray()
        out[out > 0] = 1
        return out

    def create_virtual_nodes(self, row, node_M):
        """(virtual_neighs, row) of Multigrid.py:438-454: a node with fewer than 6 neighbours gets 6 - k virtual ones
        worth node_M / down each, and every virtual neighbour a patch row [node_M * up, 5 x node_M / down], with
        (up, down) = scaling_vnodes(k).  The per-node steps that follow in the reference (direct_neighs,
        intersecting_rows, single_extraction) are one CUDA thread per coarse node here (csrc/nn_kernels.cu, reached
        through extract_patches)."""
        row = np.asarray(row, dtype=np.float64)
        k = len(row)
        if k >= 6:
            return [], row
        up, down = self.scaling_vnodes(k)
        row = np.concatenate([row, np.full(6 - k, node_M / down)])
        virtual = np.tile(np.concatenate([[node_M * up], np.full(5, node_M / down)]), 6 - k)
        return virtual, row

    def coarsening(self, _conn):
        """(CC, FF, CC_neighs, FF_neighs) as Multigrid.py:401-426; CC in selection (= ascending) order"""
        nb = self._nb()
        Mh = F.canonical_csr(sp.csr_matrix(_conn))
        cmap, clist, nc = nb.coarsen(nb.upload(Mh))
        CC = [int(v) for v in clist.cpu().numpy()]
        is_c = cmap.cpu().numpy() >= 0
        FF = [int(i) for i in np.flatnonzero(~is_c)]
        offd = Mh.copy()
        offd.setdiag(0)
        offd.eliminate_zeros()

        def neighs(i):
            r = offd.getrow(i)
            return r.indices[r.data > 0]
        return CC, FF, {i: neighs(i) for i in CC}, {i: neighs(i) for i in FF}

    def extract_patches(self, CC, _mat):
        nb = self._nb()
        torch = nb.torch
        Mh = F.canonical_csr(sp.csr_matrix(_mat))
        n = Mh.shape[0]
        cmap = -np.ones(n, dtype=np.int32)
        cmap[np.asarray(CC, dtype=np.int64)] = np.arange(len(CC), dtype=np.int32)
        clist = torch.from_numpy(np.asarray(CC, dtype=np.int32)).to(nb.dev)
        patches, fill = nb.extract(nb.upload(Mh), torch.from_numpy(cmap).to(nb.dev), clist)
        return patches.cpu().numpy(), fill.cpu().numpy().astype(int)

    def fill_B(self, _res, _idx_fill, total_size, mapping, CC):
        nb = self._nb()
        torch = nb.torch
        cmap = -np.ones(total_size, dtype=np.int32)
        for k, v in mapping.items():
            cmap[int(k)] = int(v)
        pred = torch.from_numpy(np.ascontiguousarray(_res, dtype=np.float64)).to(nb.dev)
        fill = torch.from_numpy(np.ascontiguousarray(_idx_fill, dtype=np.int32)).to(nb.dev)
        B, dn = nb.fill_B(pred, fill, torch.from_numpy(cmap).to(nb.dev), total_size, len(CC))
        dn = dn.cpu().numpy()
        return nb.download(B), {k: dn[k][dn[k] >= 0].astype(int) for k in range(len(CC))}

    def pre_process(self, mass, d_neighs):
        nb = self._nb()
        torch = nb.torch
        Mh = F.canonical_csr(sp.csr_matrix(mass))
        dn = -np.ones((Mh.shape[0], 6), dtype=np.int32)
        for k, v in d_neighs.items():
            dn[int(k), :len(v)] = v
        return nb.download(nb.cut(nb.upload(Mh), torch.from_numpy(dn).to(nb.dev)))

    def define_hierarchy(self, levels=2):
        if levels == 1:
            print("Coarse grid correction not required")
            return
        nb = self._nb()
        Qs = nb.define_hierarchy(F.canonical_csr(sp.csr_matrix(self.M)), self.model, self.mean, self.std, levels)
        self.l_hierarchy = [nb.download(Q) for Q in Qs]

    def solve(self, levels=2, smoother="Jacobi", smooth_steps=1, max_iterations=100, error=1e-08,
              initial_guess=None, cycle="V", first_call=True, **kw):
        if len(self.l_hierarchy) < levels - 1:
            self.define_hierarchy(levels)
        super().solve(levels, smoother, smooth_steps, max_iterations, error, initial_guess, cycle, first_call, **kw)

    def _given_transfers(self):
        return self.l_hierarchy
