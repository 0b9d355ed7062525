"""Restarted GMRES, right-preconditioned by a multigrid V-cycle, on the GPU.  Unlike CG it needs neither a symmetric
operator nor a symmetric preconditioner: the reference's own row-Dirichlet operators, the forward multicolour and
index-order Gauss-Seidel cycles, the algebraic hierarchies and convection-diffusion problems all qualify."""
import numpy as np

from .CG import _same_operator
from .Solver import IterativeSolver


class GMRES(IterativeSolver):

    def __init__(self, matrix, rhs):
        super().__init__(matrix, rhs)
        self.label = "GMRES"

    def solve(self, max_iterations=1000, error=1e-08, initial_guess=None, preconditioner=None, restart=30):
        """GMRES(restart) with the absolute tolerance `error` (engine.DeviceHierarchy.gmres).  `preconditioner` must
        be `Multigrid.as_preconditioner(...)` of a multigrid built from this matrix: the whole iteration runs in its
        device hierarchy (any Multigrid subclass, every smoother, also after `distribute()`).
        iterations counts Arnoldi steps and accumulates over calls; track_res is ||b - A x0|| followed by the GMRES
        estimate after every step; residual and residual_vector are the true residual b - A x of the solution."""
        h = getattr(preconditioner, "hierarchy", None)
        if h is None or not _same_operator(getattr(preconditioner, "matrix", None), self.matrix,
                                           getattr(preconditioner, "matrix_src", None),
                                           getattr(self, "_matrix_src", None)):
            raise ValueError("GMRES runs inside the device hierarchy of a multigrid preconditioner: pass "
                             "Multigrid.as_preconditioner(...) of a multigrid built from this matrix")
        x, track, its, res = h.gmres(self.rhs, preconditioner.params, error=error, max_iterations=max_iterations,
                                     restart=restart, x0=initial_guess)
        r = h.gmres_residual_vector()
        if getattr(h, "comm", None) is not None:            # partitioned: x and r are this rank's row blocks
            if not getattr(self, "local_solution", False):
                x, r = h.global_rows(x, r)
            h.check()
        self.iterations += its
        self.solution = x
        self.residual = res
        self.track_res = np.array(track, dtype=float).reshape(-1, 1)
        self.residual_vector = r
        self.last_timing = getattr(h, "last_gmres_timing", None)
