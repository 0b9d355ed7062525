"""Conjugate gradients with the reference's interface (learn_multigrid/solvers/CG.py:5-50) on the GPU, plus an
optional V-cycle preconditioner (BASELINE.json configs[4]: MG-preconditioned CG)."""
import numpy as np

from .. import _lib
from .Solver import IterativeSolver


def _same_operator(P, A, P_src=None, A_src=None):
    """True only if the preconditioner was built from THIS operator (same object -- the stored matrix or the object the
    caller constructed both solvers from -- or the same CSC arrays entry for entry); a multigrid built from another
    matrix of the same sparsity must not replace A in `A p`."""
    if P is None:
        return False
    if P is A or (P_src is not None and P_src is A_src):
        return True
    if P.shape != A.shape or P.nnz != A.nnz or P.format != A.format:
        return False
    return (np.array_equal(P.indptr, A.indptr) and np.array_equal(P.indices, A.indices)
            and np.array_equal(P.data, A.data))


class CG(IterativeSolver):

    def __init__(self, matrix, rhs):
        super().__init__(matrix, rhs)
        self.label = "CG"

    def solve(self, max_iterations=1000, error=1e-08, initial_guess=None, preconditioner=None):
        """Textbook CG (CG.py:12-50): history starts with the initial residual, absolute tolerance.
        The reference evaluates `alpha * A @ p` (rescales A, second SpMV, CG.py:37); here A p is reused, which
        changes results only in the last bits.  `preconditioner(r_dev, z_dev)` applies z = M^-1 r on device
        vectors (see solvers.Multigrid.Multigrid.as_preconditioner)."""
        h = getattr(preconditioner, "hierarchy", None)
        if (h is not None and initial_guess is None
                and _same_operator(getattr(preconditioner, "matrix", None), self.matrix,
                                   getattr(preconditioner, "matrix_src", None), getattr(self, "_matrix_src", None))):
            # the preconditioner's hierarchy already holds this operator on the device (SELL, level-0 ordering): run
            # the whole iteration there (engine.DeviceHierarchy.pcg: scalars on the device, one CUDA graph per
            # iteration; also on a row-partitioned hierarchy) instead of uploading a second copy of the matrix
            x, track, its = h.pcg(self.rhs, preconditioner.params, error=error, max_iterations=max_iterations)
            r = h._from_level0(h.levels[0].b)                         # the residual lives in the level-0 rhs buffer
            if getattr(h, "comm", None) is not None:                  # partitioned: x and r are this rank's row blocks
                if not getattr(self, "local_solution", False):
                    x, r = h.global_rows(x, r)
                h.check()
            self.iterations += its
            self.solution = x
            self.residual = track[-1]
            self.track_res = np.array(track, dtype=float).reshape(-1, 1)
            self.residual_vector = r
            self.last_timing = getattr(h, "last_pcg_timing", None)
            return
        if h is not None and getattr(h, "null", None) is not None:
            # the host loop projects neither b nor x: with a singular operator it would not converge
            raise ValueError("a multigrid preconditioner with a declared null space runs CG inside its hierarchy only: "
                             "call solve() without initial_guess, on the preconditioner's own matrix")
        d = self._device_csr()
        torch, lib, n = d["torch"], d["lib"], d["n"]
        st = _lib.stream_handle(torch)
        if initial_guess is None:
            x0 = np.zeros(shape=(self.get_dimension(), 1))
        else:
            x0 = initial_guess
        x = self._upload(x0)
        b = self._upload(self.rhs)
        r = torch.empty_like(x)
        Ap = torch.empty_like(x)
        self._residual(x, b, r)
        self.residual = self._norm(r)
        track = [self.residual]
        if preconditioner is None:
            z = r
        else:
            z = torch.empty_like(x)
            preconditioner(r, z)
        p = z.clone()
        rz = self._dot(r, z)

        def axpby(a, xx, bb, yy, out):
            _lib.check(lib.mg_axpby(n, float(a), xx.data_ptr(), float(bb), yy.data_ptr(), out.data_ptr(), st),
                       "mg_axpby")

        for _ in range(0, max_iterations):
            self.iterations += 1
            _lib.check(lib.mg_spmv_csr(n, d["indptr"].data_ptr(), d["indices"].data_ptr(), d["values"].data_ptr(),
                                       p.data_ptr(), Ap.data_ptr(), st), "mg_spmv_csr")
            pAp = self._dot(p, Ap)
            alpha = rz / pAp
            axpby(alpha, p, 1.0, x, x)            # x = x + alpha p
            axpby(-alpha, Ap, 1.0, r, r)          # r = r - alpha A p
            self.residual = self._norm(r)
            track.append(self.residual)
            if self.residual <= error:
                break
            if preconditioner is not None:
                preconditioner(r, z)
            rz_new = self._dot(r, z)
            beta = rz_new / rz
            rz = rz_new
            axpby(beta, p, 1.0, z, p)             # p = z + beta p
        self.solution = x.cpu().numpy().reshape(self.dim, 1)
        self.residual_vector = r.cpu().numpy().reshape(self.dim, 1)
        self.track_res = np.array(track, dtype=float).reshape(-1, 1)
