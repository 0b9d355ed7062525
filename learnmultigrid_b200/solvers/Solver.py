"""Solver base classes with the reference's interface (learn_multigrid/solvers/Solver.py:8-84).

State lives on the host exactly like the reference (`solution`, `residual_vector` are (n,1) float64 arrays,
`track_res` is (k,1)); the compute behind `solve()` runs on the GPU through libmgb200.
"""
import ctypes

import numpy as np
import scipy.sparse as sp
from scipy.sparse import csc_matrix

from .. import _lib
from .. import formats as F


class Solver:
    def __init__(self, matrix, rhs):
        # Solver.py:14-21 (rhs may also be a pinned torch tensor: it is then copied to the device without staging)
        self.dim = int(rhs.numel()) if hasattr(rhs, "numel") else rhs.size
        shape = tuple(rhs.shape)
        self.residual_vector = np.empty(shape=shape)
        self.residual = 0.0
        self._matrix_src = matrix            # the caller's object: lets two solvers recognise the same operator
        # an operator that already lives in device memory (setup_device.DevCSR from assembly_device / problems_device)
        # stays there; anything else is held as the reference holds it
        self.matrix = matrix if hasattr(matrix, "ptrs") else csc_matrix(matrix)
        self.rhs = rhs
        self.solution = np.empty(shape=shape)
        self.track_res = np.ndarray(shape=(0, 1), dtype=float)
        self._dev = None

    # accessors of Solver.py:23-48 (read access is generated from the table below the class)
    def set_matrix(self, matrix):
        self.matrix = matrix
        self._matrix_src = matrix
        self._dev = None                 # the device copy belongs to the old matrix

    def set_rhs(self, rhs):
        self.rhs = rhs

    # ---- device plumbing shared by the stationary solvers and CG (natural ordering, CSR kernels) ----------
    def _device_csr(self):
        if self._dev is None:
            torch = _lib.require_cuda()
            A = F.canonical_csr(self.matrix)
            dev = torch.device("cuda", torch.cuda.current_device())
            d = {"torch": torch, "lib": _lib.load(), "n": A.shape[0], "host": A, "dev": dev,
                 "indptr": torch.from_numpy(A.indptr).to(dev), "indices": torch.from_numpy(A.indices).to(dev),
                 "values": torch.from_numpy(A.data).to(dev)}
            d["ws"] = torch.zeros(8192, dtype=torch.float64, device=dev)
            d["out"] = torch.zeros(1, dtype=torch.float64, device=dev)
            self._dev = d
        return self._dev

    def _upload(self, v):
        d = self._device_csr()
        v = np.ascontiguousarray(np.asarray(v, dtype=np.float64).reshape(-1))
        return d["torch"].from_numpy(v).to(d["dev"])

    def _norm(self, t):
        d = self._device_csr()
        st = _lib.stream_handle(d["torch"])
        _lib.check(d["lib"].mg_dot(t.numel(), t.data_ptr(), t.data_ptr(), d["ws"].data_ptr(), d["out"].data_ptr(), st),
                   "mg_dot")
        return float(np.sqrt(d["out"].item()))

    def _dot(self, a, b):
        d = self._device_csr()
        st = _lib.stream_handle(d["torch"])
        _lib.check(d["lib"].mg_dot(a.numel(), a.data_ptr(), b.data_ptr(), d["ws"].data_ptr(), d["out"].data_ptr(), st),
                   "mg_dot")
        return float(d["out"].item())

    def _residual(self, x, b, r):
        d = self._device_csr()
        st = _lib.stream_handle(d["torch"])
        _lib.check(d["lib"].mg_residual_csr(d["n"], d["indptr"].data_ptr(), d["indices"].data_ptr(),
                                            d["values"].data_ptr(), x.data_ptr(), b.data_ptr(), r.data_ptr(), st),
                   "mg_residual_csr")


def _reader(attribute):
    def read(self):
        return getattr(self, attribute)
    read.__name__ = read.__qualname__ = "get_" + attribute
    read.__doc__ = "the solver's `%s`" % attribute
    return read


for _name, _attribute in (("get_matrix", "matrix"), ("get_rhs", "rhs"), ("get_solution", "solution"),
                          ("get_residual", "residual"), ("get_residual_vector", "residual_vector"),
                          ("get_dimension", "dim"), ("get_track_res", "track_res")):
    setattr(Solver, _name, _reader(_attribute))


class DirectSolver(Solver):
    """spsolve replacement (Solver.py:51-59) on the device, for any sparse system: explicit inverse up to 4096 unknowns,
    block cyclic reduction beyond (after a reverse Cuthill-McKee reordering when the numbering is not banded,
    coarse.build_coarse_solver), followed by steps of iterative refinement with the residual formed in fp64 on the
    device until it stops shrinking."""

    DENSE_MAX = 4096
    REFINE_STEPS = 3

    def __init__(self, matrix, rhs):
        super().__init__(matrix, rhs)

    def solve(self, null_space=None):
        """null_space: None, "constant" or n values -- the null vector nu of a singular SYMMETRIC matrix.  The solve
        then runs through the pinned factor and returns the minimum-norm solution of the system with nu removed from
        the right-hand side (rhs_null_component: nu^T b / ||nu|| of what was removed; the least-squares solution when
        it is not 0); the refinement steps work on that projected system."""
        from ..coarse import build_coarse_solver, apply_coarse
        d = self._device_csr()
        torch, lib, n = d["torch"], d["lib"], d["n"]
        st = _lib.stream_handle(torch)
        nu = None
        if null_space is not None:
            from ..engine import declared_null_vector
            nu, _ = declared_null_vector(torch, d["dev"], d["host"], null_space)
        solver = build_coarse_solver(torch, d["dev"], n, d["indptr"], d["indices"], d["values"], self.DENSE_MAX,
                                     (d["host"].indptr, d["host"].indices), singular=nu is not None,
                                     label="DirectSolver")
        self.method = "dense inverse" if solver.kind == _lib.MG_COARSE_DENSE else (
            "block cyclic reduction" + (" after reverse Cuthill-McKee" if getattr(solver, "perm", None) is not None else ""))
        self.null_info = getattr(solver, "null_info", None)

        def apply(rhs, out):
            if nu is not None:
                apply_coarse(solver, rhs.clone(), out)
            elif solver.kind == _lib.MG_COARSE_DENSE:
                _lib.check(lib.mg_dense_gemv(n, n, solver.inv.data_ptr(), rhs.data_ptr(), out.data_ptr(), st),
                           "mg_dense_gemv")
            else:
                solver.solve(torch, rhs, out)

        def project(v):
            if nu is not None:
                _lib.check(lib.mg_project_out(n, nu.data_ptr(), inv_nn, -1, v.data_ptr(), d["ws"].data_ptr(), None, st),
                           "mg_project_out")

        b = self._upload(self.rhs)
        self.rhs_null_component = None
        if nu is not None:
            inv_nn = 1.0 / self._dot(nu, nu)
            self.rhs_null_component = self._dot(nu, b) * float(np.sqrt(inv_nn))
            project(b)
        x = torch.empty_like(b)
        apply(b, x)
        r = torch.empty_like(b)
        self._residual(x, b, r)
        res = self._norm(r)
        e = torch.empty_like(b)
        for _ in range(self.REFINE_STEPS):
            if res == 0.0:
                break
            apply(r, e)
            xn = x + e                     # one elementwise add per refinement step (setup-grade work)
            rn = torch.empty_like(b)
            self._residual(xn, b, rn)
            resn = self._norm(rn)
            if not resn < res:
                break
            x, r, res = xn, rn, resn
        project(x)
        self.solution = x.cpu().numpy().reshape(self.dim, 1)
        self.residual_vector = r.cpu().numpy().reshape(self.dim, 1)
        self.residual = res


class IterativeSolver(Solver):
    def __init__(self, matrix, rhs):
        super().__init__(matrix, rhs)
        self.iterations = 0          # Solver.py:72, never reset by the reference
        self.label = "Iterative Solver"

    def plot(self, scale="linear"):
        """Residual plot (Solver.py:75-81); needs matplotlib, which is optional here."""
        import matplotlib.pyplot as plt
        plt.plot(self.track_res, label=self.label)
        plt.yscale(scale)
        plt.legend()
        plt.title("Residual decreasing")
        plt.ylabel('residual')
        plt.xlabel('iterations')

    def get_iterations(self):
        return self.iterations
