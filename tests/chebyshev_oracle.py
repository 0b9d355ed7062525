"""CPU reference of the Chebyshev smoother (test infrastructure): one step and a V-cycle oracle that smooths with it.

The residual comes from the oracle's C residual kernel (storage order, no FMA), the element-wise steps from NumPy,
which rounds every product and sum on its own -- the definition of the device step (csrc/sell_modes_cheby.cu).  The
coefficient table is an input: the oracle never estimates bounds itself.
"""
import numpy as np
from scipy.sparse import csr_matrix

from oracle import kernels as K
from oracle.vcycle import OracleMultigrid


def cheby_step(A, x, b, d, dinv, c_d, c_r, first):
    """one step: returns (x_out, d_out) as flat float64 arrays"""
    r = np.ravel(K.residual(A, np.ravel(x), np.ravel(b)))
    t = dinv * r
    dn = c_r * t if first else (c_d * d) + (c_r * t)
    return np.ravel(x) + dn, dn


def cheby_smooth(A, u, rhs, table, steps):
    """`steps` applications of the polynomial whose (degree, 2) table of (c_d, c_r) is given"""
    A = csr_matrix(A)
    dinv = 1.0 / A.diagonal()
    x = np.array(np.ravel(u), dtype=np.float64, copy=True)
    b = np.ascontiguousarray(np.ravel(rhs), dtype=np.float64)
    d = np.zeros_like(x)
    for _ in range(int(steps)):
        for k in range(len(table)):
            x, d = cheby_step(A, x, b, d, dinv, float(table[k][0]), float(table[k][1]), k == 0)
    return x.reshape(np.shape(u))


class ChebyshevOracle(OracleMultigrid):
    """OracleMultigrid with smoother="chebyshev": cheby_coefficients = one (degree, 2) table per smoothing level"""

    def __init__(self, A, rhs, Q_list=None, smoother="chebyshev", cheby_coefficients=None, **kw):
        super().__init__(A, rhs, Q_list, smoother=smoother, **kw)
        self.cheby_coefficients = cheby_coefficients

    def _smooth(self, A, u, rhs, steps, level, post=False):
        if self.smoother != "chebyshev":
            return super()._smooth(A, u, rhs, steps, level, post)
        return cheby_smooth(A, u, rhs, self.cheby_coefficients[level], steps)
