"""NumPy restatement of the device GMRES (csrc/krylov_kernels.cu, cycle.cu mg_gmres_*, engine.DeviceHierarchy.gmres),
operation for operation: right preconditioning, restarts, classical Gram-Schmidt in one pass, the Givens formulas with
every operation rounded on its own, and the true-residual rule at a restart and at exit.  Test infrastructure."""
import math

import numpy as np
from scipy.sparse import csr_matrix


def gmres(A, b, precond=None, error=1e-8, max_iterations=1000, restart=30, x0=None):
    """precond(v) -> z = M^-1 v (None: z = v).  Returns (x, history, steps, true residual of x): the history is
    ||b - A x0||, then |g_{j+1}| after every step; the solve restarts from the updated x while its true residual is
    above `error` and steps remain."""
    if restart < 1:
        raise ValueError("restart must be >= 1")
    A = csr_matrix(A)
    b = np.asarray(b, dtype=np.float64).reshape(-1)
    n = b.size
    x = np.zeros(n) if x0 is None else np.asarray(x0, dtype=np.float64).reshape(-1).copy()
    m = restart
    its = 0
    track = []
    while True:
        r = b - A @ x                                        # mg_gmres_start
        beta = math.sqrt(float(r @ r))
        if not track:
            track.append(beta)
        if beta <= error or its >= max_iterations:
            break
        V = np.zeros((m + 1, n))
        Z = np.zeros((m, n))
        H = np.zeros((m + 1, m))                             # H[i, j]
        cs, sn = np.zeros(m), np.zeros(m)
        g = np.zeros(m + 1)
        g[0] = beta
        V[0] = r / beta if beta != 0.0 else r
        k = 0
        while k < m and its < max_iterations:
            j = k
            Z[j] = V[j] if precond is None else np.asarray(precond(V[j].reshape(-1, 1)), dtype=np.float64).reshape(-1)
            w = A @ Z[j]
            h = V[:j + 1] @ w                                # classical Gram-Schmidt: all dots against the same w
            for i in range(j + 1):
                w = w - h[i] * V[i]
            hn = math.sqrt(float(w @ w))
            for i in range(j):                               # earlier rotations on column j
                a, bb = h[i], h[i + 1]
                h[i] = cs[i] * a + sn[i] * bb
                h[i + 1] = -sn[i] * a + cs[i] * bb
            a = h[j]
            t = math.sqrt(a * a + hn * hn)
            c, s = (1.0, 0.0) if t == 0.0 else (a / t, hn / t)
            cs[j], sn[j] = c, s
            H[:j, j] = h[:j]
            H[j, j] = t
            gj = g[j]
            g[j + 1] = -s * gj
            g[j] = c * gj
            if hn != 0.0:
                V[j + 1] = w / hn
            its += 1
            k += 1
            est = math.sqrt(g[j + 1] * g[j + 1])
            track.append(est)
            if est <= error:
                break
        y = np.zeros(k)                                      # mg_gmres_finish: R y = g, x += sum y_c z_c
        for i in range(k - 1, -1, -1):
            acc = g[i]
            for c in range(i + 1, k):
                acc = acc - H[i, c] * y[c]
            y[i] = acc / H[i, i]
        for c in range(k):
            x = x + y[c] * Z[c]
    return x.reshape(-1, 1), track, its, beta
