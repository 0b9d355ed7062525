"""Synthetic P1 problems of BASELINE.json's configurations, generated with vectorised NumPy (host side).

The structured 2D generators write the assembled operator directly (closed form of the reference's element
loop on the right-triangle mesh) so that 16M / 64M-DOF inputs are produced in seconds; tests check them against
the reference's own assembly on small meshes (tests/golden/assembly_2d.npz).
"""
import numpy as np
import scipy.sparse as sp

from . import formats as F


def symmetric_dirichlet(A, boundary):
    """Zero the columns of the Dirichlet nodes in the other rows (their values are 0, so the solution is unchanged):
    the operator becomes symmetric, as MG-preconditioned CG needs (the 1D scripts do the same: `A[1,0]=0;
    A[-2,-1]=0`, test/test_NN.py:176-177).  Explicit zeros are dropped."""
    A = sp.csr_matrix(A)
    keep = np.ones(A.shape[0])
    keep[boundary] = 0.0
    D = sp.diags(keep)
    B = sp.csr_matrix(A @ D + sp.diags(1.0 - keep) @ sp.diags(A.diagonal()))
    B.eliminate_zeros()
    B.sort_indices()
    return F.raw_csr(B.indptr.astype(np.int32), B.indices.astype(np.int32), B.data, B.shape)


def boundary_nodes_2d(N):
    W = N + 1
    iy, ix = np.divmod(np.arange(W * W, dtype=np.int64), W)
    return np.flatnonzero((ix == 0) | (ix == N) | (iy == 0) | (iy == N))


def structured_laplacian_2d(N, coefficient=None, rows=None, Ny=None):
    """P1 stiffness matrix of -div(k grad u) on the reference's structured mesh Mesh2D(N*N) ((N+1)^2 nodes, row
    major), with boundary rows replaced by identity rows exactly as test/thesis_structured_2d.py:407-414.
    k = 1 gives the 5-point stencil [-1,-1,4,-1,-1] (hypotenuse couplings are exact zeros and not stored);
    `coefficient(x, y)` is evaluated at element centroids.  Returns canonical CSR.
    rows=(r0, r1): only that row block (global column ids) -- what one rank of a row-partitioned run generates, so
    that no process ever holds the global operator (partition_setup.py).
    Ny: number of squares in y (default N): the domain is [0, 1] x [0, Ny/N] with the same square cells of side 1/N --
    the stacked strips of a weak-scaling run (one N x N square per GPU)."""
    Ny = N if Ny is None else int(Ny)
    W = N + 1
    n = W * (Ny + 1)
    r0, r1 = (0, n) if rows is None else (int(rows[0]), int(rows[1]))
    if not 0 <= r0 <= r1 <= n:
        raise ValueError("row block outside the matrix")
    if (r1 - r0) * 5 >= 2 ** 31 or n >= 2 ** 31:
        raise OverflowError("nnz does not fit int32")
    iy, ix = np.divmod(np.arange(r0, r1, dtype=np.int64), W)
    interior = (ix > 0) & (ix < N) & (iy > 0) & (iy < Ny)
    counts = np.where(interior, 5, 1).astype(np.int64)
    indptr = np.zeros(r1 - r0 + 1, dtype=np.int64)
    np.cumsum(counts, out=indptr[1:])
    indices = np.empty(indptr[-1], dtype=np.int32)
    data = np.empty(indptr[-1], dtype=np.float64)
    b = np.flatnonzero(~interior)
    indices[indptr[b]] = b + r0
    data[indptr[b]] = 1.0
    loc = np.flatnonzero(interior)
    r = loc + r0                                   # global row ids of the interior rows of the block
    base = indptr[loc]
    if coefficient is None:
        vals = (-1.0, -1.0, 4.0, -1.0, -1.0)
        for k, off in enumerate((-W, -1, 0, 1, W)):
            indices[base + k] = r + off
            data[base + k] = vals[k]
    else:
        h = 1.0 / N
        # element coefficients: lower triangle (type 1: [k,k+1,k+W+1]) and upper (type 2: [k,k+W+1,k+W]) of square (sx,sy)
        def k1(sx, sy):
            return coefficient((sx + 2.0 / 3.0) * h, (sy + 1.0 / 3.0) * h)

        def k2(sx, sy):
            return coefficient((sx + 1.0 / 3.0) * h, (sy + 2.0 / 3.0) * h)
        x, y = ix[loc], iy[loc]
        # horizontal edge (x,y)-(x+1,y): shared by type-1 of square (x,y) [legs] and type-2 of square (x,y-1)
        east = -0.5 * (k1(x, y) + k2(x, y - 1))
        west = -0.5 * (k1(x - 1, y) + k2(x - 1, y - 1))
        # vertical edge (x,y)-(x,y+1): type-2 of square (x,y) and type-1 of square (x-1,y)
        north = -0.5 * (k2(x, y) + k1(x - 1, y))
        south = -0.5 * (k2(x, y - 1) + k1(x - 1, y - 1))
        diag = -(east + west + north + south)
        for k, (off, v) in enumerate(((-W, south), (-1, west), (0, diag), (1, east), (W, north))):
            indices[base + k] = r + off
            data[base + k] = v
    return F.raw_csr(indptr.astype(np.int32), indices, data, (r1 - r0, n))


def convection_diffusion_2d(N, eps, beta):
    """-eps * Laplace(u) + beta . grad(u) on the mesh of structured_laplacian_2d(N), scaled like it (by h^2): the
    5-point diffusion stencil times eps plus first-order upwind convection times h (for beta_x > 0 the row gets
    +h beta_x on the diagonal and -h beta_x on its west neighbour, for beta_x < 0 the same with |beta_x| and the east
    neighbour; likewise in y).  Boundary rows are identity rows as in structured_laplacian_2d, so for beta != 0 the
    operator is nonsymmetric twice over; eps = 1, beta = (0, 0) gives structured_laplacian_2d(N) entry for entry.
    Interior rows sum to zero, the diagonal is positive and the off-diagonals are negative (an M-matrix).
    Canonical CSR."""
    eps = float(eps)
    bx, by = (float(v) for v in beta)
    if not eps > 0.0:
        raise ValueError("eps must be positive")
    A = structured_laplacian_2d(N)
    h = 1.0 / N
    base = A.indptr[:-1][np.diff(A.indptr) == 5].astype(np.int64)    # interior rows: (south, west, diag, east, north)
    d = A.data
    idx = base[:, None] + np.arange(5)
    d[idx] = eps * d[idx]
    for b, lo, hi in ((bx, 1, 3), (by, 0, 4)):               # (component, upwind slot for b > 0, for b < 0)
        c = h * abs(b)
        if c == 0.0:
            continue
        d[base + 2] = d[base + 2] + c
        up = lo if b > 0 else hi
        d[base + up] = d[base + up] - c
    return A


def structured_rhs_2d(N, f_value=-1.0, rows=None, Ny=None):
    """load vector of f = const on the structured mesh with Dirichlet rows zeroed: interior entries f*h^2
    (six triangles of area h^2/2, each contributing f*area/3), thesis_structured_2d.py:17-19,403,414.
    rows / Ny as in structured_laplacian_2d."""
    Ny = N if Ny is None else int(Ny)
    W = N + 1
    h = 1.0 / N
    r0, r1 = (0, W * (Ny + 1)) if rows is None else (int(rows[0]), int(rows[1]))
    iy, ix = np.divmod(np.arange(r0, r1, dtype=np.int64), W)
    interior = (ix > 0) & (ix < N) & (iy > 0) & (iy < Ny)
    return np.where(interior, f_value * h * h, 0.0).reshape(-1, 1)


def linear_P_2d(Nf, rows=None, Nyf=None):
    """linear interpolation from the nested coarse mesh Mesh2D((Nf/2)^2) to Mesh2D(Nf^2): coincident nodes 1,
    edge midpoints 1/2 + 1/2 (horizontal, vertical and the lower-left/upper-right diagonal).  CSR.
    rows=(r0, r1): only that block of fine rows (global coarse column ids).
    Nyf: squares in y of the fine mesh (default Nf), for the rectangular meshes of structured_laplacian_2d(Ny=)."""
    Nyf = Nf if Nyf is None else int(Nyf)
    if Nf % 2 or Nyf % 2:
        raise ValueError("Nf must be even")
    Wf, Wc = Nf + 1, Nf // 2 + 1
    nf, nc = Wf * (Nyf + 1), Wc * (Nyf // 2 + 1)
    r0, r1 = (0, nf) if rows is None else (int(rows[0]), int(rows[1]))
    if not 0 <= r0 <= r1 <= nf:
        raise ValueError("row block outside the matrix")
    iy, ix = np.divmod(np.arange(r0, r1, dtype=np.int64), Wf)
    cx, cy = ix // 2, iy // 2
    ox, oy = ix % 2, iy % 2
    two = (ox + oy) > 0
    counts = np.where(two, 2, 1)
    indptr = np.zeros(r1 - r0 + 1, dtype=np.int64)
    np.cumsum(counts, out=indptr[1:])
    indices = np.empty(indptr[-1], dtype=np.int32)
    data = np.empty(indptr[-1], dtype=np.float64)
    first = cy * Wc + cx
    second = (cy + oy) * Wc + (cx + ox)
    indices[indptr[:-1]] = first
    data[indptr[:-1]] = np.where(two, 0.5, 1.0)
    t = np.flatnonzero(two)
    indices[indptr[t] + 1] = second[t]
    data[indptr[t] + 1] = 0.5
    return F.raw_csr(indptr.astype(np.int32), indices, data, (r1 - r0, nc))


def structured_mass_2d(N):
    """P1 mass matrix on Mesh2D(N*N) through the vectorised assembly (7-point pattern)."""
    from .mesh.Mesh2D import Mesh2D
    from .assembly.MassMatrix import MassMatrix
    from .assembly.Quadrature import Quadrature2D
    from .assembly.ShapeFunction import FunctionTriangle
    return MassMatrix(Mesh2D(N * N)).compute_mass_2d(FunctionTriangle(1), Quadrature2D(3), format="csr")


def quasi_l2_Q_2d(Nf):
    """semi-geometric quasi-L2 transfer between the nested structured meshes: Q = rownormalise(M_h P)."""
    P = linear_P_2d(Nf)
    B = sp.csr_matrix(structured_mass_2d(Nf) @ P)
    s = np.asarray(B.sum(axis=1)).ravel()
    Q = sp.csr_matrix(sp.diags(1.0 / s) @ B)
    Q.sort_indices()
    return Q


def structured_hierarchy_2d(N, levels, transfer="linear", Ny=None):
    """[Q_0, ..., Q_{levels-2}] for the nested structured meshes N, N/2, ...  (Ny: squares in y, linear transfers only)"""
    if Ny is not None and transfer != "linear":
        raise ValueError("rectangular meshes: linear transfers only")
    qs = []
    n, ny = N, (N if Ny is None else int(Ny))
    for _ in range(levels - 1):
        if n % 2 or n < 2 or ny % 2 or ny < 2:
            raise ValueError("mesh cannot be coarsened %d times" % (levels - 1))
        qs.append(linear_P_2d(n, Nyf=ny) if transfer == "linear" else quasi_l2_Q_2d(n))
        n //= 2
        ny //= 2
    return qs


def redblack_colors_2d(N):
    W = N + 1
    iy, ix = np.divmod(np.arange(W * W), W)
    return ((ix + iy) % 2).astype(np.int32)


def structured_colors_2d(N, levels):
    """Per-level colourings for the structured hierarchy with LINEAR transfers: red-black (ix+iy)%2 for the 5-point
    fine operator, (ix+iy)%3 for the 7-point Galerkin operators (stencil offsets (+-1,0), (0,+-1), +-(1,1) never
    differ by a multiple of 3).  One colour fewer than first-fit greedy on the coarse levels, i.e. one launch and one
    halo exchange fewer per sweep; the last (coarsest) level is solved directly and gets None."""
    out = []
    n = N
    for l in range(levels - 1):
        W = n + 1
        iy, ix = np.divmod(np.arange(W * W), W)
        out.append(((ix + iy) % (2 if l == 0 else 3)).astype(np.int32))
        n //= 2
    out.append(None)
    return out


def stencil_offsets_2d(A, N):
    """set of (dx, dy) grid offsets of the off-diagonal entries of an operator on the (N+1)^2 row-major grid"""
    W = N + 1
    A = sp.coo_matrix(A)
    off = (A.row != A.col) & (A.data != 0)
    r, c = A.row[off].astype(np.int64), A.col[off].astype(np.int64)
    d = np.unique(np.stack([c % W - r % W, c // W - r // W], axis=1), axis=0)
    return [tuple(int(v) for v in t) for t in d]


def lattice_rule(offsets, max_colors=40):
    """smallest m and (alpha, beta) such that colour = (alpha*ix + beta*iy) mod m separates every pair of grid points
    whose offset is in `offsets`"""
    d = np.asarray(offsets, dtype=np.int64)
    if len(d) == 0:
        return 1, 0, 0
    for m in range(2, max_colors + 1):
        for alpha in range(m):
            for beta in range(m):
                if np.all((alpha * d[:, 0] + beta * d[:, 1]) % m != 0):
                    return m, alpha, beta
    raise ValueError("no lattice colouring with at most %d colours" % max_colors)


def lattice_colors_2d(N, levels, transfer="linear", coefficient=None, model_N=None):
    """Per-level lattice colourings (alpha*ix + beta*iy) mod m for the structured hierarchy.  The stencil offsets of
    every level are read off a SMALL instance of the same hierarchy (model_N, default 16 * 2^(levels-1) capped at N;
    translation-invariant stencils do not depend on the grid size), so no Galerkin product of the big problem is
    needed on the host.  Fewer colours than first-fit greedy: 2 / 3 for the 5- / 7-point operators, 7 / 12-13 for the
    19- / 37-point ones of quasi-L2 transfers."""
    if model_N is None:
        model_N = min(N, 16 * 2 ** (levels - 1))
    A = sp.csr_matrix(structured_laplacian_2d(model_N, coefficient))
    Qs = structured_hierarchy_2d(model_N, levels, transfer=transfer)
    rules = []
    n = model_N
    for l in range(levels - 1):
        rules.append(lattice_rule(stencil_offsets_2d(A, n)))
        A = sp.csr_matrix(Qs[l].T @ A @ Qs[l])
        n //= 2
    out = []
    n = N
    for m, alpha, beta in rules:
        W = n + 1
        iy, ix = np.divmod(np.arange(W * W, dtype=np.int64), W)
        out.append(((alpha * ix + beta * iy) % m).astype(np.int32))
        n //= 2
    out.append(None)
    return out


def coloring_is_valid(A, colors):
    """no off-diagonal entry of A joins two rows of the same colour"""
    A = sp.coo_matrix(A)
    off = A.row != A.col
    return not np.any(colors[A.row[off]] == colors[A.col[off]])


def irregular_p1_2d(N, seed=42, f_value=-1.0):
    """BASELINE configs[1] (C2): the reference's own notion of an unstructured mesh -- Mesh2D((N/2)^2) followed by one
    irregular red refinement (Mesh2D.refine(regular=False): new edge points at r in [0.3, 0.7] along each edge,
    Mesh2D.py:110-135; parents are numbered first, edge nodes in element-edge discovery order) -- with P1 stiffness,
    mass and load (f = const) and row-replaced Dirichlet rows (thesis_structured_2d.py:407-414).  (N+1)^2 nodes.
    Returns dict(A, M, rhs, boundary, mesh)."""
    from .mesh.Mesh2D import Mesh2D
    from .assembly.MassMatrix import MassMatrix
    from .assembly.StiffnessMatrix import StiffnessMatrix
    from .assembly.LoadVector import LoadVector
    from .assembly.Quadrature import Quadrature2D
    from .assembly.ShapeFunction import FunctionTriangle, GradientTriangle
    if N % 2:
        raise ValueError("N must be even")
    np.random.seed(seed)
    mesh = Mesh2D((N // 2) ** 2)
    mesh.refine(regular=False)
    q = Quadrature2D(3)
    A = StiffnessMatrix(mesh).compute_stiffness_2d(GradientTriangle(1), q, format="csr")
    M = MassMatrix(mesh).compute_mass_2d(FunctionTriangle(1), q, format="csr")
    from .assembly.LoadFunction import LoadFunction
    rhs = LoadVector(mesh).compute_rhs_2d(LoadFunction(lambda pts: f_value), FunctionTriangle(1), q)
    p = np.asarray(mesh.get_points())
    eps = 1e-12
    boundary = np.flatnonzero((p[:, 0] < eps) | (p[:, 0] > 1 - eps) | (p[:, 1] < eps) | (p[:, 1] > 1 - eps))
    A = sp.lil_matrix(A)
    for i in boundary:                      # A[nodes,:] = I[nodes,:]
        A.rows[i] = [int(i)]
        A.data[i] = [1.0]
    A = F.canonical_csr(sp.csr_matrix(A))
    rhs = np.asarray(rhs, dtype=np.float64).reshape(-1, 1).copy()
    rhs[boundary] = 0.0
    return {"A": A, "M": F.canonical_csr(sp.csr_matrix(M)), "rhs": rhs, "boundary": boundary, "mesh": mesh}


def variable_coefficient(x, y):
    """k(x,y) = 1 + 0.9 sin(2 pi x) sin(2 pi y)  (SURVEY.md 8d, config C4)"""
    return 1.0 + 0.9 * np.sin(2 * np.pi * x) * np.sin(2 * np.pi * y)
