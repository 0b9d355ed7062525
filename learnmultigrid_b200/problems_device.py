"""The structured synthetic problems of problems.py generated directly in device memory (benchmark inputs).

Same closed forms, same entry order, same float64 arithmetic as the host generators -- structured_laplacian_2d,
structured_rhs_2d, linear_P_2d -- evaluated with elementwise torch operations on the GPU, so a 67 M-DOF operator and
its five transfer operators exist in HBM after a fraction of a second instead of being built in NumPy and uploaded
(bench.py: generate_s).  Constant-coefficient output is bit-identical to the host generators; with a variable
coefficient the element coefficients go through the device's sin(), which may differ from NumPy's in the last bit.
This is input generation for the benchmark, not part of the solver: the P1 assembly of arbitrary meshes on the device
is assembly_device.py.
"""
import numpy as np

from . import _lib
from .setup_device import DevCSR


def _grid(torch, dev, N, Ny):
    W = N + 1
    n = W * (Ny + 1)
    if n * 5 >= 2 ** 31:
        raise OverflowError("nnz does not fit int32")
    i = torch.arange(n, dtype=torch.int64, device=dev)
    iy = torch.div(i, W, rounding_mode="floor")
    ix = i - iy * W
    return W, n, i, ix, iy


def variable_coefficient(torch, x, y):
    """k(x,y) = 1 + 0.9 sin(2 pi x) sin(2 pi y)  (problems.variable_coefficient)"""
    return 1.0 + 0.9 * torch.sin(2 * np.pi * x) * torch.sin(2 * np.pi * y)


def structured_laplacian_2d(N, coefficient=None, Ny=None, device=None, symmetric=False, boundary="dirichlet"):
    """problems.structured_laplacian_2d as a DevCSR; coefficient: None or a callable (torch, x, y) -> k.
    symmetric=True: problems.symmetric_dirichlet of it -- the couplings of interior rows to Dirichlet nodes are dropped
    (their values are zero, so the solution is unchanged) and the operator is symmetric, as conjugate gradients need.
    boundary="neumann": no Dirichlet rows (problems.structured_laplacian_2d(boundary="neumann")); symmetric as it is."""
    from .problems import _check_boundary
    _check_boundary(boundary)
    torch = _lib.require_cuda()
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    Ny = N if Ny is None else int(Ny)
    if boundary == "neumann":
        return _neumann_laplacian_2d(torch, dev, N, coefficient, Ny)
    if symmetric:
        return _symmetric_laplacian_2d(torch, dev, N, coefficient, Ny)
    W, n, i, ix, iy = _grid(torch, dev, N, Ny)
    interior = (ix > 0) & (ix < N) & (iy > 0) & (iy < Ny)
    counts = torch.where(interior, 5, 1)
    indptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    torch.cumsum(counts, 0, out=indptr[1:])
    nnz = int(indptr[-1].item())
    indices = torch.empty(nnz, dtype=torch.int32, device=dev)
    data = torch.empty(nnz, dtype=torch.float64, device=dev)
    b = torch.nonzero(~interior).reshape(-1)
    indices[indptr[b]] = b.to(torch.int32)
    data[indptr[b]] = 1.0
    r = torch.nonzero(interior).reshape(-1)
    base = indptr[r]
    del i, counts, interior, b
    if coefficient is None:
        vals = (-1.0, -1.0, 4.0, -1.0, -1.0)
        for k, off in enumerate((-W, -1, 0, 1, W)):
            indices[base + k] = (r + off).to(torch.int32)
            data[base + k] = vals[k]
    else:
        h = 1.0 / N
        x, y = ix[r].to(torch.float64), iy[r].to(torch.float64)

        def k1(sx, sy):
            return coefficient(torch, (sx + 2.0 / 3.0) * h, (sy + 1.0 / 3.0) * h)

        def k2(sx, sy):
            return coefficient(torch, (sx + 1.0 / 3.0) * h, (sy + 2.0 / 3.0) * h)
        east = -0.5 * (k1(x, y) + k2(x, y - 1))
        west = -0.5 * (k1(x - 1, y) + k2(x - 1, y - 1))
        north = -0.5 * (k2(x, y) + k1(x - 1, y))
        south = -0.5 * (k2(x, y - 1) + k1(x - 1, y - 1))
        diag = -(east + west + north + south)
        for k, (off, v) in enumerate(((-W, south), (-1, west), (0, diag), (1, east), (W, north))):
            indices[base + k] = (r + off).to(torch.int32)
            data[base + k] = v
    return DevCSR((n, n), indptr.to(torch.int32), indices, data)


def _symmetric_laplacian_2d(torch, dev, N, coefficient, Ny):
    """five candidate entries per interior row (south, west, centre, east, north), those that point at a boundary node
    removed; boundary rows are identity rows.  Entry order inside a row as on the host (ascending column)."""
    W, n, i, ix, iy = _grid(torch, dev, N, Ny)
    interior = (ix > 0) & (ix < N) & (iy > 0) & (iy < Ny)
    h = 1.0 / N
    x, y = ix.to(torch.float64), iy.to(torch.float64)
    if coefficient is None:
        one = torch.ones(n, dtype=torch.float64, device=dev)
        south = west = east = north = -one
        diag = 4.0 * one
    else:
        def k1(sx, sy):
            return coefficient(torch, (sx + 2.0 / 3.0) * h, (sy + 1.0 / 3.0) * h)

        def k2(sx, sy):
            return coefficient(torch, (sx + 1.0 / 3.0) * h, (sy + 2.0 / 3.0) * h)
        east = -0.5 * (k1(x, y) + k2(x, y - 1))
        west = -0.5 * (k1(x - 1, y) + k2(x - 1, y - 1))
        north = -0.5 * (k2(x, y) + k1(x - 1, y))
        south = -0.5 * (k2(x, y - 1) + k1(x - 1, y - 1))
        diag = -(east + west + north + south)
    # keep[k]: candidate k of the row exists -- an interior row keeps a neighbour only if that neighbour is interior
    keep = torch.stack([interior & (iy - 1 > 0), interior & (ix - 1 > 0), torch.ones_like(interior),
                        interior & (ix + 1 < N), interior & (iy + 1 < Ny)], dim=1)
    cols = torch.stack([i - W, i - 1, i, i + 1, i + W], dim=1)
    vals = torch.stack([south, west, torch.where(interior, diag, torch.ones_like(diag)), east, north], dim=1)
    indptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    torch.cumsum(keep.sum(dim=1), 0, out=indptr[1:])
    if int(indptr[-1].item()) >= 2 ** 31:
        raise OverflowError("nnz does not fit int32")
    return DevCSR((n, n), indptr.to(torch.int32), cols[keep].to(torch.int32), vals[keep].contiguous())


def _neumann_laplacian_2d(torch, dev, N, coefficient, Ny):
    """the closed form of problems.neumann_stencil_2d: five candidate entries per row, those outside the grid removed"""
    from .problems import neumann_stencil_2d
    W, n, i, ix, iy = _grid(torch, dev, N, Ny)
    h = 1.0 / N
    if coefficient is None:
        def kf(x, y):
            return torch.ones_like(x)
    else:
        def kf(x, y):
            return coefficient(torch, x, y)
    x, y = ix.to(torch.float64), iy.to(torch.float64)
    del ix, iy
    vals, exists = neumann_stencil_2d(x, y, float(N), float(Ny),
                                      lambda sx, sy: kf((sx + 2.0 / 3.0) * h, (sy + 1.0 / 3.0) * h),
                                      lambda sx, sy: kf((sx + 1.0 / 3.0) * h, (sy + 2.0 / 3.0) * h), xp=torch)
    keep = torch.stack(exists, dim=1)
    cols = torch.stack([i - W, i - 1, i, i + 1, i + W], dim=1)
    indptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    torch.cumsum(keep.sum(dim=1), 0, out=indptr[1:])
    if int(indptr[-1].item()) >= 2 ** 31:
        raise OverflowError("nnz does not fit int32")
    return DevCSR((n, n), indptr.to(torch.int32), cols[keep].to(torch.int32), torch.stack(vals, dim=1)[keep].contiguous())


def structured_rhs_2d(N, f_value=-1.0, Ny=None, device=None):
    """problems.structured_rhs_2d as a device vector (n,)"""
    torch = _lib.require_cuda()
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    Ny = N if Ny is None else int(Ny)
    W, n, i, ix, iy = _grid(torch, dev, N, Ny)
    h = 1.0 / N
    interior = (ix > 0) & (ix < N) & (iy > 0) & (iy < Ny)
    out = torch.zeros(n, dtype=torch.float64, device=dev)
    out[interior] = f_value * h * h
    return out


def linear_P_2d(Nf, Nyf=None, device=None):
    """problems.linear_P_2d as a DevCSR"""
    torch = _lib.require_cuda()
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    Nyf = Nf if Nyf is None else int(Nyf)
    if Nf % 2 or Nyf % 2:
        raise ValueError("Nf must be even")
    Wf, nf, i, ix, iy = _grid(torch, dev, Nf, Nyf)
    Wc = Nf // 2 + 1
    nc = Wc * (Nyf // 2 + 1)
    cx, cy = torch.div(ix, 2, rounding_mode="floor"), torch.div(iy, 2, rounding_mode="floor")
    ox, oy = ix - 2 * cx, iy - 2 * cy
    two = (ox + oy) > 0
    indptr = torch.zeros(nf + 1, dtype=torch.int64, device=dev)
    torch.cumsum(torch.where(two, 2, 1), 0, out=indptr[1:])
    nnz = int(indptr[-1].item())
    indices = torch.empty(nnz, dtype=torch.int32, device=dev)
    data = torch.empty(nnz, dtype=torch.float64, device=dev)
    first = cy * Wc + cx
    second = (cy + oy) * Wc + (cx + ox)
    indices[indptr[:-1]] = first.to(torch.int32)
    data[indptr[:-1]] = torch.where(two, 0.5, 1.0).to(torch.float64)
    t = torch.nonzero(two).reshape(-1)
    indices[indptr[t] + 1] = second[t].to(torch.int32)
    data[indptr[t] + 1] = 0.5
    return DevCSR((nf, nc), indptr.to(torch.int32), indices, data)


def structured_hierarchy_2d(N, levels, Ny=None, device=None):
    """[Q_0, ..., Q_{levels-2}] (linear interpolation) for the nested structured meshes N, N/2, ... as DevCSR"""
    qs = []
    n, ny = N, (N if Ny is None else int(Ny))
    for _ in range(levels - 1):
        if n % 2 or n < 2 or ny % 2 or ny < 2:
            raise ValueError("mesh cannot be coarsened %d times" % (levels - 1))
        qs.append(linear_P_2d(n, Nyf=ny, device=device))
        n //= 2
        ny //= 2
    return qs
