"""Pure-Neumann problems on one GPU: the cost of a declared null space and today's behaviour without one.

    python tools/bench_neumann.py [--n 8192] [--levels 6] [--reps 40] [--out FILE]

Problem: the P1 stiffness matrix of -div(k grad u), k = 1 + 0.9 sin(2 pi x) sin(2 pi y), on (n+1)^2 nodes with natural
boundary conditions (problems_device.structured_laplacian_2d(boundary="neumann")), linear transfers, multicolour
Gauss-Seidel V(1,1); with 6 levels the coarsest level is 257^2 and solved by block cyclic reduction.  JSON lines:
  * "step": ms per step (one V-cycle plus the residual norm, CUDA events around graph replays, median over --reps, the
    Neumann hierarchy with null_space="constant" and its Dirichlet twin timed in alternating blocks) and launches per
    step of both;
  * "solve": V-cycles and MG-preconditioned CG iterations to 1e-10 (absolute) from a hashed right-hand side;
  * "coarse_setup": seconds to set up the coarsest solver pinned (null space declared) and unpinned;
  * "no_null_space": 20 cycles on the same Neumann problem built WITHOUT a null space (the plain inverse of a singular
    coarsest operator), residual history and the largest entry of the coarse solution.
The GPU's name and power limit go with every line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(torch):
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    return name, pl


def step_ms(torch, h, params, reps):
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        h.vcycle(params, with_norm=True)
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return ms


def rhs(torch, h, n):
    from learnmultigrid_b200 import formats as F
    v = F.chebyshev_start_vector(torch.arange(n, dtype=torch.int64, device=h.device)) * 1e-3
    return v.contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=8192)
    ap.add_argument("--levels", type=int, default=6)
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from learnmultigrid_b200 import problems_device as PD
    from learnmultigrid_b200.coarse import build_coarse_solver
    from learnmultigrid_b200.engine import DeviceHierarchy
    torch.cuda.set_device(0)
    name, plimit = gpu_info(torch)
    N, L = args.n, args.levels
    out = open(args.out, "a") if args.out else None

    def emit(d):
        d.update({"n": N, "levels": L, "gpu": name, "power_limit": plimit})
        line = json.dumps(d)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    coef = PD.variable_coefficient
    Qs = PD.structured_hierarchy_2d(N, L)
    hs = {}
    for kind in ("neumann", "dirichlet"):
        A = PD.structured_laplacian_2d(N, coef, boundary=kind)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        hs[kind] = DeviceHierarchy(A, Qs, smoother="mcgs", keep_host=kind == "neumann",      # its coarsest: below
                                   null_space="constant" if kind == "neumann" else None)
        torch.cuda.synchronize()
        hs[kind].setup_s = time.perf_counter() - t0
        del A
    n = hs["neumann"].n
    params = hs["neumann"].make_params(1, 1)
    for kind, h in hs.items():
        h.set_rhs(rhs(torch, h, n))
        h.project_rhs()
        h.zero_x()
        step_ms(torch, h, params, 5)
    times = {k: [] for k in hs}
    for _ in range(4):                      # alternating blocks
        for kind, h in hs.items():
            times[kind] += step_ms(torch, h, params, args.reps // 4)
    emit({"kind": "step", **{"%s_ms" % k: float(np.median(v)) for k, v in times.items()},
          **{"%s_ms_min" % k: float(np.min(v)) for k, v in times.items()},
          **{"%s_launches" % k: int(h.last_launches) for k, h in hs.items()},
          **{"%s_setup_s" % k: h.setup_s for k, h in hs.items()},
          "null_info": hs["neumann"].null_info})

    # cycles and PCG iterations to 1e-10
    h = hs.pop("neumann")
    del hs
    b = rhs(torch, h, n)
    h.set_rhs(b)
    h.project_rhs()
    h.zero_x()
    hist = [h.residual_norm()]
    while hist[-1] > 1e-10 and len(hist) < 60:
        h.vcycle(params, with_norm=True)
        hist.append(h.last_norm())
    _, track, its = h.pcg(b, h.make_params(1, 1, reverse_post=True), error=1e-10, max_iterations=60)
    emit({"kind": "solve", "cycles": len(hist) - 1, "history": hist, "pcg_iterations": its, "pcg_history": track,
          "rhs_null_component": h.rhs_null_component})

    # coarsest setup, pinned and unpinned, on the hierarchy's own coarsest operator
    lev = h.levels[-1]
    Ac = h.level_matrix(L - 1)
    ip, ix, va = (torch.from_numpy(np.ascontiguousarray(a)).to(h.device) for a in (Ac.indptr, Ac.indices, Ac.data))
    setup = {}
    for singular in (True, False, True, False):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        s = build_coarse_solver(torch, h.device, Ac.shape[0], ip, ix, va, 4096, (Ac.indptr, Ac.indices),
                                singular=singular)
        torch.cuda.synchronize()
        setup.setdefault("pinned" if singular else "unpinned", []).append(time.perf_counter() - t0)
        del s
    emit({"kind": "coarse_setup", "rows": int(Ac.shape[0]), "coarse_kind": int(lev.coarse_kind),
          **{k + "_s": min(v) for k, v in setup.items()}})
    del h, lev

    # today's behaviour: the same problem without a declared null space
    from learnmultigrid_b200 import _lib
    A = PD.structured_laplacian_2d(N, coef, boundary="neumann")
    try:
        h = DeviceHierarchy(A, Qs, smoother="mcgs", keep_host=False)
    except _lib.MgError as e:
        emit({"kind": "no_null_space", "error": str(e)})
        return
    del A
    b = rhs(torch, h, n)
    b -= b.mean()                           # a consistent right-hand side (to rounding)
    h.set_rhs(b)
    h.zero_x()
    hist = [h.residual_norm()]
    for _ in range(20):
        h.vcycle(params, with_norm=True)
        hist.append(h.last_norm())
    c = h.levels[-1]
    emit({"kind": "no_null_space", "history": hist, "coarse_x_max": float(c.x.abs().max().item()),
          "x_mean": float(h.levels[0].x.mean().item()), "x_max": float(h.levels[0].x.abs().max().item())})


if __name__ == "__main__":
    main()
