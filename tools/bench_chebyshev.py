"""Multicolour Gauss-Seidel against the Chebyshev smoother (degrees 2 and 3), all V(1,1), on one GPU.

    python tools/bench_chebyshev.py [--configs c8193,v8193,q4097,nn1025] [--reps 30] [--out FILE]

For each configuration and smoother one JSON line: ms per step (CUDA events around graph replays of one V-cycle,
median of --reps after warm-up), launches per cycle, the convergence factor (geometric mean of the residual ratios
over cycles 5-15 from a seeded random start), ms per decade of residual reduction, the setup split (colouring vs
Lanczos bounds) and, on the variable-coefficient problem, MG-preconditioned CG iterations to 1e-10 (on the operator
with its Dirichlet couplings eliminated symmetrically).  The GPU's name and power limit go with every line.  The
problems are bench.build_problem's.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {
    "c8193": dict(n=8192, levels=6, transfer="linear", mesh="structured", coefficient="constant"),
    "v8193": dict(n=8192, levels=6, transfer="linear", mesh="structured", coefficient="variable"),
    "q4097": dict(n=4096, levels=6, transfer="quasi", mesh="structured", coefficient="constant"),
    "nn1025": dict(n=1024, levels=4, transfer="nn", mesh="irregular", coefficient="constant"),
}
SMOOTHERS = [("mcgs", None), ("chebyshev", 2), ("chebyshev", 3)]


def gpu_info(torch):
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    return name, pl


def build(A, Qs, kind, degree):
    from learnmultigrid_b200.engine import DeviceHierarchy
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    kw = {"cheby_degree": degree} if kind == "chebyshev" else {}
    h = DeviceHierarchy(A, Qs, smoother=kind, keep_host=False, **kw)
    torch.cuda.synchronize()
    return h, time.perf_counter() - t0


def time_steps(h, params, reps, warmup=5):
    import torch
    for _ in range(warmup):
        h.vcycle(params)
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        h.vcycle(params)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), h.last_launches


def convergence(h, params, rhs, n):
    x0 = np.random.default_rng(12345).standard_normal(n)
    h.set_rhs(rhs)
    h.set_x(x0)
    res = [h.residual_norm()]
    for _ in range(15):
        h.vcycle(params)
        res.append(h.residual_norm())
    return float((res[15] / res[5]) ** (1.0 / 10.0)), res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default=",".join(CONFIGS))
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import bench
    from learnmultigrid_b200 import problems as P
    name, plimit = gpu_info(torch)
    out = open(a.out, "w") if a.out else None
    for cname in a.configs.split(","):
        cfg = CONFIGS[cname]
        args = types.SimpleNamespace(**cfg)
        A, rhs, Qs = bench.build_problem(args, cfg["n"])
        n = A.shape[0]
        for kind, degree in SMOOTHERS:
            h, setup_s = build(A, Qs, kind, degree)
            params = h.make_params(nu_pre=1, nu_post=1, omega=2.0 / 3.0)
            factor, _ = convergence(h, params, rhs, n)
            ms, launches = time_steps(h, params, a.reps)
            phases = getattr(h, "setup_timing", None) or {}
            rec = {"config": cname, "rows": n, "levels": cfg["levels"], "transfer": cfg["transfer"],
                   "coefficient": cfg["coefficient"], "smoother": kind if degree is None else "chebyshev-%d" % degree,
                   "cycle": "V(1,1)", "ms_per_step": round(ms, 4), "launches_per_cycle": launches,
                   "convergence_factor": round(factor, 4),
                   "ms_per_decade": round(ms / -np.log10(factor), 4) if 0 < factor < 1 else None,
                   "setup_s": round(setup_s, 3), "colouring_s": round(phases.get("colouring", 0.0), 3),
                   "lanczos_s": round(phases.get("Chebyshev bounds (Lanczos)", 0.0), 3),
                   "cheby_lambda": None if h.cheby_lambda is None else [round(v, 6) for v in h.cheby_lambda],
                   "timing": "CUDA events around one graph replay, median of %d after 5 warm-up replays" % a.reps,
                   "gpu": name, "power_limit": plimit}
            del h
            torch.cuda.empty_cache()
            if cname == "v8193":
                As = P.symmetric_dirichlet(A, P.boundary_nodes_2d(cfg["n"]))
                hs, _ = build(As, Qs, kind, degree)
                ps = hs.make_params(nu_pre=1, nu_post=1, reverse_post=kind == "mcgs")
                _, track, its = hs.pcg(rhs, ps, error=1e-10, max_iterations=200)
                rec["pcg_iterations_to_1e-10"] = its
                rec["pcg_final_residual"] = float(track[-1])
                del hs
                torch.cuda.empty_cache()
            line = json.dumps(rec)
            print(line, flush=True)
            if out:
                out.write(line + "\n")
                out.flush()


if __name__ == "__main__":
    main()
