"""Classical AMG (AlgebraicMG's device-built transfer operators) against the project's other hierarchies, one GPU.

    python tools/bench_amg.py [--configs c4097,v8193,nn1025] [--reps 30] [--out FILE]

    c4097   4097^2 constant coefficient: AMG (6 levels) vs linear_P_2d (6 levels), V(1,1) multicolour GS
    v8193   8193^2 variable coefficient: AMG (7 levels) vs linear_P_2d (6 levels), V(1,1) multicolour GS, plus PCG to
            1e-10 on the operator with its Dirichlet couplings eliminated symmetrically (each arm builds its own
            hierarchy for that operator)
    nn1025  1025^2 irregular mesh: AMG vs the NN builder with MassSurrogate, both 4 levels, V(3,3) multicolour GS

The AMG level counts stop the coarsening near the coarsest size of the structured hierarchies (PMIS coarsens by ~2.7x
on the fine level and ~4x below, against 4x per level for the structured meshes).  One JSON line per arm: ms per step
(CUDA events around one graph replay, median of --reps after warm-up; the 4097^2 and 8193^2 fine levels are larger
than the 126 MB L2, the 1025^2 irregular hierarchy fits in it),
launches per cycle, convergence factor (geometric mean of the residual ratios over cycles 5-15 from a seeded random
start), ms per decade, the hierarchy's rows and complexities and, for AMG, the setup split per level (strength / PMIS /
interpolation / Galerkin, ms), PMIS rounds and promoted points.  DeviceHierarchy forms the Galerkin products again from
the same Q list; its time is reported as galerkin_in_hierarchy_ms.  The GPU's name and power limit go with every line.
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
    "c4097": dict(n=4096, levels=6, amg_levels=6, transfer="linear", mesh="structured", coefficient="constant", nu=1),
    "v8193": dict(n=8192, levels=6, amg_levels=7, transfer="linear", mesh="structured", coefficient="variable", nu=1),
    "nn1025": dict(n=1024, levels=4, amg_levels=4, transfer="nn", mesh="irregular", coefficient="constant", nu=3),
}


def gpu_info(torch):
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    return name, pl


def amg_transfers(A, levels):
    import torch
    from learnmultigrid_b200 import formats as F
    from learnmultigrid_b200.amg import AmgBuilder
    b = AmgBuilder()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    Qs = b.define_hierarchy(F.canonical_csr(A), levels)
    torch.cuda.synchronize()
    gc, oc = b.complexities()
    info = {"amg_setup_s": round(time.perf_counter() - t0, 3), "grid_complexity": round(gc, 4),
            "operator_complexity": round(oc, 4), "amg_levels": b.stats}
    return Qs, info


def hierarchy(A, Qs):
    import torch
    from learnmultigrid_b200.engine import DeviceHierarchy
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    h = DeviceHierarchy(A, Qs, smoother="mcgs", keep_host=False)
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
    h.set_rhs(rhs)
    h.set_x(np.random.default_rng(12345).standard_normal(n))
    res = [h.residual_norm()]
    for _ in range(15):
        h.vcycle(params)
        res.append(h.residual_norm())
    return float((res[15] / res[5]) ** (1.0 / 10.0))


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
    amg_transfers(P.structured_laplacian_2d(64), 3)       # load the kernels before any setup split is timed
    out = open(a.out, "w") if a.out else None
    for cname in a.configs.split(","):
        cfg = CONFIGS[cname]
        A, rhs, Q_ref = bench.build_problem(types.SimpleNamespace(**cfg), cfg["n"])
        n = A.shape[0]
        arms = [("amg", cfg["amg_levels"]), (cfg["transfer"], cfg["levels"])]
        for arm, levels in arms:
            info = {}
            if arm == "amg":
                Qs, info = amg_transfers(A, levels)
            else:
                Qs = Q_ref
            h, setup_s = hierarchy(A, Qs)
            params = h.make_params(nu_pre=cfg["nu"], nu_post=cfg["nu"])
            factor = convergence(h, params, rhs, n)
            ms, launches = time_steps(h, params, a.reps)
            phases = getattr(h, "setup_timing", None) or {}
            rec = {"config": cname, "arm": arm, "rows": n, "levels": levels, "coefficient": cfg["coefficient"],
                   "mesh": cfg["mesh"], "cycle": "V(%d,%d)" % (cfg["nu"], cfg["nu"]), "smoother": "mcgs",
                   "level_rows": [lv.n for lv in h.levels], "ms_per_step": round(ms, 4),
                   "launches_per_cycle": launches, "convergence_factor": round(factor, 4),
                   "ms_per_decade": round(ms / -np.log10(factor), 4) if 0 < factor < 1 else None,
                   "hierarchy_setup_s": round(setup_s, 3),
                   "galerkin_in_hierarchy_ms": round(phases.get("Galerkin SpGEMM", 0.0) * 1e3, 1)}
            rec.update(info)
            if arm != "amg":
                nnz = [h.levels[0].nnz_A] + [lv.nnz_A for lv in h.levels[1:]]
                rows = [lv.n for lv in h.levels]
                rec["grid_complexity"] = round(sum(rows) / rows[0], 4)
                rec["operator_complexity"] = round(sum(nnz) / nnz[0], 4)
            del h
            torch.cuda.empty_cache()
            if cname == "v8193":
                As = P.symmetric_dirichlet(A, P.boundary_nodes_2d(cfg["n"]))
                Qp = amg_transfers(As, levels)[0] if arm == "amg" else Qs
                hs, _ = hierarchy(As, Qp)
                ps = hs.make_params(nu_pre=1, nu_post=1, reverse_post=True)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                _, track, its = hs.pcg(rhs, ps, error=1e-10, max_iterations=200)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                rec["pcg_iterations_to_1e-10"] = its
                rec["pcg_final_residual"] = float(track[-1])
                rec["pcg_ms_per_iteration"] = round(dt * 1e3 / max(its, 1), 4)
                del hs, Qp
                torch.cuda.empty_cache()
            rec["timing"] = "CUDA events around one graph replay, median of %d after 5 warm-up replays" % a.reps
            rec["gpu"], rec["power_limit"] = name, plimit
            line = json.dumps(rec)
            print(line, flush=True)
            if out:
                out.write(line + "\n")
                out.flush()
            del Qs
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
