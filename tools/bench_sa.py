"""Smoothed aggregation (SmoothedAggregationMG's device-built transfer operators) against classical AMG and the
project's supplied hierarchies, one GPU, in the same run.

    python tools/bench_sa.py [--configs c4097,v8193,nn1025] [--reps 30] [--out FILE]

    c4097   4097^2 constant coefficient: SA (4 levels), AMG (6 levels), linear_P_2d (6 levels), V(1,1) multicolour GS
    v8193   8193^2 variable coefficient: SA (4 levels), AMG (7 levels), linear_P_2d (6 levels), V(1,1) multicolour GS,
            plus PCG to 1e-10 on the operator with its Dirichlet couplings eliminated symmetrically (each arm builds its
            own hierarchy for that operator)
    nn1025  1025^2 irregular mesh: SA (3 levels), AMG (4 levels), the NN builder with MassSurrogate (4 levels), V(3,3)

The SA level counts stop the coarsening near the coarsest size of the other arms: SA coarsens the 5-point operators by
~5.5x on the fine level and ~14x below (the irregular mesh by ~9x and ~15x), against ~2.7x / 4x for PMIS and 4x for the
structured meshes.  One JSON line per arm, with the fields of tools/bench_amg.py: ms per step (CUDA events around one
graph replay, median of --reps after warm-up), launches per cycle, convergence factor (cycles 5-15 from a seeded random
start), ms per decade, rows and complexities per level, the setup split per level (SA: strength / MIS(2) / aggregation /
smoothing / Galerkin in ms, MIS(2) rounds, isolated points, lambda_max, omega_eff), and the GPU's name and power limit.
"""
import argparse
import json
import os
import sys
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_amg import CONFIGS as AMG_CONFIGS, amg_transfers, convergence, gpu_info, hierarchy, time_steps  # noqa: E402

SA_LEVELS = {"c4097": 4, "v8193": 4, "nn1025": 3}


def sa_transfers(A, levels):
    import torch
    from learnmultigrid_b200 import formats as F
    from learnmultigrid_b200.sa import SaBuilder
    b = SaBuilder()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    Ps = b.define_hierarchy(F.canonical_csr(A), levels)
    torch.cuda.synchronize()
    gc, oc = b.complexities()
    info = {"sa_setup_s": round(time.perf_counter() - t0, 3), "grid_complexity": round(gc, 4),
            "operator_complexity": round(oc, 4), "sa_levels": b.stats}
    return Ps, info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default=",".join(SA_LEVELS))
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import bench
    from learnmultigrid_b200 import problems as P
    name, plimit = gpu_info(torch)
    sa_transfers(P.structured_laplacian_2d(64), 3)       # load the kernels before any setup split is timed
    amg_transfers(P.structured_laplacian_2d(64), 3)
    builders = {"sa": sa_transfers, "amg": amg_transfers}
    out = open(a.out, "w") if a.out else None
    for cname in a.configs.split(","):
        cfg = AMG_CONFIGS[cname]
        A, rhs, Q_ref = bench.build_problem(types.SimpleNamespace(**cfg), cfg["n"])
        n = A.shape[0]
        arms = [("sa", SA_LEVELS[cname]), ("amg", cfg["amg_levels"]), (cfg["transfer"], cfg["levels"])]
        for arm, levels in arms:
            info = {}
            if arm in builders:
                Qs, info = builders[arm](A, levels)
            else:
                Qs = Q_ref
            h, setup_s = hierarchy(A, Qs)
            params = h.make_params(nu_pre=cfg["nu"], nu_post=cfg["nu"])
            factor = convergence(h, params, rhs, n)
            ms, launches = time_steps(h, params, a.reps)
            rows = [lv.n for lv in h.levels]
            nnz = [lv.nnz_A for lv in h.levels]
            rec = {"config": cname, "arm": arm, "rows": n, "levels": levels, "coefficient": cfg["coefficient"],
                   "mesh": cfg["mesh"], "cycle": "V(%d,%d)" % (cfg["nu"], cfg["nu"]), "smoother": "mcgs",
                   "level_rows": rows, "ms_per_step": round(ms, 4), "launches_per_cycle": launches,
                   "convergence_factor": round(factor, 4),
                   "ms_per_decade": round(ms / -np.log10(factor), 4) if 0 < factor < 1 else None,
                   "hierarchy_setup_s": round(setup_s, 3),
                   "grid_complexity": round(sum(rows) / rows[0], 4),
                   "operator_complexity": round(sum(nnz) / nnz[0], 4)}
            rec.update(info)
            del h
            torch.cuda.empty_cache()
            if cname == "v8193":
                As = P.symmetric_dirichlet(A, P.boundary_nodes_2d(cfg["n"]))
                Qp = builders[arm](As, levels)[0] if arm in builders else Qs
                hs, _ = hierarchy(As, Qp)
                ps = hs.make_params(nu_pre=1, nu_post=1, reverse_post=True)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                _, track, its = hs.pcg(rhs, ps, error=1e-10, max_iterations=200)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                rec["pcg_iterations_to_1e-10"] = its
                rec["pcg_final_residual"] = float(track[-1])
                rec["pcg_ms_total"] = round(dt * 1e3, 2)
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
