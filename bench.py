#!/usr/bin/env python
"""bench.py -- V-cycle throughput of the B200 multigrid engine (BASELINE.json metric) + roofline + CPU baseline.

    python bench.py --gpus 1 --steps K --warmup W            # our arm
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port) on host cores

A "step" is one outer iteration of Multigrid.solve (learn_multigrid/solvers/Multigrid.py:59-73): fused
residual + 2-norm on the fine level, then one V(nu,nu) cycle over the prebuilt hierarchy.  `value` is fine-grid
DOF per second with everything resident in HBM; `e2e` is the same metric through the reference-facing API
(SemiGeometricMG.solve with host rhs / host solution, H2D and D2H inside the timed region, `cycles_per_solve`
V-cycles per call).  One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "vcycle_fine_grid_dof_per_s"
UNIT = "DOF/s"
DUMP_SAMPLE = 1 << 22          # float64 entries of the iterate written by --dump-outputs: 32 MB


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=int(os.environ.get("MGB_BENCH_N", "8192")),
                    help="elements per side of the structured mesh ((n+1)^2 DOF)")
    ap.add_argument("--levels", type=int, default=int(os.environ.get("MGB_BENCH_LEVELS", "6")))
    ap.add_argument("--transfer", default=os.environ.get("MGB_BENCH_TRANSFER", "linear"), choices=["linear", "quasi", "nn"],
                    help="nn: transfer operators from the mass matrix through NeuralMG_2D.define_hierarchy (device "
                         "builder, mass-surrogate predictor: the reference's trained weights are not shipped)")
    ap.add_argument("--mesh", default=os.environ.get("MGB_BENCH_MESH", "structured"), choices=["structured", "irregular"],
                    help="irregular: Mesh2D((n/2)^2) + one irregular red refinement, parents numbered first (configs[1])")
    ap.add_argument("--smoother", default=os.environ.get("MGB_BENCH_SMOOTHER", "GaussSeidel"),
                    choices=["GaussSeidel", "Jacobi"])
    ap.add_argument("--nu", type=int, default=1)
    ap.add_argument("--coefficient", default="constant", choices=["constant", "variable", "variable-symmetric"],
                    help="variable: k = 1 + 0.9 sin(2 pi x) sin(2 pi y) (BASELINE configs[3]); variable-symmetric: the same "
                         "with the Dirichlet couplings eliminated symmetrically (the operator of the PCG configuration; "
                         "device generation only)")
    ap.add_argument("--cycles-per-solve", type=int, default=10)
    ap.add_argument("--cpu-n", type=int, default=2048,
                    help="mesh size of the bounded CPU sample (SURVEY 8d: <= 4 M DOF measured, the rest labelled extrapolated)")
    ap.add_argument("--setup", default=os.environ.get("MGB_BENCH_SETUP", "device"), choices=["host", "device"])
    ap.add_argument("--generate", default=os.environ.get("MGB_BENCH_GENERATE", "device"), choices=["device", "host"],
                    help="device (default; structured meshes with linear transfers): the synthetic operator and transfer "
                         "operators are generated in HBM (problems_device.py) instead of in NumPy + upload")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip config.extra: the variable-coefficient V-cycle (BASELINE configs[3]) and the MG-preconditioned "
                         "CG solve to 1e-10 (configs[4]) measured in the same run after the headline")
    ap.add_argument("--no-parity-check", action="store_true",
                    help="N > 1: skip the small partitioned-vs-single-GPU bit-identity check run before the benchmark")
    ap.add_argument("--profile-step", action="store_true",
                    help="bracket ONE extra step with cudaProfilerStart/Stop (ncu --profile-from-start off)")
    ap.add_argument("--multi", default=os.environ.get("MGB_BENCH_MULTI", "partitioned"),
                    choices=["partitioned", "replicas"],
                    help="N>1: row-partition ONE problem over the GPUs (strong scaling, SURVEY 8e) or run N replicas")
    ap.add_argument("--colors", default=os.environ.get("MGB_BENCH_COLORS", "greedy"), choices=["structured", "greedy", "lattice"],
                    help="greedy (default, at every GPU count): first-fit colouring of the matrix graph, 2 colours on the "
                         "5-point level and 4 on the 7-point Galerkin levels; structured: (ix+iy)%%2 / %%3 (linear "
                         "transfers only) -- one launch and one exchange site fewer per coarse sweep (3%% faster per "
                         "cycle at 8 GPUs) but a worse smoother: V(1,1) convergence factor 0.23 instead of 0.20 "
                         "(profiles/r01_convergence_factors.txt), so it loses on time to solution")
    ap.add_argument("--min-rows-per-rank", type=int, default=int(os.environ.get("MGB_MIN_ROWS", "65536")))
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR as float64 .npy files: "
                         "solution.npy (the fine-grid iterate, or a fixed seeded sample of %d of its entries) and "
                         "residual_norm.npy (the residual norm that step computed); the inputs depend on the arguments "
                         "only, so two builds can be compared output for output" % DUMP_SAMPLE)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def dump_outputs(path, solution, residual_norm):
    """--dump-outputs: the iterate (all of it up to DUMP_SAMPLE entries, otherwise the entries at a fixed seeded sample
    of indices in increasing order) and the residual norm, as float64 .npy files under `path`."""
    x = np.asarray(solution, dtype=np.float64).reshape(-1)
    if x.size > DUMP_SAMPLE:
        x = x[np.sort(np.random.default_rng(0).choice(x.size, DUMP_SAMPLE, replace=False))]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "solution.npy"), x)
    np.save(os.path.join(path, "residual_norm.npy"), np.array([residual_norm], dtype=np.float64))


def workload_name(a, n):
    return "2D %s P1 %s %dx%d grid (%d DOF), %d-level V(%d,%d), %s, %s transfers" % (
        "structured" if a.mesh == "structured" else "irregularly refined (unstructured numbering)",
        "Laplacian" if a.coefficient == "constant" else "variable-coefficient stiffness" + (
            " (Dirichlet couplings eliminated symmetrically)" if a.coefficient == "variable-symmetric" else ""), n + 1, n + 1,
        (n + 1) ** 2, a.levels, a.nu, a.nu,
        ("multicolour Gauss-Seidel (greedy colouring)" if a.mesh == "irregular" else
         "multicolour (red-black on the fine level) Gauss-Seidel") if a.smoother == "GaussSeidel" else "damped Jacobi (omega=2/3)",
        a.transfer)


class ClockSampler:
    """SM clock / throttle reasons sampled through NVML from a thread DURING the timed regions."""

    def __init__(self, index=0, period=0.005):
        self.index, self.period = index, period
        self.samples = []
        self.on = False
        self.ok = False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.ok = True
        except Exception as e:   # pragma: no cover
            self.err = repr(e)
            return
        self.on = True
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        while self.on:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                self.samples.append((time.perf_counter(), sm, rs, pw))
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self, windows=None):
        """windows: list of (t0, t1) perf_counter intervals that count as 'under load'"""
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self.on = False
        self.t.join(timeout=1)
        nv = self.nv
        smax = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        sel = [s for s in self.samples if windows is None or any(a <= s[0] <= b for a, b in windows)]
        if not sel:
            sel = self.samples
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                "hw_power_brake": 0x80}
        reasons = sorted(k for k, m in bits.items() if any(s[2] & m for s in sel))
        return {"sm_mhz": float(np.median([s[1] for s in sel])) if sel else None, "sm_max_mhz": float(smax),
                "power_w_max": max(s[3] for s in sel) if sel else None, "samples_under_load": len(sel),
                "samples": len(self.samples), "reasons": reasons}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


NN_BUILD = {}


def build_problem(a, n):
    from learnmultigrid_b200 import problems as P
    if a.mesh == "irregular" or a.transfer == "nn":
        if a.mesh != "irregular" or a.transfer != "nn":
            raise SystemExit("--mesh irregular and --transfer nn go together (BASELINE configs[1])")
        from learnmultigrid_b200.neural2d import MassSurrogate
        from learnmultigrid_b200.solvers.Multigrid import NeuralMG_2D
        pb = P.irregular_p1_2d(n, seed=42)
        asm_ms = None
        try:                         # the same operators by the device assembler, timed (informational)
            import torch
            from learnmultigrid_b200.assembly_device import DeviceAssembler
            from learnmultigrid_b200.assembly.LoadFunction import LoadFunction
            from learnmultigrid_b200.assembly.Quadrature import Quadrature2D
            from learnmultigrid_b200.assembly.ShapeFunction import FunctionTriangle, GradientTriangle
            asm = DeviceAssembler()
            q = Quadrature2D(3)
            for rep in range(2):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                m = asm.mesh_to_device(pb["mesh"])
                Ad = asm.stiffness(*m, GradientTriangle(1), q)
                Md = asm.mass(*m, FunctionTriangle(1), q)
                bd = asm.load(*m, LoadFunction(lambda pts: -1.0), FunctionTriangle(1), q)
                Ad = asm.dirichlet(Ad, pb["boundary"], bd)
                torch.cuda.synchronize()
                asm_ms = (time.perf_counter() - t0) * 1e3
            assert Ad.nnz == pb["A"].nnz and Md.nnz == pb["M"].nnz
            del Ad, Md, bd, asm
        except ImportError:
            pass
        nmg = NeuralMG_2D(pb["A"], pb["rhs"], MassSurrogate(), pb["M"], np.ones(43), np.zeros(43))
        t0 = time.perf_counter()
        nmg.define_hierarchy(a.levels)
        NN_BUILD[n] = {"define_hierarchy_s": round(time.perf_counter() - t0, 3), "device_assembly_A_M_rhs_ms": asm_ms,
                       "coarse_nodes": [int(q.shape[1]) for q in nmg.l_hierarchy],
                       "nnz_Q": [int(q.nnz) for q in nmg.l_hierarchy]}
        return pb["A"], pb["rhs"], nmg.l_hierarchy
    coef = None if a.coefficient == "constant" else P.variable_coefficient
    A = P.structured_laplacian_2d(n, coef)
    if a.coefficient == "variable-symmetric":
        A = P.symmetric_dirichlet(A, P.boundary_nodes_2d(n))
    rhs = P.structured_rhs_2d(n)
    Qs = P.structured_hierarchy_2d(n, a.levels, transfer=a.transfer)
    return A, rhs, Qs


# ------------------------------------------------------------------------------------------------------------
def cpu_cycle_rate(a, n, reference_style, budget_s=25.0, max_cycles=10):
    """DOF/s of the oracle V-cycle (SciPy SpMV / transfers, PyAMG Gauss-Seidel kernel restated in C, SciPy
    Galerkin, SuperLU) on one host core.  reference_style=True repeats the Galerkin products and the coarse
    factorisation in every cycle exactly as the reference does (Multigrid.py:97-98,106)."""
    from oracle.vcycle import OracleMultigrid
    A, rhs, Qs = build_problem(a, n)
    sm = "gs" if a.smoother == "GaussSeidel" else "jacobi"
    o = OracleMultigrid(A, rhs, Qs, smoother=sm, omega=2.0 / 3.0, hoist_setup=not reference_style)
    t_setup = 0.0
    if not reference_style:
        t0 = time.perf_counter()
        o.build_hierarchy(a.levels)
        t_setup = time.perf_counter() - t0
    x = np.zeros_like(rhs)
    Af = o.matrix
    times = []
    t_begin = time.perf_counter()
    for _ in range(max_cycles):
        t0 = time.perf_counter()
        r = rhs - Af.dot(x)
        np.linalg.norm(r)
        x = o.v_cycle(Af, x, rhs, a.nu, a.levels)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_begin > budget_s:
            break
    per = float(np.median(times))
    return (n + 1) ** 2 / per, per, len(times), t_setup


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = a.cpu_n
    times = []
    # each step = one reference-style V-cycle iteration on the bounded sample
    from oracle.vcycle import OracleMultigrid
    A, rhs, Qs = build_problem(a, n)
    sm = "gs" if a.smoother == "GaussSeidel" else "jacobi"
    o = OracleMultigrid(A, rhs, Qs, smoother=sm, omega=2.0 / 3.0, hoist_setup=False)
    x = np.zeros_like(rhs)
    Af = o.matrix
    for it in range(a.warmup + a.steps):
        t0 = time.perf_counter()
        r = rhs - Af.dot(x)
        res = np.linalg.norm(r)
        x = o.v_cycle(Af, x, rhs, a.nu, a.levels)
        dt = time.perf_counter() - t0
        if it >= a.warmup:
            times.append(dt)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, x, res)
    per = float(np.mean(times))
    val = (n + 1) ** 2 / per
    sample = ("%dx%d grid (%d DOF) of the same %d-level V(%d,%d) configuration, %d timed cycles, Galerkin products "
              "and coarse LU repeated in every cycle as the reference does") % (n + 1, n + 1, (n + 1) ** 2, a.levels,
                                                                                   a.nu, a.nu, len(times))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": len(times),
            "warmup": a.warmup, "ms_per_step": per * 1e3, "higher_is_better": True,
            "scaling": "strong" if a.multi == "partitioned" else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(a, a.n), "sample": sample,
                       "smoother": ("index-order Gauss-Seidel (PyAMG's sweep restated in C: what the reference runs whatever "
                                    "`smoother` says, Multigrid.py:88,121)" if a.smoother == "GaussSeidel" else "damped Jacobi")},
            "extrapolated": n != a.n,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample,
                             "extrapolated": n != a.n},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def multi_rank_parity(torch, dist, fab, a):
    """N > 1: the partitioned cycle (real ranks, real NVLink exchanges) against the single-GPU cycle every rank also
    runs, on a small problem of the same kind: iterates must agree bit for bit, norms to rounding.  Returns a dict for
    `config` (the driver's scaling run then carries multi-process parity)."""
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.distributed import DistributedHierarchy
    from learnmultigrid_b200.engine import DeviceHierarchy
    N, levels, cycles = 512, 5, 3
    coef = P.variable_coefficient if a.coefficient == "variable" else None
    A = P.structured_laplacian_2d(N, coef)
    Qs = P.structured_hierarchy_2d(N, levels, transfer="linear")
    rng = np.random.default_rng(11)
    n = A.shape[0]
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    h1 = DeviceHierarchy(A, Qs, smoother="mcgs")
    hd = DistributedHierarchy(A, Qs, fab, smoother="mcgs", colors=h1.colors, n_dist=3, timeout_s=30.0)
    for h in (h1, hd):
        h.set_rhs(b)
        h.set_x(x0)
    p1, pd = h1.make_params(nu_pre=a.nu, nu_post=a.nu), hd.make_params(nu_pre=a.nu, nu_post=a.nu)
    same, close = True, True
    for _ in range(cycles):
        h1.vcycle(p1, with_norm=True)
        hd.vcycle(pd, norm_after=True)
        n1, nd = h1.last_norm(), hd.last_norm()
        o0, o1 = int(hd.offsets[0][fab.rank]), int(hd.offsets[0][fab.rank + 1])
        same = same and np.array_equal(h1.get_x()[o0:o1], hd.get_x_local())
        close = close and abs(n1 - nd) <= 1e-12 * n1
    hd.check()
    t = torch.tensor([1 if same else 0, 1 if close else 0], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    hd.close()
    del h1, hd
    torch.cuda.empty_cache()
    return {"problem": "%dx%d grid, %d levels (3 partitioned), V(%d,%d), %d cycles, every rank vs its own single-GPU cycle"
                       % (N + 1, N + 1, levels, a.nu, a.nu, cycles),
            "iterates_bit_identical": bool(int(t[0].item())), "norms_equal_to_1e-12": bool(int(t[1].item()))}


def extra_configs(torch, dist, a, n, Qs, rhs, fab, world, rank):
    """config.extra: BASELINE configs[3] and [4] on the same grid, same run, same GPU count -- the variable-coefficient
    operator k = 1 + 0.9 sin(2 pi x) sin(2 pi y) with its Dirichlet couplings eliminated symmetrically: (a) the V-cycle
    step, (b) hierarchy setup and conjugate gradients preconditioned by one symmetric V(1,1) cycle per iteration down
    to ||r||_2 <= 1e-10.  Informational: measured after the headline, never allowed to cost it."""
    from learnmultigrid_b200 import problems_device as PD
    from learnmultigrid_b200.engine import DeviceHierarchy
    def build(symmetric):
        t0 = time.perf_counter()
        A2 = PD.structured_laplacian_2d(n, PD.variable_coefficient, symmetric=symmetric)
        torch.cuda.synchronize()
        t_gen = time.perf_counter() - t0
        t0 = time.perf_counter()
        if fab is not None:
            from learnmultigrid_b200.distributed import DistributedHierarchy
            hh = DistributedHierarchy(A2, Qs, fab, smoother="mcgs", min_rows_per_rank=a.min_rows_per_rank, timeout_s=30.0)
        else:
            hh = DeviceHierarchy(A2, Qs, smoother="mcgs")
        torch.cuda.synchronize()
        return hh, t_gen, time.perf_counter() - t0

    h2, t_gen, t_setup = build(False)
    params = h2.make_params(nu_pre=a.nu, nu_post=a.nu)
    h2.set_rhs(rhs)
    h2.zero_x()

    def step():
        if fab is not None:
            h2.vcycle(params, norm_after=True)
        else:
            h2.vcycle(params, with_norm=True)
    for _ in range(3):
        step()
    h2.zero_x()
    torch.cuda.synchronize()
    if fab is not None:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.steps
    if fab is not None:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ndof = (n + 1) ** 2
    out = {"variable_coefficient_vcycle": {
        "workload": "BASELINE configs[3]: variable-coefficient stiffness, same grid / levels / smoother",
        "ms_per_step": ms, "dof_per_s": ndof / (ms * 1e-3),
        "generate_s": round(t_gen, 2), "setup_s": round(t_setup, 2),
        "setup_phases_s": {k: round(v, 3) for k, v in (getattr(h2, "setup_timing", None) or {}).items()},
        "setup_galerkin_per_level": getattr(h2, "setup_galerkin", None),
        "value_dictionary_on_A": getattr(h2.levels[0].A, "val_idx", None) is not None}}
    if fab is not None:
        h2.close()
    del h2
    torch.cuda.empty_cache()
    h2, t_gen, t_setup = build(True)            # conjugate gradients need the symmetrically eliminated operator
    psym = h2.make_params(nu_pre=1, nu_post=1, reverse_post=True)
    pin = torch.from_numpy(np.ascontiguousarray(rhs.reshape(-1))).pin_memory()
    h2.pcg(pin, psym, error=0.0, max_iterations=2)                      # warm-up: graph capture
    torch.cuda.synchronize()
    if fab is not None:
        dist.barrier()
    t0 = time.perf_counter()
    _, hist, its = h2.pcg(pin, psym, error=1e-10, max_iterations=100, view=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    tm = h2.last_pcg_timing
    if fab is not None:
        t = torch.tensor([dt, tm["iterations_s"]], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt, it_s = float(t[0].item()), float(t[1].item())
        h2.check()
    else:
        it_s = tm["iterations_s"]
    out["mg_preconditioned_cg"] = {
        "workload": "BASELINE configs[4]: CG preconditioned by one symmetric V(1,1) cycle per iteration to ||r||_2 <= 1e-10, "
                    "scalars on the device, one CUDA graph per iteration", "iterations": its, "final_residual": hist[-1],
        "ms_per_iteration": it_s * 1e3 / max(its, 1), "solve_ms": dt * 1e3,
        "solve_split_ms": {"rhs_host_to_device": tm["transfer_in_s"] * 1e3, "iterations": it_s * 1e3,
                           "solution_device_to_host": tm["transfer_out_s"] * 1e3},
        "dof_per_s_to_tolerance": ndof / dt, "hierarchy_setup_s": round(t_setup, 2)}
    if fab is not None:
        h2.close()
    return out


# ------------------------------------------------------------------------------------------------------------
def run_b200(a):
    import torch
    import torch.distributed as dist
    from learnmultigrid_b200 import _lib
    from learnmultigrid_b200.solvers.Multigrid import SemiGeometricMG

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = a.n
    ndof = (n + 1) ** 2
    t0 = time.perf_counter()
    on_device = a.generate == "device" and a.mesh == "structured" and a.transfer == "linear" and a.setup == "device"
    if on_device:
        from learnmultigrid_b200 import problems as P, problems_device as PD
        A = PD.structured_laplacian_2d(n, None if a.coefficient == "constant" else PD.variable_coefficient,
                                       symmetric=a.coefficient == "variable-symmetric")
        Qs = PD.structured_hierarchy_2d(n, a.levels)
        rhs = P.structured_rhs_2d(n)            # host vector: the end-to-end leg copies it in through the API
        torch.cuda.synchronize()
    else:
        A, rhs, Qs = build_problem(a, n)
    t_gen = time.perf_counter() - t0
    mg = SemiGeometricMG(A, rhs, Qs)
    mg.setup = a.setup
    part = world > 1 and a.multi == "partitioned"
    parity = None
    fab = None
    if part:
        from learnmultigrid_b200.distributed import TorchFabric
        fab = TorchFabric()
        if a.smoother == "GaussSeidel" and not a.no_parity_check:
            parity = multi_rank_parity(torch, dist, fab, a)
        mg.distribute(fab, min_rows_per_rank=a.min_rows_per_rank, timeout_s=30.0)
        mg.local_solution = True
    t0 = time.perf_counter()
    kw = dict(levels=a.levels, smoother=a.smoother, smooth_steps=a.nu, omega=2.0 / 3.0)
    from learnmultigrid_b200 import problems as P
    colors = None
    if a.colors == "structured" and a.transfer == "linear" and a.mesh == "structured" and a.smoother == "GaussSeidel":
        colors = P.structured_colors_2d(n, a.levels)
    if a.colors == "lattice" and a.mesh == "structured" and a.transfer != "nn" and a.smoother == "GaussSeidel":
        # (alpha*ix + beta*iy) mod m from the stencil offsets of a small model hierarchy: 7 / 13 colours instead of
        # first-fit's 9 / 16 on the 19- / 37-point levels of quasi-L2 transfers
        colors = P.lattice_colors_2d(n, a.levels, transfer=a.transfer,
                                     coefficient=P.variable_coefficient if a.coefficient == "variable" else None)
    h = mg._hierarchy(a.levels, a.smoother, "multicolor", colors, True)
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t0
    params = h.make_params(nu_pre=a.nu, nu_post=a.nu, omega=2.0 / 3.0)
    lib = h.lib
    import ctypes
    h.set_rhs(rhs)
    h.zero_x()
    lev0 = h.levels[0]
    st = _lib.stream_handle(torch)

    # One outer iteration of Multigrid.solve in steady state = one program / one graph: the V-cycle, then the residual
    # norm of its result (what the next iteration tests, Multigrid.py:62-63,69).  With multicolour Gauss-Seidel the
    # last colour's share of the norm comes out of the last sweep's registers (mg_vcycle_norm / mg_dist_norm.after).
    if part:
        def step():
            h.vcycle(params, norm_after=True)
    else:
        def step():
            h.vcycle(params, with_norm=True)

    sampler = ClockSampler(local)
    sampler.start()                  # before the warm-up: NVML initialisation is over when the timed region starts
    for _ in range(max(a.warmup, 3)):
        step()
    torch.cuda.synchronize()
    launches_per_step = h.last_launches
    h.zero_x()                       # time from a fresh start so the iterate stays meaningful
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    windows = []
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    tw = time.perf_counter()
    e0.record()
    for _ in range(a.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    windows.append((tw, time.perf_counter()))
    ms_total = e0.elapsed_time(e1)
    if world > 1:
        dist.barrier()
        t = torch.tensor([ms_total], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / a.steps
    if a.dump_outputs:
        x_last, norm_last = h.get_x(view=True), h.last_norm()   # partitioned: get_x gathers the row blocks of all ranks
        if rank == 0:
            dump_outputs(a.dump_outputs, x_last, norm_last)
        del x_last
    if a.profile_step:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    res_after = h.residual_norm()
    ms_dry = None
    if part:
        h.check()                    # no exchange timed out
        # the same program with its exchange kernels launched as no-ops: kernel time without waiting for peers
        for _ in range(3):
            h.vcycle(params, norm_after=True, dry=True)
        torch.cuda.synchronize()
        dist.barrier()
        e0.record()
        for _ in range(a.steps):
            h.vcycle(params, norm_after=True, dry=True)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / a.steps], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_dry = float(t.item())
        h.zero_x()
        dist.barrier()

    # ---- dominant kernel: one fine-level smoothing sweep (sell_kernel<GS> per colour / sell_kernel<JACOBI>) ----
    S = getattr(lev0, "local_nnz_A", lev0.nnz_A) * 12 + 4 * (lev0.n + 1)      # this rank's rows
    sweep_bytes = S + 24 * lev0.n
    reps = 50
    nlaunch = len(lev0.color_ptr) - 1 if lev0.color_ptr is not None else 1

    def sweep():
        if lev0.color_ptr is not None:
            for c in range(len(lev0.color_ptr) - 1):
                _lib.check(lib.mg_sell_gs_rows(ctypes.byref(lev0.A.struct), lev0.x.data_ptr(), lev0.b.data_ptr(),
                                               int(lev0.color_ptr[c]), int(lev0.color_ptr[c + 1]), st))
        else:
            _lib.check(lib.mg_sell_jacobi(ctypes.byref(lev0.A.struct), lev0.dinv.data_ptr(), lev0.x.data_ptr(),
                                          lev0.b.data_ptr(), lev0.tmp.data_ptr(), 2.0 / 3.0, st))
    for _ in range(3):
        sweep()
    torch.cuda.synchronize()
    tw = time.perf_counter()
    e0.record()
    for _ in range(reps):
        sweep()
    e1.record()
    torch.cuda.synchronize()
    windows.append((tw, time.perf_counter()))
    ms_sweep = e0.elapsed_time(e1) / reps
    peak, peak_src = peaks()
    ach = sweep_bytes / (ms_sweep * 1e-3) / 1e9
    cyc = h.cycle_bytes(a.nu, a.nu)
    cyc_gbs = cyc["total"] / (ms_step * 1e-3) / 1e9
    # DRAM bytes per launch of that kernel from a stored `ncu --set full` capture -- only quoted for the configuration
    # it was taken on (1 GPU, this grid, constant coefficient, the kernel variant that runs by default)
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "r02_gs_traffic.json")
    implied = getattr(lev0.A, "slice_rec", None) is not None and os.environ.get("MGB_IMPLIED_COLUMNS", "1") != "0"
    if os.path.exists(tpath) and world == 1 and lev0.color_ptr is not None:
        t = json.load(open(tpath))
        vdict = getattr(lev0.A, "val_idx", None) is not None and os.environ.get("MGB_VALUE_DICT", "1") != "0"
        impv = (getattr(lev0.A, "rec_vals", None) is not None and implied and vdict
                and os.environ.get("MGB_IMPLIED_VALUES", "1") != "0")
        if (t.get("n") == n and t.get("coefficient") == a.coefficient and bool(t.get("implied_columns")) == implied
                and bool(t.get("value_dictionary")) == vdict and bool(t.get("implied_values")) == impv):
            traffic = t["traffic_per_launch"]
            traffic_src = "stored ncu --set full capture (%s), not measured in this run" % t.get("source", tpath)
    per_gpu = world if part else 1
    moved = h.cycle_bytes_moved(a.nu, a.nu) if hasattr(h, "cycle_bytes_moved") else None
    nsl0 = (lev0.n + 31) // 32
    sweep_moved = (lev0.A.stream_bytes() if hasattr(lev0.A, "stream_bytes") else S) + 24 * lev0.n
    roofline = {"bound": "hbm", "kernel": "sell_kernel<GS> (fine-level colour sweep)" if lev0.color_ptr is not None
                else "sell_kernel<JACOBI> (fine-level sweep)",
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src,
                "traffic": traffic, "traffic_source": traffic_src,
                "bytes_per_launch": sweep_bytes / nlaunch, "launches_per_sweep": nlaunch,
                "ms_per_launch": ms_sweep / nlaunch,
                "implied_columns": implied,
                "implied_values": getattr(lev0.A, "rec_vals", None) is not None and implied
                and os.environ.get("MGB_IMPLIED_VALUES", "1") != "0" and os.environ.get("MGB_VALUE_DICT", "1") != "0",
                # what the kernel actually streams (values + columns or per-slice offsets + b, x in, x out): the
                # algorithmic yardstick above stays the CSR bytes of SURVEY 8d, so byte-saving shows as frac > 1
                "moved_bytes_per_launch": sweep_moved / nlaunch,
                "moved_frac": sweep_moved / (ms_sweep * 1e-3) / 1e9 / peak,
                # whole step; per GPU (a partitioned run moves 1/world of the global bytes on each GPU)
                "cycle": {"algorithmic_bytes": cyc["total"], "algorithmic_bytes_per_gpu": cyc["total"] / per_gpu,
                          "achieved": cyc_gbs / per_gpu, "frac": cyc_gbs / per_gpu / peak,
                          "frac_of_8TBps": cyc_gbs / per_gpu / 8000.0, "bytes_per_dof": cyc["total"] / ndof,
                          "moved_bytes_per_gpu": None if moved is None else moved["total"],
                          "moved_frac": None if moved is None else moved["total"] / (ms_step * 1e-3) / 1e9 / peak,
                          "moved_model": None if moved is None else moved["model"]}}

    tw_spmv = time.perf_counter()
    # ---- SpMV per level (the metric's second half): y = A_l x on every smoothed level, algorithmic bytes
    # S(nnz, n) + 16 n (SURVEY 8d) over the CUDA-event time of back-to-back launches; this rank's rows when partitioned.
    # Informational: a failure here must not cost the headline numbers.
    try:
        per_level = []
        for l, lev in enumerate(h.levels[:-1]):
            nnz_l = getattr(lev, "local_nnz_A", lev.nnz_A)
            bytes_l = 12 * nnz_l + 4 * (lev.n + 1) + 16 * lev.n
            reps_l = 20 if lev.n > (1 << 20) else 100
            for _ in range(3):
                _lib.check(lib.mg_sell_spmv(ctypes.byref(lev.A.struct), lev.x.data_ptr(), lev.r.data_ptr(), st))
            torch.cuda.synchronize()
            e0.record()
            for _ in range(reps_l):
                _lib.check(lib.mg_sell_spmv(ctypes.byref(lev.A.struct), lev.x.data_ptr(), lev.r.data_ptr(), st))
            e1.record()
            torch.cuda.synchronize()
            ms_l = e0.elapsed_time(e1) / reps_l
            gbs_l = bytes_l / (ms_l * 1e-3) / 1e9
            per_level.append({"level": l, "rows": int(lev.n), "nnz": int(nnz_l), "us_per_launch": round(ms_l * 1e3, 2),
                              "gbs": round(gbs_l, 1), "frac": round(gbs_l / peak, 4),
                              # back-to-back launches on the same operands: what fits the 126 MB L2 is re-read from
                              # there, so fractions of levels that (partly) fit are not HBM fractions
                              "working_set_mb": round(bytes_l / 1e6, 1),
                              "l2_resident_share": round(min(1.0, 126e6 / bytes_l), 2)})
        roofline["spmv_per_level"] = per_level
    except Exception as exc:         # pragma: no cover
        roofline["spmv_per_level"] = {"error": repr(exc)}

    windows.append((tw_spmv, time.perf_counter()))
    # ---- end to end through the reference-facing API (host rhs -> solve -> host solution) -----------------------
    e2e = None
    if not a.no_e2e and (rank == 0 or part):
        C = a.cycles_per_solve
        pin = torch.from_numpy(np.ascontiguousarray(rhs.reshape(-1))).pin_memory()
        mg.rhs = pin
        mg.pinned_io = True
        solve_kw = dict(kw, error=0.0, max_iterations=C, gs_order="multicolor", colors=colors)
        mg.solve(**solve_kw)                                     # warm-up (graph already captured)
        reps_e = 3
        torch.cuda.synchronize()
        if part:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(reps_e):
            mg.solve(**solve_kw)
            _ = float(mg.solution[mg.solution.shape[0] // 2, 0])
        torch.cuda.synchronize()
        windows.append((t0, time.perf_counter()))
        dt = (time.perf_counter() - t0) / reps_e
        if part:
            t = torch.tensor([dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
            h.check()
        # partitioned: every rank copies its own row block of the rhs in and of the solution out (bytes summed over ranks)
        e2e = {"value": ndof * C / dt, "unit": UNIT, "h2d_bytes_per_step": ndof * 8, "d2h_bytes_per_step": ndof * 8 + 8 * C * (world if part else 1),
               "cycles_per_solve": C, "ms_per_solve": dt * 1e3,
               "api": "learnmultigrid_b200.solvers.Multigrid.SemiGeometricMG.solve (pinned host rhs, host solution"
                      + ("; each rank moves its own row block)" if part else ")")}

    # clocks / throttle reasons over every measured region of this process: the timed steps, the sweep and SpMV loops and
    # the end-to-end solves (the timed steps alone last ~60 ms, one or two NVML samples)
    clocks = sampler.stop(windows)
    extra = None
    if not a.no_extra and on_device and a.smoother == "GaussSeidel" and a.coefficient == "constant":
        try:
            extra = extra_configs(torch, dist, a, n, Qs, rhs, fab if part else None, world, rank)
        except Exception as exc:         # pragma: no cover
            extra = {"error": repr(exc)}

    cpu = None
    if not a.no_cpu_baseline and rank == 0:
        v, per, ncyc, tset = cpu_cycle_rate(a, a.cpu_n, reference_style=False)
        cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "extrapolated": a.cpu_n != n,
               "sample": "%dx%d grid (%d DOF) of the same %d-level V(%d,%d) configuration, %d cycles, hierarchy built "
                         "once (setup %.1f s excluded); SciPy sparsetools + C Gauss-Seidel are single-threaded; "
                         "host has %d cores" % (a.cpu_n + 1, a.cpu_n + 1, (a.cpu_n + 1) ** 2, a.levels, a.nu, a.nu,
                                                ncyc, tset, os.cpu_count()),
               "ms_per_cycle": per * 1e3}

    if rank == 0:
        line = {"metric": METRIC, "value": ndof * (1 if part else world) / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world,
                "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong" if a.multi == "partitioned" else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload_name(a, n), "l2": "inputs_exceed_l2 (%.1f GB of operators per cycle)"
                           % (cyc["total"] / 1e9), "setup": a.setup, "levels_rows": list(getattr(h, "_global_n", [l.n for l in h.levels])),
                           "levels_nnz": [l.nnz_A for l in h.levels], "colors": [None if l.color_ptr is None else
                                                                              len(l.color_ptr) - 1 for l in h.levels],
                           "generate_s": round(t_gen, 2), "generated_on": "device" if on_device else "host",
                           "setup_s": round(t_setup, 2), "nn_builder": NN_BUILD.get(n),
                           "setup_phases_s": {k: round(v, 3) for k, v in (getattr(h, "setup_timing", None) or {}).items()},
                           # BASELINE configs[4], setup sweep: per Galerkin product Q^T A Q its wall time (first build of
                           # the process: includes allocator / library warm-up; config.extra repeats it warm) and the
                           # SURVEY 8(d) byte count S(a,n) + 2 S(q) + 2 S(nnz(AQ),n) + S(a_c,n_c) over it
                           "setup_galerkin_per_level": getattr(h, "setup_galerkin", None),
                           "pinned_staging_alloc_s": (None if getattr(h, "pinned_alloc_s", None) is None
                                                      else round(h.pinned_alloc_s, 3)),
                           "residual_after_timed_steps": res_after, "multi_rank_parity": parity, "extra": extra,
                           "step": "V-cycle + residual norm of its result (one graph): steady-state outer iteration of "
                                   "Multigrid.solve; cycle fusion %s, implied columns %s"
                                   % ("off" if os.environ.get("MGB_CYCLE_FUSION", "1") == "0" else "on",
                                      "on" if implied else "off"),
                           "ms_per_step_without_exchange_waits": ms_dry,
                           "exchange": ("halo sites riding on the SELL kernel that reads the vector (peer-memory stores)"
                                        if part else None),
                           "parallelism": ("row-partitioned x%d, levels 0..%d partitioned, %d replicated, halo exchange by peer-memory "
                                           "stores over NVLink inside the cycle graph" % (world, h.n_dist - 1, a.levels - h.n_dist))
                           if part else ("replicas" if world > 1 else "single")},
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches_per_step * a.steps,
                "clocks": clocks}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
