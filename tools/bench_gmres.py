"""Restarted GMRES (DeviceHierarchy.gmres) against the stationary V-cycle iteration and against PCG, one GPU, and the
Gram-Schmidt kernels on their own.

    python tools/bench_gmres.py [--configs v8193,c4097,sym8193,kernels] [--tol 1e-10] [--restart 30] [--out FILE]

    v8193    8193^2 variable coefficient with row-Dirichlet rows (BASELINE configs[3]'s operator): linear_P_2d (6 levels),
             SmoothedAggregationMG's (4 levels) and AlgebraicMG's (7 levels) transfer operators
    c4097    4097^2 convection-diffusion, eps = 0.01, beta = (1, 0.5): AlgebraicMG (6 levels) and linear_P_2d (6 levels)
    sym8193  the 8193^2 operator with its Dirichlet couplings eliminated symmetrically: GMRES against PCG (reverse
             post-smoothing, the symmetric preconditioner CG needs) on linear_P_2d
    kernels  multi-dot and multi-axpy with norm at 67 M rows (8193^2) for j+1 in {1, 8, 16, 31}: us per launch (CUDA
             events over 50 launches after 5 warm-ups; the 31 vectors are 16.6 GB, far beyond L2) and bytes moved over
             time against a device-to-device copy of the same rows timed the same way

Every arm uses forward multicolour Gauss-Seidel V(1,1) (the preconditioner of GMRES and the stationary iteration),
absolute tolerance --tol on ||b - A x|| from x = 0 with the structured right-hand side.  Per arm: iterations, ms to
tolerance (host clock around work that ends in a synchronise, second run: the graphs are captured in the first), ms per
iteration, and for GMRES the orthogonalisation share: the multi-dot and multi-axpy kernels of one cycle timed with
events on their own at the problem's size, over the ms of the same number of GMRES steps.  One JSON line per arm; the
GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except Exception:
        out = "unknown"
    return out


def sync_time(torch, fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def stationary(h, b, params, tol, max_it=400):
    """Multigrid.solve's loop on the device: ||b - A x|| first, then cycles that leave the norm of their iterate"""
    h.set_rhs(b)
    h.zero_x()
    res = h.residual_norm()
    its = 0
    while res > tol and its < max_it:
        h.vcycle(params, with_norm=True)
        res = h.last_norm()
        its += 1
    return its, res


def event_ms(torch, fn, reps=50, warm=5):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def ortho_ms(torch, lib, n, steps, restart):
    """ms of the multi-dot + multi-axpy launches of `steps` GMRES steps at n rows: step i works on j + 1 = i mod restart
    + 1 vectors (full cycles, as every run here ends by its estimate in the last one); each j timed with events"""
    m = restart + 1
    ld = (n + 31) // 32 * 32
    V = torch.ones(m * ld, dtype=torch.float64, device="cuda")
    h = torch.full((m,), 1e-3, dtype=torch.float64, device="cuda")
    parts = torch.zeros(int(lib.mg_krylov_partials(n, m)), dtype=torch.float64, device="cuda")
    out = torch.zeros(m + 1, dtype=torch.float64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    per_j = []
    for j in range(min(steps, restart)):
        w = V.data_ptr() + 8 * (j + 1) * ld

        def f():
            lib.mg_multi_dot(n, V.data_ptr(), ld, j + 1, w, parts.data_ptr(), out.data_ptr(), st)
            lib.mg_multi_axpy_norm(n, V.data_ptr(), ld, j + 1, h.data_ptr(), w, parts.data_ptr(), out.data_ptr(), st)
        per_j.append(event_ms(torch, f, reps=10, warm=2))
    del V
    return sum(per_j[i % restart] for i in range(steps))


def run_arm(torch, lib, name, A, b, Qs, tol, restart, emit, pcg=False):
    from learnmultigrid_b200.engine import DeviceHierarchy
    h, setup = sync_time(torch, lambda: DeviceHierarchy(A, Qs, smoother="mcgs", keep_host=False))
    base = {"config": name, "rows": int(A.shape[0]), "levels": len(Qs) + 1, "setup_s": round(setup, 3)}
    fwd = h.make_params(nu_pre=1, nu_post=1)
    if pcg:
        sym = h.make_params(nu_pre=1, nu_post=1, reverse_post=True)
        h.pcg(b, sym, error=tol, max_iterations=200)
        (x, track, its), t = sync_time(torch, lambda: h.pcg(b, sym, error=tol, max_iterations=200))
        emit(dict(base, method="PCG (reverse post-smoothing)", iterations=its, ms_total=round(1e3 * t, 2),
                  ms_per_iteration=round(1e3 * t / its, 3), final=track[-1]))
    else:
        stationary(h, b, fwd, tol)
        (its, res), t = sync_time(torch, lambda: stationary(h, b, fwd, tol))
        emit(dict(base, method="stationary V(1,1)", iterations=its, ms_total=round(1e3 * t, 2),
                  ms_per_iteration=round(1e3 * t / max(its, 1), 3), final=res))
    h.gmres(b, fwd, error=tol, max_iterations=400, restart=restart)
    (x, track, its, res), t = sync_time(torch, lambda: h.gmres(b, fwd, error=tol, max_iterations=400, restart=restart))
    tim = h.last_gmres_timing
    orth = ortho_ms(torch, lib, h.n, its, restart)
    emit(dict(base, method="GMRES(%d) forward V(1,1)" % restart, iterations=its, ms_total=round(1e3 * t, 2),
              ms_iterations=round(1e3 * tim["iterations_s"], 2),
              ms_per_iteration=round(1e3 * tim["iterations_s"] / max(its, 1), 3), final=res,
              orthogonalisation_ms=round(orth, 2),
              orthogonalisation_share=round(orth / (1e3 * tim["iterations_s"]), 4)))
    del h
    torch.cuda.empty_cache()


def kernels(torch, lib, emit):
    n = 8193 * 8193
    ld = (n + 31) // 32 * 32
    V = torch.ones(32 * ld, dtype=torch.float64, device="cuda")
    h = torch.full((32,), 1e-3, dtype=torch.float64, device="cuda")
    parts = torch.zeros(int(lib.mg_krylov_partials(n, 32)), dtype=torch.float64, device="cuda")
    out = torch.zeros(32, dtype=torch.float64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    src, dst = V[:n], V[ld:ld + n]
    copy_ms = event_ms(torch, lambda: dst.copy_(src))
    copy_bw = 16 * n / (copy_ms * 1e-3)
    for m in (1, 8, 16, 31):
        w = V.data_ptr() + 8 * m * ld
        dot = event_ms(torch, lambda: lib.mg_multi_dot(n, V.data_ptr(), ld, m, w, parts.data_ptr(), out.data_ptr(), st))
        axp = event_ms(torch, lambda: lib.mg_multi_axpy_norm(n, V.data_ptr(), ld, m, h.data_ptr(), w, parts.data_ptr(),
                                                            out.data_ptr(), st))
        bdot = n * (8 * m + 8 * ((m + 7) // 8))          # V read once, w once per tile of 8
        baxp = n * (8 * m + 16)                          # V read, w read and written
        emit({"config": "kernels", "rows": n, "j+1": m, "multi_dot_us": round(1e3 * dot, 1),
              "multi_dot_TBps": round(bdot / (dot * 1e-3) / 1e12, 3), "multi_axpy_norm_us": round(1e3 * axp, 1),
              "multi_axpy_norm_TBps": round(baxp / (axp * 1e-3) / 1e12, 3),
              "copy_TBps": round(copy_bw / 1e12, 3), "multi_dot_of_copy": round(bdot / (dot * 1e-3) / copy_bw, 3),
              "multi_axpy_norm_of_copy": round(baxp / (axp * 1e-3) / copy_bw, 3)})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="v8193,c4097,sym8193,kernels")
    ap.add_argument("--tol", type=float, default=1e-10)
    ap.add_argument("--restart", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from learnmultigrid_b200 import _lib
    from learnmultigrid_b200 import formats as F
    from learnmultigrid_b200 import problems as P
    from learnmultigrid_b200.amg import AmgBuilder
    from learnmultigrid_b200.sa import SaBuilder
    lib = _lib.load()
    card = gpu_info()
    outf = open(a.out, "a") if a.out else None

    def emit(d):
        d["gpu"] = card
        line = json.dumps(d)
        print(line, flush=True)
        if outf:
            outf.write(line + "\n")
            outf.flush()
    cfgs = a.configs.split(",")
    if "v8193" in cfgs:
        N = 8192
        A = P.structured_laplacian_2d(N, P.variable_coefficient)
        b = P.structured_rhs_2d(N)
        run_arm(torch, lib, "v8193 linear", A, b, P.structured_hierarchy_2d(N, 6, transfer="linear"), a.tol,
                a.restart, emit)
        run_arm(torch, lib, "v8193 SA", A, b, SaBuilder().define_hierarchy(F.canonical_csr(A), 4), a.tol, a.restart,
                emit)
        run_arm(torch, lib, "v8193 AMG", A, b, AmgBuilder().define_hierarchy(F.canonical_csr(A), 7), a.tol, a.restart,
                emit)
    if "c4097" in cfgs:
        N = 4096
        A = P.convection_diffusion_2d(N, 0.01, (1.0, 0.5))
        b = P.structured_rhs_2d(N)
        run_arm(torch, lib, "c4097 AMG", A, b, AmgBuilder().define_hierarchy(F.canonical_csr(A), 6), a.tol, a.restart,
                emit)
        run_arm(torch, lib, "c4097 linear", A, b, P.structured_hierarchy_2d(N, 6, transfer="linear"), a.tol,
                a.restart, emit)
    if "sym8193" in cfgs:
        N = 8192
        A = P.symmetric_dirichlet(P.structured_laplacian_2d(N, P.variable_coefficient), P.boundary_nodes_2d(N))
        run_arm(torch, lib, "sym8193 linear", A, P.structured_rhs_2d(N), P.structured_hierarchy_2d(N, 6, "linear"),
                a.tol, a.restart, emit, pcg=True)
    if "kernels" in cfgs:
        kernels(torch, lib, emit)


if __name__ == "__main__":
    main()
