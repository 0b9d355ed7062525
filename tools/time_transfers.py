"""Per-kernel times of the level-0 and level-1 transfer operators of the flagship hierarchy (2D P1 Laplacian, linear
transfers, multicolour Gauss-Seidel ordering), with the implied transfer columns on and off in the same process
(mg_set_implied_transfers): the restriction y = Q^T r over all coarse rows and the prolongation u += Q e onto the
rows the cycle corrects (all colours but the first).  CUDA events around every launch; L2 (126 MB on a B200) is
overwritten with a 512 MB fill before each one, so every launch reads its operands from HBM.  Prints the card, its
power limit, and one JSON line per launch and setting."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=8192, help="squares per side of the fine mesh ((n+1)^2 unknowns)")
    ap.add_argument("--levels", type=int, default=6)
    ap.add_argument("--reps", type=int, default=50)
    a = ap.parse_args()
    import torch
    from learnmultigrid_b200 import _lib, problems_device as PD
    from learnmultigrid_b200.engine import DeviceHierarchy
    torch.cuda.set_device(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print("device:", torch.cuda.get_device_name(0), "|", q[0] if q else "nvidia-smi unavailable")
    lib = _lib.load()
    A = PD.structured_laplacian_2d(a.n, None)
    Qs = PD.structured_hierarchy_2d(a.n, a.levels)
    h = DeviceHierarchy(A, Qs, smoother="mcgs")
    st = _lib.stream_handle(torch)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    launches = []
    for l in (0, 1):
        lev, nxt = h.levels[l], h.levels[l + 1]
        r = torch.randn(lev.n, dtype=torch.float64, device="cuda")
        e = torch.randn(nxt.n, dtype=torch.float64, device="cuda")
        yc = torch.empty(nxt.n, dtype=torch.float64, device="cuda")
        u = torch.randn(lev.n, dtype=torch.float64, device="cuda")
        p0 = int(lev.color_ptr[1])
        launches.append(("restriction", l, lev.QT, nxt.n,
                         lambda T=lev.QT, r=r, yc=yc: lib.mg_sell_spmv(T.struct, r.data_ptr(), yc.data_ptr(), st)))
        launches.append(("prolongation", l, lev.Q, lev.n - p0,
                         lambda T=lev.Q, e=e, u=u, p0=p0, n=lev.n: lib.mg_sell_prolong_correct_rows(
                             T.struct, e.data_ptr(), u.data_ptr(), u.data_ptr(), p0, n, st)))
    for on in (1, 0, 1, 0):
        lib.mg_set_implied_transfers(on)
        for name, l, T, rows, fn in launches:
            ts = []
            for i in range(a.reps + 3):
                flush.fill_(i & 0xff)
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                _lib.check(fn(), name)
                t1.record()
                t1.synchronize()
                if i >= 3:
                    ts.append(t0.elapsed_time(t1) * 1e3)
            ts.sort()
            print(json.dumps({"launch": name, "level": l, "implied_transfers": on, "rows": rows,
                              "median_us": round(ts[len(ts) // 2], 2), "min_us": round(ts[0], 2),
                              "p90_us": round(ts[int(0.9 * len(ts))], 2),
                              "pattern_slices": T.pattern_slices, "slices": int(T.struct.nslices),
                              "records": -int(T.struct.nrec),
                              "matrix_bytes_per_pass": int(T.stream_bytes() * rows / T.shape[0])}))
    lib.mg_set_implied_transfers(1)


if __name__ == "__main__":
    main()
