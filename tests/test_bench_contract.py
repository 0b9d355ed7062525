"""bench.py contract checks: the reference arm (`--impl reference`: the oracle with the reference's per-cycle Galerkin
products and LU, on host cores) prints ONE JSON line with the keys a caller reads, the argument parser accepts the
documented command lines, and --dump-outputs writes what the last timed step computed (the B200 arm's check needs a
GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import history_tolerance

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, env=None, gpu=False):
    e = dict(os.environ, **(env or {}))
    if not gpu:
        e["CUDA_VISIBLE_DEVICES"] = ""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=600, env=e, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def test_reference_arm_prints_one_contract_line():
    d = run_bench("--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "1", "--cpu-n", "64")
    assert d["impl"] == "reference" and d["metric"] == "vcycle_fine_grid_dof_per_s" and d["unit"] == "DOF/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] >= 1 and d["value"] > 0
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["scaling"] in ("strong", "weak") and "workload" in d["config"] and "sample" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert abs(d["ms_per_step"] * 1e-3 * d["value"] - 65 * 65) < 1e-6 * 65 * 65        # value = sample DOF / time


def test_reference_arm_on_a_non_zero_rank_exits_without_work():
    e = dict(os.environ, CUDA_VISIBLE_DEVICES="", RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "0", "--cpu-n", "32"], capture_output=True, text=True,
                         timeout=300, env=e, cwd=ROOT)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def load_dump(path):
    out = {name: np.load(os.path.join(path, name + ".npy")) for name in ("solution", "residual_norm")}
    assert all(v.dtype == np.float64 for v in out.values()) and out["residual_norm"].shape == (1,)
    return out


def test_reference_arm_dumps_its_last_step(tmp_path):
    """--steps sets the number of timed steps; --dump-outputs writes the iterate the last step left and the residual
    norm it computed (that of the iterate it started from), the same bits in two runs"""
    from learnmultigrid_b200 import problems as P
    d = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-n", "32",
                  "--dump-outputs", str(tmp_path / "first"))
    assert d["steps"] == 1
    first = load_dump(tmp_path / "first")
    assert first["solution"].shape == (33 * 33,)
    assert first["residual_norm"][0] == np.linalg.norm(P.structured_rhs_2d(32))        # started from x = 0
    dumps = []
    for k in range(2):
        d = run_bench("--impl", "reference", "--steps", "3", "--warmup", "1", "--cpu-n", "32",
                      "--dump-outputs", str(tmp_path / str(k)))
        assert d["steps"] == 3
        dumps.append(load_dump(tmp_path / str(k)))
    for name in dumps[0]:
        assert np.array_equal(dumps[0][name], dumps[1][name])
    assert dumps[0]["residual_norm"][0] < first["residual_norm"][0]


@pytest.mark.gpu
def test_b200_arm_dumps_its_last_step(tmp_path):
    """the timed path's iterate after exactly --steps cycles from zero and the residual norm of that iterate, the same
    bits in two runs"""
    from learnmultigrid_b200 import problems as P
    N = 128
    dumps = []
    for k, warmup in enumerate((1, 4)):
        d = run_bench("--gpus", "1", "--steps", "4", "--warmup", str(warmup), "--n", str(N), "--levels", "4",
                      "--no-cpu-baseline", "--no-e2e", "--no-extra", "--dump-outputs", str(tmp_path / str(k)), gpu=True)
        assert d["steps"] == 4
        dumps.append(load_dump(tmp_path / str(k)))
    for name in dumps[0]:
        assert np.array_equal(dumps[0][name], dumps[1][name])
    A, b = P.structured_laplacian_2d(N), P.structured_rhs_2d(N).reshape(-1)
    x = dumps[0]["solution"]
    assert x.shape == ((N + 1) ** 2,)
    assert abs(dumps[0]["residual_norm"][0] - np.linalg.norm(b - A @ x)) <= history_tolerance(A, x)
