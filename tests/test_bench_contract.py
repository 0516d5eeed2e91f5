"""bench.py's reference arm on the host (no GPU needed): the JSON line keeps the contract's keys, times the oracle
port only, and names the same workload as the GPU arm.  On the GPU: --dump-outputs writes the timed step's result."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference"
    assert line["metric"].startswith("min-snap solves/sec") and line["unit"] == "solves/s"
    assert line["higher_is_better"] is True and line["dtype"] == "f64" and line["vs_baseline"] is None
    assert line["value"] > 0 and line["ms_per_step"] > 0 and line["steps"] == 1
    base = line["cpu_baseline"]
    assert base["kind"] == "port" and base["cores"] >= 1 and base["value"] == line["value"] and base["sample"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    # both arms print the same config dict (the driver compares them)
    sys.path.insert(0, ROOT)
    import bench
    assert line["config"] == bench.CONFIG
    assert "workload" in line["config"] and "model" not in line["config"]


def test_gpu_arm_refuses_without_a_device():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]])
def test_bad_arguments_are_refused(args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 2 and "error" in out.stderr


@pytest.mark.gpu
def test_dump_outputs_hold_the_timed_solve(tmp_path, ms, torch_cuda):
    """--dump-outputs writes what the headline step returns for the sampled trajectories, bit for bit."""
    torch = torch_cuda
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--skip-configs",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["coeffs.npy"]
    got = np.load(tmp_path / "coeffs.npy")
    sys.path.insert(0, ROOT)
    import bench
    rows = bench.dump_rows(bench.B_PER_GPU)
    assert got.dtype == np.float64 and got.shape == (len(rows), bench.K_SEG, bench.DIM, bench.NCOEF)
    assert got.nbytes <= 64 << 20
    pos = torch.from_numpy(ms.random_positions_host(bench.B_PER_GPU, bench.K_SEG, bench.BOX_LO, bench.BOX_HI,
                                                    bench.BASE_SEED)).cuda()
    times = ms.estimate_segment_times(pos, bench.V_MAX, bench.A_MAX, bench.MAGIC)
    coeffs = torch.empty((bench.B_PER_GPU, bench.K_SEG, bench.DIM, bench.NCOEF), dtype=torch.float64, device="cuda")
    ms.solve_standard(pos, times, coeffs=coeffs, want_status=False)
    assert np.array_equal(got, coeffs.cpu().numpy()[rows])
