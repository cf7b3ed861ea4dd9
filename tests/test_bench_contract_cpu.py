"""bench.py's workload and JSON contract, as far as it can be checked without a GPU."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_workload_is_baseline_config1_and_deterministic():
    import bench
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert bench.METRIC.startswith("mlpg_frames") and "frames" in base["metric"]
    lens, m, v = bench.make_batch(0)
    lens2, m2, v2 = bench.make_batch(0)
    assert np.array_equal(lens, lens2) and np.array_equal(m, m2) and np.array_equal(v, v2)
    assert len(lens) == 256 and lens.min() >= 540 and lens.max() <= 660
    assert m.shape == (int(lens.sum()), 187) and m.dtype == np.float32 and v.min() >= 0.1
    assert not np.array_equal(bench.make_batch(1)[0], lens)  # other ranks get other utterances (weak scaling)
    # SURVEY 8(d): 186 mean + 186 variance columns in, 62 trajectories + the copied vuv column in/out, float32
    assert bench.ALGO_BYTES_PER_FRAME == 4 * (186 + 186 + 62 + 2) == 1744
    cfg = bench.config(1)
    assert "workload" in cfg and "model" not in cfg
    assert bench.usable_cores() >= 1


def test_reference_arm_line_on_a_tiny_sample(monkeypatch):
    """--impl reference on the CPU: same metric / unit / config keys, impl tag, zero-copy e2e object."""
    import oracle
    env = dict(os.environ)
    code = (
        "import bench, sys, json\n"
        "bench.N_UTT = 8\n"  # bounded sample so that the CPU suite stays fast
        "sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0']\n"
        "bench.main()\n")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "mlpg_frames_per_sec" and line["unit"] == "frames/s"
    assert line["higher_is_better"] is True and line["value"] > 0 and line["gpu_launches"] == 0
    assert line["e2e"] == {"value": line["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] == ("reference" if oracle.reference_available() else "port") and cb["cores"] >= 1


def test_dump_outputs_is_refused_where_it_does_not_apply(tmp_path):
    for extra in (["--impl", "reference"], ["--gpus", "2"]):
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(tmp_path / "out")] + extra
        out = subprocess.run(cmd, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
        assert out.returncode == 2 and "--dump-outputs" in out.stderr
    assert not (tmp_path / "out").exists()
