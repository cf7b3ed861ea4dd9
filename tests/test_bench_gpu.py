"""GPU: bench.py --dump-outputs writes what the timed step computed, for the seeded configs[1] batch."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, rel_err

pytestmark = pytest.mark.gpu


def test_dump_outputs_are_the_timed_trajectories(tmp_path):
    import bench
    import oracle
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--e2e-steps", "1",
           "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(tmp_path / "out")]
    out = subprocess.run(cmd, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    assert os.listdir(tmp_path / "out") == ["trajectories.npy"]
    y = np.load(tmp_path / "out" / "trajectories.npy")
    lens, means, variances = bench.make_batch(0)
    off = np.concatenate([[0], np.cumsum(lens)])
    assert y.dtype == np.float32 and y.shape == (int(lens.sum()), bench.D_OUT)
    for u in (0, len(lens) - 1):
        a, b = off[u], off[u + 1]
        assert rel_err(y[a:b, :60], oracle.mlpg(means[a:b, :180], variances[a:b, :180], bench.WINDOWS)) < 1e-6
        assert np.array_equal(y[a:b, 61], means[a:b, 183])  # the copied vuv column
