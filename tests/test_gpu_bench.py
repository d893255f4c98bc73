"""-m gpu: bench.py's native path prints its JSON line and `--dump-outputs` writes what the last timed step returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dumps_the_outputs_of_the_last_timed_step(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", "2", "--warmup", "1",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900,
                         cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == 2 and d["value"] > 0
    names = {f[:-4] for f in os.listdir(tmp_path)}
    assert {"id_src", "src_pts", "tar_pts", "scores", "pred_poses", "M", "idx_failed"} <= names
    for name in names:
        a = np.load(tmp_path / f"{name}.npy")
        assert a.dtype in (np.float32, np.float64) and a.shape[0] == 1, (name, a.dtype, a.shape)
    assert np.load(tmp_path / "pred_poses.npy").shape == (1, 5, 4, 4)
