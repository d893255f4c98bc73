"""bench.py contract on the CPU: the reference arm (`--impl reference`, the one leg that runs without a GPU) prints
exactly one JSON line on stdout with the keys the driver reads; `rows_config` names every §8 row."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--workload", "c1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "detections/s" and d["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data",
                "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert "workload" in d["config"] and "model" not in d["config"]


def test_rows_config_lists_every_native_row():
    sys.path.insert(0, ROOT)
    import bench
    native = bench.rows_config()
    assert native["library_rows"] == [] and len(native["native_rows"]) == 9
    assert any(r.startswith("a6") for r in native["native_rows"])


def test_dump_outputs_writes_exact_float_arrays_and_a_seeded_sample_above_the_limit(tmp_path):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    g = torch.Generator().manual_seed(0)
    out = {"id_src": torch.randint(0, 10**6, (40, 5), generator=g), "idx_failed": torch.rand(40, 5, generator=g) > 0.5,
           "pred_poses": torch.randn(40, 5, 4, 4, generator=g), "M": torch.randn(40, 5, 3, 3, dtype=torch.float64, generator=g)}
    assert bench.dump_outputs(out, str(tmp_path / "all")) == sorted(out)
    for name, t in out.items():
        a = np.load(tmp_path / "all" / f"{name}.npy")
        assert a.dtype == (np.float32 if name == "pred_poses" else np.float64), name
        assert np.array_equal(a, t.double().numpy()), name
    row_bytes = 5 * 8 + 5 * 8 + 5 * 16 * 4 + 5 * 9 * 8
    limit = 7 * row_bytes + 100
    for d in ("a", "b"):
        assert bench.dump_outputs(out, str(tmp_path / d), limit=limit) == sorted(out) + ["sample_rows"]
    files = sorted(os.listdir(tmp_path / "a"))
    assert sum(os.path.getsize(tmp_path / "a" / f) - 128 for f in files) <= limit      # 128-byte .npy headers
    rows = np.load(tmp_path / "a" / "sample_rows.npy").astype(np.int64)
    assert len(rows) == 7 and len(set(rows.tolist())) == 7
    for f in files:
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes(), f
    assert np.array_equal(np.load(tmp_path / "a" / "pred_poses.npy"), out["pred_poses"][rows].numpy())


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr
