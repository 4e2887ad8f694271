"""bench.py's output contract, as far as it can be checked without a GPU: the reference arm (the CPU port of the
reference's EventLoop path) prints exactly ONE line on stdout, and that line is the JSON object the driver parses."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--cpu-groups", "1024"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout
    rec = json.loads(lines[0])
    assert rec["impl"] == "reference" and rec["metric"] == "AppendEntries/sec across Raft groups" and rec["unit"] == "acks/s"
    assert rec["higher_is_better"] is True and rec["n_gpus"] == 1 and rec["steps"] == 2 and rec["warmup"] == 1
    assert rec["vs_baseline"] is None and rec["data"] == "synthetic"
    assert rec["value"] > 0 and rec["ms_per_step"] > 0
    assert rec["cpu_baseline"]["kind"] == "port" and rec["cpu_baseline"]["value"] == rec["value"] and rec["cpu_baseline"]["cores"] >= 1
    assert rec["e2e"] == {"value": rec["value"], "unit": "acks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in rec["config"]


def test_dump_outputs_writes_the_last_outbox_the_same_way_every_run(tmp_path):
    import numpy as np
    dumps = []
    for run in ("a", "b"):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                              "--cpu-groups", "1024", "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True,
                             timeout=300, cwd=ROOT)
        assert res.returncode == 0, res.stderr[-2000:]
        dumps.append({p.name: np.load(p) for p in sorted((tmp_path / run).iterdir())})
    a, b = dumps
    assert set(a) == set(b) and {"gids.npy", "commit_index.npy", "plan_meta.npy", "last_entry.npy"} <= set(a)
    assert sum((tmp_path / "a" / name).stat().st_size for name in a) <= 64 * 10 ** 6
    for name in a:
        assert a[name].dtype == np.float64 and np.array_equal(a[name], b[name]), name
    assert np.array_equal(a["gids.npy"], np.arange(1024))                   # 1024 groups fit: no sampling
    assert a["plan_meta.npy"].shape == (16, 1024, 2, 2) and a["commit_index.npy"].max() > 0


def test_steps_below_one_are_refused():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert res.returncode == 2 and "--steps" in res.stderr and not res.stdout.strip()


def test_engine_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--no-cpu", "--no-e2e"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert res.returncode != 0 and not res.stdout.strip()              # no CPU fallback, no fake line
