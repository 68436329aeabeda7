"""bench.py: the CPU arm (--impl reference) prints one JSON line with the headline's keys; --dump-outputs writes what the
timed path returned"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _reference_line(env=None):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--quick"], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "RANGE+ embeddings/sec" and d["unit"] == "queries/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "sample" in d["config"]
    return d


def test_reference_arm_prints_one_json_line():
    """the unmodified reference when it is staged under oracle/_ref/reference (build container, GPU box), else the port"""
    sys.path.insert(0, ROOT)
    from oracle import ref_harness
    d = _reference_line()
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_harness.available() else "port")


def test_reference_arm_falls_back_to_the_port():
    d = _reference_line(dict(os.environ, RANGE_BENCH_REFERENCE="port"))
    assert d["cpu_baseline"]["kind"] == "port"


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_path(tmp_path, sh_entries):
    """the step's float32 result and model(locs)'s float64 array on the same sampled rows: they agree with each other
    (other batch boundaries in model(locs): last-bit fp16 rounding differences only) and with the exact CPU oracle"""
    from oracle import range_oracle as O
    import bench
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    assert json.loads(p.stdout.splitlines()[-1])["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["embeddings.npy", "model_embeddings.npy"]
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 << 20
    rows = bench.dump_rows()
    e, m = np.load(tmp_path / "embeddings.npy"), np.load(tmp_path / "model_embeddings.npy")
    assert e.dtype == np.float32 and m.dtype == np.float64 and e.shape == m.shape == (len(rows), 1280)
    assert np.isfinite(m).all() and np.abs(e[:, 1024:] - m[:, 1024:]).max() <= 1e-7
    rel = np.linalg.norm(e[:, :1024] - m[:, :1024], axis=1) / np.linalg.norm(m[:, :1024], axis=1)
    assert rel.max() <= 5e-4, rel.max()
    db, weights, coords = bench.synthetic_inputs()
    sub = np.arange(0, len(rows), len(rows) // 16)
    ref = O.RangeOracle("RANGE+", weights, sh_entries, db, beta=bench.BETA, exact=True)(coords[rows[sub]])
    rel = np.linalg.norm(m[sub, :1024] - ref[:, :1024], axis=1) / np.linalg.norm(ref[:, :1024], axis=1)
    assert rel.max() <= 1e-3 and np.abs(m[sub, 1024:] - ref[:, 1024:]).max() <= 1e-3, rel.max()
