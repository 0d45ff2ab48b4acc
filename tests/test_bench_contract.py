"""bench.py contract, the part that runs without a GPU: the reference arm (`--impl reference`) must print exactly one JSON line
with the keys the driver reads, time the CPU path on this host, and mark itself as the reference implementation."""
import json
import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--ref-threads", "4"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "loop-closure queries/sec" and d["unit"] == "queries/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    # "reference" when the NN leg is the reference's own rtflann compiled into oracle/_ref, "port" when only the restatement exists
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] == 4 and d["cpu_baseline"]["value"] == d["value"]
    assert isinstance(d["cpu_baseline"].get("legs"), dict) and d["cpu_baseline"]["legs"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["top1_place_hit_rate"] == 1.0       # the CPU path finds the revisited place of every sampled frame


def test_other_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=120)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_dump_outputs_keeps_a_fixed_sample_of_frames_under_the_limit(tmp_path, monkeypatch):
    import importlib.util

    import numpy as np

    spec = importlib.util.spec_from_file_location("bench_module", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rng = np.random.default_rng(0)
    n = 50
    res = [{"ok": bool(i % 2), "n_matches": i, "n_inliers": i // 2, "iterations_run": 3 * i, "rvec": rng.random(3), "tvec": rng.random(3),
            "transform": rng.random((3, 4)).astype(np.float32), "covariance": rng.random((6, 6))} for i in range(n)]
    out = bench.step_outputs(rng.integers(0, 1 << 20, (n, 1000), dtype=np.int32), rng.random((n, 2000), dtype=np.float32),
                             rng.integers(0, 100, n, dtype=np.int32), res)
    bench.dump_outputs(str(tmp_path / "all"), out)
    assert np.array_equal(np.load(tmp_path / "all" / "frame_index.npy"), np.arange(n))
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 300_000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), out)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == sorted(["frame_index.npy"] + [k + ".npy" for k in out])
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 300_000
    frames = np.load(tmp_path / "a" / "frame_index.npy").astype(np.int64)
    assert 0 < len(frames) < n and np.all(np.diff(frames) > 0)
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b)
        if f != "frame_index.npy":
            assert np.array_equal(a, out[f[:-4]][frames])
