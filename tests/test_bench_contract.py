"""bench.py's reference arm (CPU): the JSON line carries the contract's keys, and -- where the reference's sources are
reachable -- it is the UNMODIFIED reference that is timed (kind == "reference"), at the GPU arm's K.  Also the
--dump-outputs writer and the argument checks (CPU)."""
import json
import os
import subprocess
import sys

import numpy as np

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "stdout must carry exactly one JSON line"
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "stage2_reranked_triplets_per_s" and d["unit"] == "triplets/s"
    assert d["vs_baseline"] is None and d["value"] > 0 and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "K=100" in d["config"]["workload"] and "K=100" in d["cpu_baseline"]["sample"]
    assert d["cpu_baseline"]["kind"] == ("reference" if bench.find_reference() else "port")


def test_dump_outputs_writes_float_arrays(tmp_path):
    rng = np.random.default_rng(1)
    scores = rng.standard_normal((5, 4)).astype(np.float32)
    order = np.argsort(-scores, axis=1, kind="stable").astype(np.int32)
    bench.dump_outputs(str(tmp_path), scores, order, np.array([3, 5], np.int64))
    got = {n: np.load(tmp_path / f"{n}.npy") for n in ("scores", "order", "recall_hits_at_10_50", "rows")}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert np.array_equal(got["scores"], scores) and np.array_equal(got["order"], order)
    assert got["recall_hits_at_10_50"].tolist() == [3.0, 5.0] and got["rows"].tolist() == [0, 1, 2, 3, 4]


def test_dump_outputs_samples_rows_under_the_limit(tmp_path):
    Q, K = 1000, 50
    scores = np.arange(Q * K, dtype=np.float32).reshape(Q, K)
    order = np.tile(np.arange(K, dtype=np.int32), (Q, 1))
    limit = 100_000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), scores, order, [1, 2], limit=limit)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= limit
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert 0 < len(rows) < Q and np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy"))      # fixed sample
    assert np.array_equal(np.load(tmp_path / "a" / "scores.npy"), scores[rows.astype(np.int64)])


def test_bench_rejects_zero_steps():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=600, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), cwd=ROOT)
    assert out.returncode != 0 and "--steps must be >= 1" in out.stderr


def test_find_reference_lookup(tmp_path, monkeypatch):
    """$CIR_REFERENCE wins when it holds the reference's sources; otherwise only ./baseline/_ref is looked at."""
    (tmp_path / "ref" / "src").mkdir(parents=True)
    (tmp_path / "ref" / "src" / "blip_stage2.py").write_text("")
    monkeypatch.setenv("CIR_REFERENCE", str(tmp_path / "ref"))
    assert bench.find_reference() == str(tmp_path / "ref")
    in_tree = os.path.join(ROOT, "baseline", "_ref")
    want = in_tree if os.path.exists(os.path.join(in_tree, "src", "blip_stage2.py")) else None
    monkeypatch.setenv("CIR_REFERENCE", str(tmp_path))                     # no src/blip_stage2.py there
    assert bench.find_reference() == want
    monkeypatch.delenv("CIR_REFERENCE")
    assert bench.find_reference() == want
