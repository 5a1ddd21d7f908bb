"""bench.py --dump-outputs on the GPU: the last timed step's outputs land in DIR, and two runs with the same arguments
write the same arrays (seeded inputs)."""
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

import bench

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Q, K, G = 24, 50, 64


def _run(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--queries", str(Q), "--k", str(K),
           "--gallery", str(G), "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip())
    assert line["steps"] == 2 and line["warmup"] == 1
    return {n: np.load(os.path.join(out_dir, f"{n}.npy")) for n in ("scores", "order", "recall_hits_at_10_50", "rows")}


def test_dump_outputs_of_the_timed_step(tmp_path):
    a, b = _run(tmp_path / "a"), _run(tmp_path / "b")
    assert a["scores"].shape == a["order"].shape == (Q, K) and a["rows"].tolist() == list(range(Q))
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    order = a["order"].astype(np.int64)
    assert all(sorted(r) == list(range(K)) for r in order.tolist())
    ranked = np.take_along_axis(a["scores"], order, axis=1)
    assert (np.diff(ranked, axis=1) <= 0).all()                          # descending re-rank of the scores written
    # the counters belong to the order written: recount them from it and the bench's own seeded labels
    labels = bench.synth_workload(SimpleNamespace(queries=Q, k=K, gallery=G, length=32))[5].numpy()
    ranked_labels = np.take_along_axis(labels, order, axis=1)
    assert a["recall_hits_at_10_50"].tolist() == [float(ranked_labels[:, :k].sum()) for k in (10, 50)]
    for n in a:
        assert np.array_equal(a[n], b[n]), n
