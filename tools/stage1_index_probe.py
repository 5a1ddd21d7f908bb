"""Stage-I search over a 1M-row gallery: per-call cir_stage1_topk against the resident index (cir_stage1_index), eager and replayed
from a CUDA graph.  One GPU, G = 1,048,576 unit rows, K = 200, Q in {1, 16, 256, 4181}.

For each Q the three variants run in the same process, alternating round by round, each round timed with CUDA events over
enough calls for ~50 ms; rounds continue until every variant has at least --seconds of timed work.  Reported: median
ms per call and the spread (min, max, p10, p90) over rounds.  The gallery (1 GB fp32 + 0.5 GB bf16) is larger than the L2,
so every call reads it from HBM.  Also: the build time of the 1M-row index as one add and as 16-row appends (the
extract_index_features batch).  Every Q asserts that the three variants return the same lists bit for bit.

    python tools/stage1_index_probe.py --out profiles/r03_stage1_index.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import cir_b200 as cir


def unit(n, seed, dev, chunk=1 << 18):
    g = torch.Generator(device=dev).manual_seed(seed)
    out = torch.empty(n, 256, device=dev)
    for r0 in range(0, n, chunk):
        x = torch.randn(min(chunk, n - r0), 256, generator=g, device=dev)
        out[r0:r0 + x.shape[0]] = torch.nn.functional.normalize(x, dim=-1)
    return out


def device_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else ""
    return {"query": q, "nvidia_smi": line, "torch_name": torch.cuda.get_device_name()}


def time_calls(fn, n):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n):
        fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / n


def stats(v):
    v = np.asarray(v)
    return {"median_ms": float(np.median(v)), "min_ms": float(v.min()), "max_ms": float(v.max()),
            "p10_ms": float(np.percentile(v, 10)), "p90_ms": float(np.percentile(v, 90)), "rounds": int(v.size)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--G", type=int, default=1 << 20)
    ap.add_argument("--K", type=int, default=200)
    ap.add_argument("--Q", type=str, default="1,16,256,4181")
    ap.add_argument("--seconds", type=float, default=1.0, help="least timed work per (Q, variant)")
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stage1_index_probe needs a GPU")
    dev = torch.device("cuda", torch.cuda.current_device())
    eng = cir.engine.get_engine(dev, "bf16")
    G, K = a.G, a.K
    g = unit(G, 1, dev)
    res = {"device": device_info(), "G": G, "K": K, "precision": "bf16",
           "variants": {"a": "eng.stage1_topk per call (transient bf16 view of the gallery built in the workspace every call)",
                        "b": "Stage1Index.topk, eager", "c": "Stage1Index.topk replayed from a CUDA graph"}}

    # build time: one add of G rows, and G/16 appends of 16 rows (host-bound: one C-ABI call per append)
    one_shot = []
    for _ in range(3):
        idx = eng.stage1_index(G)
        torch.cuda.synchronize()
        one_shot.append(time_calls(lambda: idx.add(g), 1))
        del idx
    idx16 = eng.stage1_index(G)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for r0 in range(0, G, 16):
        idx16.add(g[r0:r0 + 16])
    torch.cuda.synchronize()
    append_s = time.perf_counter() - t0
    idx = eng.stage1_index(G).add(g)
    res["build"] = {"one_add_ms": stats(one_shot), "appends_of_16_rows_s": append_s, "appends": G // 16}

    res["points"] = []
    for Q in [int(x) for x in a.Q.split(",")]:
        q = unit(Q, 100 + Q, dev)
        outs = {v: (torch.empty(Q, K, device=dev), torch.empty(Q, K, dtype=torch.int32, device=dev)) for v in "abc"}
        exact = torch.zeros(Q, dtype=torch.int32, device=dev)

        def run_a():
            outs["a"] = eng.stage1_topk(q, g, K)

        def run_b():
            idx.topk(q, K, out=outs["b"], exact_rows=exact)

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            run_b()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            idx.topk(q, K, out=outs["c"])
        fns = {"a": run_a, "b": run_b, "c": graph.replay}
        for f in fns.values():                                  # warm-up
            for _ in range(3):
                f()
        torch.cuda.synchronize()
        same = all(torch.equal(outs["a"][j], outs[v][j]) for v in "bc" for j in (0, 1))
        assert same, f"Q={Q}: variants differ"
        per = {v: time_calls(fns[v], 1) for v in "abc"}
        n = {v: max(1, int(50.0 / max(per[v], 1e-3))) for v in "abc"}
        samples = {v: [] for v in "abc"}
        spent = {v: 0.0 for v in "abc"}
        while min(spent.values()) < a.seconds * 1e3 or min(len(s) for s in samples.values()) < 10:
            for v in "abc":
                ms = time_calls(fns[v], n[v])
                samples[v].append(ms)
                spent[v] += ms * n[v]
        torch.cuda.synchronize()
        same_after = all(torch.equal(outs["a"][j], outs[v][j]) for v in "bc" for j in (0, 1))
        assert same_after, f"Q={Q}: variants differ after timing"
        pt = {"Q": Q, "bit_equal_a_b_c": bool(same and same_after), "exact_fallback_queries": int(exact.sum()),
              "calls_per_round": n, "timed_s": {v: spent[v] / 1e3 for v in "abc"}}
        for v in "abc":
            pt[v] = stats(samples[v])
        pt["b_over_a"] = pt["b"]["median_ms"] / pt["a"]["median_ms"]
        pt["c_over_a"] = pt["c"]["median_ms"] / pt["a"]["median_ms"]
        res["points"].append(pt)
        print(json.dumps({k: pt[k] for k in ("Q", "bit_equal_a_b_c", "exact_fallback_queries", "b_over_a", "c_over_a")} |
                         {v: round(pt[v]["median_ms"], 4) for v in "abc"}), flush=True)
        del graph
    res["device_after"] = device_info()
    js = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(js + "\n")
    print(js)


if __name__ == "__main__":
    main()
