"""Compacted and subset stage-I indexes against the filtered search they replace.  One GPU, G = 1,048,576 unit rows, K = 200,
Q in {1, 16, 256, 4181}; the selectivities of tools/stage1_filter_probe.py:
  rm10    10 % of the rows removed (tag 0)                     -> Stage1Index.compact() of a copy of the index
  1/3     three categories (tags 1 / 2 / 4, random rows), mask 1 -> Stage1Index.subset(1)
  1/16    sixteen categories, mask 1                             -> subset(1)
  1/256   one random row in 256 tagged 1, the rest 2, mask 1     -> subset(1)

Per point: the time of compact() / subset() itself (host clock between two device synchronisations, median of --builds runs; the
compacted / subset index is sized to the kept rows), then three variants in the same process, alternating round by round, each round
timed with CUDA events over enough calls for ~50 ms, until every variant has at least --seconds of timed work.  Reported: median ms
per call and the spread (min, max, p10, p90) over rounds.
  b  Stage1Index.topk(tags=mask) over all rows of the full index (the filtered search)
  d  Stage1Index.topk over the compacted / subset index: permanent ids, cir_stage1_index_topk_ids
  c  Stage1Index.topk over a separately built index of the eligible rows with no id table (r04's variant c; its row -> gallery row
     map is not timed), so d - c is the cost of the id mapping
Every point asserts b == d bit for bit (ids as returned, no host-side map) and b == c after the index map.  The gallery (1 GB fp32 +
0.5 GB bf16) is larger than the L2, so every call reads it from HBM.

    python tools/stage1_compact_probe.py --out profiles/r05_stage1_compact.json
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import cir_b200 as cir
from tools.stage1_filter_probe import selectivities
from tools.stage1_index_probe import device_info, stats, time_calls, unit


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, (time.perf_counter() - t0) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--G", type=int, default=1 << 20)
    ap.add_argument("--K", type=int, default=200)
    ap.add_argument("--Q", type=str, default="1,16,256,4181")
    ap.add_argument("--sel", type=str, default="rm10,1/3,1/16,1/256")
    ap.add_argument("--seconds", type=float, default=1.0, help="least timed work per (point, variant)")
    ap.add_argument("--builds", type=int, default=3, help="timed compact() / subset() runs per point")
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stage1_compact_probe needs a GPU")
    dev = torch.device("cuda", torch.cuda.current_device())
    eng = cir.engine.get_engine(dev, "bf16")
    G, K = a.G, a.K
    g = unit(G, 1, dev)
    idx = eng.stage1_index(G).add(g)
    res = {"device": device_info(), "G": G, "K": K, "precision": "bf16",
           "variants": {"b": "Stage1Index.topk(tags=mask) over all rows of the full index",
                        "d": "Stage1Index.topk over the compacted / subset index (permanent ids, cir_stage1_index_topk_ids)",
                        "c": "Stage1Index.topk over a separately built index of the eligible rows, no id table"},
           "build": "compact(): of a fresh copy of the full index with the point's tags; subset(mask, capacity=eligible rows)",
           "points": []}
    sels = selectivities(G, dev)
    for name in a.sel.split(","):
        tags, mask = sels[name]
        idx.set_tags(torch.arange(G, device=dev), tags)
        elig = torch.nonzero((tags & mask) != 0).flatten()
        n_elig = int(elig.numel())
        build_ms = []
        for _ in range(a.builds):
            if name == "rm10":
                copy = eng.stage1_index(G).add(g, tags=tags)
                sub, ms = timed(lambda: copy.compact(capacity=n_elig))
            else:
                sub, ms = timed(lambda: idx.subset(mask, capacity=n_elig))
            build_ms.append(ms)
        assert sub.rows == n_elig and torch.equal(sub.row_ids.long(), elig)
        plain = eng.stage1_index(n_elig).add(g[elig])
        for Q in [int(x) for x in a.Q.split(",")]:
            q = unit(Q, 100 + Q, dev)
            masks = torch.full((Q,), mask, dtype=torch.int32, device=dev)
            outs = {v: (torch.empty(Q, K, device=dev), torch.empty(Q, K, dtype=torch.int32, device=dev)) for v in "bdc"}
            exact = {v: torch.zeros(Q, dtype=torch.int32, device=dev) for v in "bd"}
            fns = {"b": lambda: idx.topk(q, K, out=outs["b"], exact_rows=exact["b"], tags=masks),
                   "d": lambda: sub.topk(q, K, out=outs["d"], exact_rows=exact["d"]),
                   "c": lambda: plain.topk(q, K, out=outs["c"])}
            for f in fns.values():                              # warm-up (and the workspaces)
                for _ in range(3):
                    f()
            torch.cuda.synchronize()

            def equal():
                i = outs["c"][1].long()
                mapped = torch.where(i >= 0, elig[i.clamp(min=0)], torch.full_like(i, -1)).int()
                bd = torch.equal(outs["b"][0], outs["d"][0]) and torch.equal(outs["b"][1], outs["d"][1])
                bc = torch.equal(outs["b"][0], outs["c"][0]) and torch.equal(outs["b"][1], mapped)
                return bool(bd), bool(bc)
            before = equal()
            assert all(before), f"{name} Q={Q}: (b == d, b == c) = {before}"
            per = {v: time_calls(fns[v], 1) for v in "bdc"}
            n = {v: max(1, int(50.0 / max(per[v], 1e-3))) for v in "bdc"}
            samples = {v: [] for v in "bdc"}
            spent = {v: 0.0 for v in "bdc"}
            while min(spent.values()) < a.seconds * 1e3 or min(len(s) for s in samples.values()) < 10:
                for v in "bdc":
                    ms = time_calls(fns[v], n[v])
                    samples[v].append(ms)
                    spent[v] += ms * n[v]
            torch.cuda.synchronize()
            after = equal()
            assert all(after), f"{name} Q={Q}: (b == d, b == c) = {after} after timing"
            pt = {"selectivity": name, "operation": "compact" if name == "rm10" else "subset", "eligible_rows": n_elig, "Q": Q,
                  "build_ms": stats(build_ms), "bit_equal_b_d": True, "bit_equal_b_c": True,
                  "exact_fallback_queries": {v: int(exact[v].sum()) for v in "bd"}, "calls_per_round": n,
                  "timed_s": {v: spent[v] / 1e3 for v in "bdc"}}
            for v in "bdc":
                pt[v] = stats(samples[v])
            pt["b_over_d"] = pt["b"]["median_ms"] / pt["d"]["median_ms"]
            pt["d_minus_c_ms"] = pt["d"]["median_ms"] - pt["c"]["median_ms"]
            res["points"].append(pt)
            print(json.dumps({k: pt[k] for k in ("selectivity", "Q", "b_over_d", "d_minus_c_ms")}
                             | {"build_ms": round(pt["build_ms"]["median_ms"], 3)}
                             | {v: round(pt[v]["median_ms"], 4) for v in "bdc"}), flush=True)
        del sub, plain
        if name == "rm10":
            del copy
    res["device_after"] = device_info()
    js = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(js + "\n")
    print(js)


if __name__ == "__main__":
    main()
