"""Filtered stage-I search over a 1M-row resident index against the two alternatives: the unfiltered search of the same index, and
a separately built index of only the eligible rows (what a user does without row tags).  One GPU, G = 1,048,576 unit rows,
K = 200, Q in {1, 16, 256, 4181}.

Selectivities (the fraction of rows a query may return; every query of a point uses the same mask):
  all     every row tagged 0xFFFFFFFF, mask 0xFFFFFFFF
  1/3     three disjoint categories (tags 1 / 2 / 4, rows assigned at random, as in Fashion-IQ), mask 1
  1/16    sixteen disjoint categories (tags 1 << c, rows assigned at random), mask 1
  1/256   one random row in 256 tagged 1, the rest 2, mask 1
  rm10    10 % of the rows removed (tag 0), mask 0xFFFFFFFF

For each (selectivity, Q) three variants run in the same process, alternating round by round, each round timed with CUDA events
over enough calls for ~50 ms; rounds continue until every variant has at least --seconds of timed work.  Reported: median ms per
call and the spread (min, max, p10, p90) over rounds.
  a  Stage1Index.topk over all rows, no tags (the unfiltered search)
  b  Stage1Index.topk(tags=mask) over all rows (the filtered search)
  c  Stage1Index.topk over a separate index of the eligible rows only (built once, outside the timing; its row -> gallery row
     map is not timed either)
Every point asserts that b equals c bit for bit after the index map, and records how many queries took the exact fallback.
The gallery (1 GB fp32 + 0.5 GB bf16) is larger than the L2, so every call reads it from HBM.

    python tools/stage1_filter_probe.py --out profiles/r04_stage1_filter.json
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import cir_b200 as cir
from tools.stage1_index_probe import device_info, stats, time_calls, unit

ALL = -1      # 0xFFFFFFFF as an int32 bit pattern


def selectivities(G, dev):
    gen = torch.Generator(device=dev).manual_seed(7)
    r = torch.randint(0, 1 << 30, (G,), generator=gen, device=dev)
    bit = lambda c: torch.bitwise_left_shift(torch.ones_like(c), c).int()
    return {                                                   # name -> (row tags, query mask)
        "all": (torch.full((G,), ALL, dtype=torch.int32, device=dev), ALL),
        "1/3": (bit(r % 3), 1),
        "1/16": (bit(r % 16), 1),
        "1/256": (torch.where(r % 256 == 0, 1, 2).int(), 1),
        "rm10": (torch.where(r % 10 == 0, 0, ALL).int(), ALL),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--G", type=int, default=1 << 20)
    ap.add_argument("--K", type=int, default=200)
    ap.add_argument("--Q", type=str, default="1,16,256,4181")
    ap.add_argument("--sel", type=str, default="all,1/3,1/16,1/256,rm10")
    ap.add_argument("--seconds", type=float, default=1.0, help="least timed work per (point, variant)")
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stage1_filter_probe needs a GPU")
    dev = torch.device("cuda", torch.cuda.current_device())
    eng = cir.engine.get_engine(dev, "bf16")
    G, K = a.G, a.K
    g = unit(G, 1, dev)
    idx = eng.stage1_index(G).add(g)
    res = {"device": device_info(), "G": G, "K": K, "precision": "bf16",
           "variants": {"a": "Stage1Index.topk over all rows, no tags", "b": "Stage1Index.topk(tags=mask) over all rows",
                        "c": "Stage1Index.topk over a separate index of the eligible rows only"},
           "points": []}
    sels = selectivities(G, dev)
    for name in a.sel.split(","):
        tags, mask = sels[name]
        idx.set_tags(torch.arange(G, device=dev), tags)
        elig = torch.nonzero((tags & mask) != 0).flatten()
        sub = eng.stage1_index(elig.numel()).add(g[elig])
        for Q in [int(x) for x in a.Q.split(",")]:
            q = unit(Q, 100 + Q, dev)
            masks = torch.full((Q,), mask, dtype=torch.int32, device=dev)
            outs = {v: (torch.empty(Q, K, device=dev), torch.empty(Q, K, dtype=torch.int32, device=dev)) for v in "abc"}
            exact = torch.zeros(Q, dtype=torch.int32, device=dev)
            fns = {"a": lambda: idx.topk(q, K, out=outs["a"]),
                   "b": lambda: idx.topk(q, K, out=outs["b"], exact_rows=exact, tags=masks),
                   "c": lambda: sub.topk(q, K, out=outs["c"])}
            for f in fns.values():                              # warm-up (and the workspaces)
                for _ in range(3):
                    f()
            torch.cuda.synchronize()

            def equal_b_c():
                i = outs["c"][1].long()
                mapped = torch.where(i >= 0, elig[i.clamp(min=0)], torch.full_like(i, -1)).int()
                return bool(torch.equal(outs["b"][1], mapped) and torch.equal(outs["b"][0], outs["c"][0]))
            same = equal_b_c()
            assert same, f"{name} Q={Q}: filtered search differs from the compacted index"
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
            same_after = equal_b_c()
            assert same_after, f"{name} Q={Q}: filtered search differs from the compacted index after timing"
            pt = {"selectivity": name, "eligible_rows": int(elig.numel()), "Q": Q, "bit_equal_b_c": bool(same and same_after),
                  "exact_fallback_queries_b": int(exact.sum()), "calls_per_round": n, "timed_s": {v: spent[v] / 1e3 for v in "abc"}}
            for v in "abc":
                pt[v] = stats(samples[v])
            pt["b_over_a"] = pt["b"]["median_ms"] / pt["a"]["median_ms"]
            pt["b_over_c"] = pt["b"]["median_ms"] / pt["c"]["median_ms"]
            res["points"].append(pt)
            print(json.dumps({k: pt[k] for k in ("selectivity", "Q", "bit_equal_b_c", "exact_fallback_queries_b", "b_over_a", "b_over_c")}
                             | {v: round(pt[v]["median_ms"], 4) for v in "abc"}), flush=True)
        del sub
    res["device_after"] = device_info()
    js = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(js + "\n")
    print(js)


if __name__ == "__main__":
    main()
