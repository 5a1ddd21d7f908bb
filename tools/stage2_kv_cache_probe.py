"""Stage-II scoring through the resident cross-attention K/V gallery (Stage2KVCache) against the per-chunk K/V projection it
replaces.  One GPU, the bench's synthetic weights (make_stage2_state_dict(0, 384, "reference")), G = 2,297 gallery images of
N = 577 random bf16 tokens, captions of L = 32, random z_t.

Reported: the cache bytes and the time of one fill of all G rows (host clock between two device synchronisations, median of
--fills runs), then per point the cached and the uncached call of BLIP_NLVR.score_triplets on the same inputs, alternating the two
round by round (the uncached one first), each round timed with the host clock around calls that end in a device synchronise.
Points:
  fiq       the bench's Fashion-IQ job: Q = 2,017 x K = 100 stage-I-like lists (bench.synth_workload), ~2 % of the rows inactive;
            uncached with the default chunk limits (max_candidates = 64)
  reuse_1   the bench's extras.reuse_1 shape: 22 queries x 100 disjoint candidates; uncached with max_candidates = 512 as there
  online    Q in {1, 16} x K in {50, 100} distinct random candidates per query, one chunk each
Every point records whether the cached scores equal the uncached ones bit for bit, and both chunk plans.  The K/V cache (98 GB)
and the token gallery (2 GB) are far larger than the L2.

    python tools/stage2_kv_cache_probe.py --out profiles/r06_stage2_kv_cache.json
"""
import argparse
import json
import os
import sys
import time
from types import SimpleNamespace

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import cir_b200 as cir
from bench import synth_workload
from tools.stage1_index_probe import device_info


def wall_ms(fn, n=1):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        r = fn()
    torch.cuda.synchronize()
    return r, (time.perf_counter() - t0) * 1e3 / n


def spread(ms, triplets):
    v = np.asarray(ms)
    tps = triplets / (v / 1e3)
    return {"median_ms": float(np.median(v)), "p10_ms": float(np.percentile(v, 10)), "p90_ms": float(np.percentile(v, 90)),
            "median_triplets_per_s": float(np.median(tps)), "p10_triplets_per_s": float(np.percentile(tps, 10)),
            "p90_triplets_per_s": float(np.percentile(tps, 90)), "rounds": int(v.size)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--G", type=int, default=2297)
    ap.add_argument("--L", type=int, default=32)
    ap.add_argument("--fills", type=int, default=3)
    ap.add_argument("--rounds-fiq", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=12, help="rounds of the reuse-1 and online points")
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stage2_kv_cache_probe needs a GPU")
    dev = torch.device("cuda", torch.cuda.current_device())
    syn = cir.synthetic
    G, L, N = a.G, a.L, 577
    m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=syn.make_stage2_state_dict(0, 384, "reference"), precision="bf16",
                                     device=dev)
    eng = m2.engine
    g = torch.Generator(device=dev).manual_seed(1)
    tokens = torch.empty(G, N, 768, dtype=torch.bfloat16, device=dev)
    for g0 in range(0, G, 256):
        tokens[g0:g0 + 256] = torch.randn(tokens[g0:g0 + 256].shape, generator=g, device=dev).bfloat16()
    res = {"device": device_info(), "G": G, "N": N, "L": L, "precision": "bf16", "weights": "make_stage2_state_dict(0, 384, 'reference')"}

    cache, _ = wall_ms(lambda: m2.kv_cache(tokens))
    fills = [wall_ms(lambda: cache.fill(tokens, 0))[1] for _ in range(a.fills)]
    res["cache"] = {"bytes": cache.nbytes, "bytes_per_image": cache.nbytes // G, "fill_ms": float(np.median(fills)), "fill_ms_runs": fills,
                    "fill_flop": 2.0 * G * N * 3072 * 768 * 12}
    res["cache"]["fill_tflops"] = res["cache"]["fill_flop"] / (res["cache"]["fill_ms"] / 1e3) / 1e12
    print(json.dumps(res["cache"]), flush=True)

    hg = torch.Generator().manual_seed(7)

    def queries(Q, seed):
        ids, mask = syn.make_token_ids(Q, L, seed=seed, min_len=12)
        ids[:, 0] = syn.ENC_TOKEN_ID
        z = torch.randn(Q, L, 768, generator=torch.Generator().manual_seed(seed)).to(dev).bfloat16()
        return z, ids.int().to(dev), mask.int().to(dev)

    def point(name, z, ids, mask, cand, active, rounds, max_candidates):
        n_trip = int(cand.shape[1] * (cand.shape[0] if active is None else int(np.sum(active))))
        old = eng.max_candidates

        def run(kv):
            eng.max_candidates = max_candidates if kv is None else old
            try:
                return m2.score_triplets(z, ids, mask, tokens, cand, active, kv_cache=kv)
            finally:
                eng.max_candidates = old
        base, _ = wall_ms(lambda: run(None))                                  # warm-up of both, and the equality check
        plan_u = dict(eng.last_plan)
        got, _ = wall_ms(lambda: run(cache))
        plan_c = dict(eng.last_plan)
        ms_u, ms_c = [], []
        for _ in range(rounds):
            ms_u.append(wall_ms(lambda: run(None))[1])
            ms_c.append(wall_ms(lambda: run(cache))[1])
        pt = {"point": name, "Q": int(cand.shape[0]), "K": int(cand.shape[1]), "triplets": n_trip,
              "bit_equal": bool(torch.equal(base, got)), "max_abs_diff": float((base - got).abs().max()),
              "plan_uncached": {k: plan_u[k] for k in ("chunks", "candidate_loads")},
              "plan_cached": {k: plan_c[k] for k in ("chunks", "candidate_loads")},
              "uncached": spread(ms_u, n_trip), "cached": spread(ms_c, n_trip)}
        pt["speedup_median"] = pt["uncached"]["median_ms"] / pt["cached"]["median_ms"]
        print(json.dumps({k: pt[k] for k in ("point", "Q", "K", "bit_equal", "speedup_median")}
                         | {"uncached_tps": pt["uncached"]["median_triplets_per_s"], "cached_tps": pt["cached"]["median_triplets_per_s"]}),
              flush=True)
        return pt

    pts = []
    ref, tgt, ids, mask, cand, labels = synth_workload(SimpleNamespace(queries=2017, k=100, gallery=G, length=L))
    z = torch.randn(2017, L, 768, generator=hg).to(dev).bfloat16()
    pts.append(point("fiq", z, ids.to(dev), mask.to(dev), cand.numpy(), labels.any(1).numpy(), a.rounds_fiq, eng.max_candidates))
    del z
    z, ids, mask = queries(22, 11)
    perm = torch.randperm(G, generator=hg)[: 22 * 100].view(22, 100).int().numpy()
    pts.append(point("reuse_1", z, ids, mask, perm, None, a.rounds, 512))
    for Q in (1, 16):
        z, ids, mask = queries(Q, 20 + Q)
        for K in (50, 100):
            cand = torch.stack([torch.randperm(G, generator=hg)[:K] for _ in range(Q)]).int().numpy()
            pts.append(point(f"online_Q{Q}_K{K}", z, ids, mask, cand, None, a.rounds, 4096))
    res["points"] = pts
    res["device_after"] = device_info()
    js = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(js + "\n")
    print("all bit-equal:", all(p["bit_equal"] for p in pts))


if __name__ == "__main__":
    main()
