"""Stage-II scoring through an MXFP8 K/V gallery (Stage2KVCache(fp8=True)) against the bf16 gallery and the uncached per-chunk K/V
projection.  One GPU, the bench's synthetic weights (make_stage{1,2}_state_dict(0, 384, "reference")), G = 2,297 gallery images of
N = 577 random bf16 tokens, captions of L = 32, random z_t -- the setting of profiles/r06 and r07.

Reported:
  cache     bytes per image and the time of one fill of all G rows (host clock between two device synchronisations, median of
            --fills runs) for both formats
  score     the r06 points (BLIP_NLVR.score_triplets): the Fashion-IQ job (Q = 2,017 x K = 100, bench.synth_workload), reuse_1
            (22 x 100 disjoint candidates) and online Q in {1, 16} x K in {50, 100}, chunks bounded by r06's max_candidates (64,
            512, 4,096; the bf16 cache ignores it); arms uncached / bf16 cache / fp8 cache
            alternated round by round in that order, each round timed with the host clock around calls that end in a device
            synchronise; max |score(fp8) - score(bf16)| per point
  rerank    the r07 points (BLIP_NLVR.rerank_topk on the stage-I top-K, device-planned): Q in {1, 4, 16, 64} x K in {50, 100},
            bf16 and fp8 cache alternated
  capacity  G = 6,000 rows, which only the fp8 format holds on one GPU next to the tokens (bf16 would need 255 GB): fill time, and
            the replay latency of the captured online chain (stage-I encode -> Stage1Index.topk -> rerank_topk) for 1 x 50,
            host clock around a replay that ends in a device synchronise
Times are medians with p10-p90 over the rounds.  Every cache is far larger than the L2.

    python tools/stage2_kv_fp8_probe.py --out profiles/r08_stage2_kv_fp8.json
"""
import argparse
import json
import os
import sys
from types import SimpleNamespace

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import cir_b200 as cir
from bench import synth_workload
from tools.stage1_index_probe import device_info
from tools.stage2_kv_cache_probe import spread, wall_ms


def random_tokens(G, N, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    tokens = torch.empty(G, N, 768, dtype=torch.bfloat16, device=dev)
    for g0 in range(0, G, 256):
        tokens[g0:g0 + 256] = torch.randn(tokens[g0:g0 + 256].shape, generator=g, device=dev).bfloat16()
    return tokens


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--G", type=int, default=2297)
    ap.add_argument("--G-capacity", type=int, default=6000)
    ap.add_argument("--L", type=int, default=32)
    ap.add_argument("--fills", type=int, default=3)
    ap.add_argument("--rounds-fiq", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=12)
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stage2_kv_fp8_probe needs a GPU")
    dev = torch.device("cuda", torch.cuda.current_device())
    syn = cir.synthetic
    G, L, N = a.G, a.L, 577
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=syn.make_stage1_state_dict(0, 384, "reference"), precision="bf16",
                                     device=dev)
    m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=syn.make_stage2_state_dict(0, 384, "reference"), precision="bf16",
                                     device=dev)
    eng = m2.engine
    res = {"device": device_info(), "G": G, "N": N, "L": L, "precision": "bf16",
           "weights": "make_stage{1,2}_state_dict(0, 384, 'reference')"}
    tokens = random_tokens(G, N, dev, 1)

    caches, res["cache"] = {}, {}
    for name, fp8 in (("bf16", False), ("fp8", True)):
        caches[name], _ = wall_ms(lambda: m2.kv_cache(tokens, fp8=fp8))
        fills = [wall_ms(lambda: caches[name].fill(tokens, 0))[1] for _ in range(a.fills)]
        res["cache"][name] = {"bytes": caches[name].nbytes, "bytes_per_image": caches[name].nbytes // G,
                              "fill_ms": float(np.median(fills)), "fill_ms_runs": fills}
    print(json.dumps(res["cache"]), flush=True)

    def queries(Q, seed):
        ids, mask = syn.make_token_ids(Q, L, seed=seed, min_len=12)
        ids[:, 0] = syn.ENC_TOKEN_ID
        z = torch.randn(Q, L, 768, generator=torch.Generator().manual_seed(seed)).to(dev).bfloat16()
        return z, ids.int().to(dev), mask.int().to(dev)

    def score_point(name, z, ids, mask, cand, active, rounds, max_candidates):
        n_trip = int(cand.shape[1] * (cand.shape[0] if active is None else int(np.sum(active))))
        old = eng.max_candidates

        def run(kv):             # the fp8 arm's chunks hold their dequantised K/V, so it takes the uncached arm's bound
            eng.max_candidates = max_candidates
            try:
                return m2.score_triplets(z, ids, mask, tokens, cand, active, kv_cache=kv)
            finally:
                eng.max_candidates = old
        arms = {"uncached": None, "bf16": caches["bf16"], "fp8": caches["fp8"]}
        out, plans = {}, {}
        for k, kv in arms.items():                                            # warm-up and results
            out[k], _ = wall_ms(lambda: run(kv))
            plans[k] = {q: eng.last_plan[q] for q in ("chunks", "candidate_loads")}
        ms = {k: [] for k in arms}
        for _ in range(rounds):
            for k, kv in arms.items():
                ms[k].append(wall_ms(lambda: run(kv))[1])
        act = torch.ones_like(out["bf16"], dtype=torch.bool) if active is None else torch.from_numpy(np.asarray(active)).to(dev)
        d = (out["fp8"] - out["bf16"])[act]
        pt = {"point": name, "Q": int(cand.shape[0]), "K": int(cand.shape[1]), "triplets": n_trip, "plans": plans,
              "bf16_cache_equals_uncached": bool(torch.equal(out["uncached"], out["bf16"])),
              "max_abs_dscore_fp8_vs_bf16": float(d.abs().max()), "mean_abs_dscore_fp8_vs_bf16": float(d.abs().mean())}
        pt.update({k: spread(v, n_trip) for k, v in ms.items()})
        print(json.dumps({k: pt[k] for k in ("point", "Q", "K", "max_abs_dscore_fp8_vs_bf16")}
                         | {k + "_ms": round(pt[k]["median_ms"], 3) for k in arms}), flush=True)
        return pt

    hg = torch.Generator().manual_seed(7)
    pts = []
    ref, tgt, ids, mask, cand, labels = synth_workload(SimpleNamespace(queries=2017, k=100, gallery=G, length=L))
    z = torch.randn(2017, L, 768, generator=hg).to(dev).bfloat16()
    pts.append(score_point("fiq", z, ids.to(dev), mask.to(dev), cand.numpy(), labels.any(1).numpy(), a.rounds_fiq, eng.max_candidates))
    del z
    z, ids, mask = queries(22, 11)
    perm = torch.randperm(G, generator=hg)[: 22 * 100].view(22, 100).int().numpy()
    pts.append(score_point("reuse_1", z, ids, mask, perm, None, a.rounds, 512))
    for Q in (1, 16):
        z, ids, mask = queries(Q, 20 + Q)
        for K in (50, 100):
            cand = torch.stack([torch.randperm(G, generator=hg)[:K] for _ in range(Q)]).int().numpy()
            pts.append(score_point(f"online_Q{Q}_K{K}", z, ids, mask, cand, None, a.rounds, 4096))
    res["score"] = pts

    # r07: rerank_topk on the stage-I top-K of each point's queries.  Both galleries stay resident (148 GB), so the batch path's
    # workspace is released, and so is every outgrown re-rank workspace (no graph is captured here that could still use one).
    eng._ws = None
    torch.cuda.empty_cache()
    index = m1.engine.stage1_index(G).add(m1.engine.stage1_gallery_embed(m1._w, tokens))
    eng.max_triplets = 16384
    rr = []
    for Q in (1, 4, 16, 64):
        for K in (50, 100):
            hq = torch.Generator().manual_seed(1000 * Q + K)
            ref = torch.randperm(G, generator=hq)[:Q].int().to(dev)
            ids, mask = syn.make_token_ids(Q, L, seed=Q + K, min_len=12)
            ids[:, 0] = syn.ENC_TOKEN_ID
            ids, mask = ids.int().to(dev), mask.int().to(dev)
            z_t, q_emb = eng.stage1_encode(m1._w, tokens, ref, ids, mask)
            _, cand = index.topk(q_emb, K, exclude=ref)
            out = {k: wall_ms(lambda: m2.rerank_topk(z_t, ids, mask, cand, caches[k]))[0] for k in ("bf16", "fp8")}
            ms = {k: [] for k in ("bf16", "fp8")}
            for _ in range(a.rounds):
                for k in ms:
                    ms[k].append(wall_ms(lambda: m2.rerank_topk(z_t, ids, mask, cand, caches[k]))[1])
            pt = {"Q": Q, "K": K, "triplets": Q * K, "unique_candidates": int(torch.unique(cand).numel()),
                  "max_abs_dscore_fp8_vs_bf16": float((out["fp8"][0] - out["bf16"][0]).abs().max()),
                  "same_order": bool(torch.equal(out["fp8"][1], out["bf16"][1]))}
            pt.update({k: spread(v, Q * K) for k, v in ms.items()})
            rr.append(pt)
            eng._rr_retired.clear()
            print(json.dumps({k: pt[k] for k in ("Q", "K", "max_abs_dscore_fp8_vs_bf16")}
                             | {k + "_ms": round(pt[k]["median_ms"], 3) for k in ms}), flush=True)
    res["rerank"] = rr
    del caches, index, tokens
    eng._rr_ws = None
    torch.cuda.empty_cache()

    # capacity: a gallery only the fp8 format fits on one GPU
    Gc = a.G_capacity
    tokens = random_tokens(Gc, N, dev, 2)
    kv, fill_ms = wall_ms(lambda: m2.kv_cache(tokens, fp8=True))
    index = m1.engine.stage1_index(Gc).add(m1.engine.stage1_gallery_embed(m1._w, tokens))
    chain = cir.online.OnlineReranker(m1, m2, tokens, index, kv)
    cap = chain.capture(1, L, 50)
    ms = []
    for r in range(a.rounds + 2):
        hq = torch.Generator().manual_seed(500 + r)
        ref = torch.randperm(Gc, generator=hq)[:1].int()
        ids, mask = syn.make_token_ids(1, L, seed=500 + r, min_len=12)
        ids[:, 0] = syn.ENC_TOKEN_ID
        ms.append(wall_ms(lambda: cap(ref, ids.int(), mask.int()))[1])
    res["capacity"] = {"G": Gc, "token_bytes": tokens.numel() * 2, "fp8_cache_bytes": kv.nbytes,
                       "bf16_cache_bytes_would_be": int(eng._lib.cir_stage2_kv_cache_bytes(eng.ctx, Gc, N)),
                       "fill_ms_with_alloc": fill_ms, "chain_1x50_replay": spread(ms[2:], 50),
                       "max_memory_allocated": torch.cuda.max_memory_allocated(dev)}
    print(json.dumps(res["capacity"]), flush=True)
    res["device_after"] = device_info()
    js = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(js + "\n")


if __name__ == "__main__":
    main()
