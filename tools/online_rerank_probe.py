"""Online re-ranking of a device-resident top-K list: the host-planned stage-II call against the on-device plan, eager and from a
CUDA graph, and the whole online chain.  One GPU, the bench's synthetic weights (make_stage{1,2}_state_dict(0, 384, "reference")),
a resident K/V gallery of G = 2,297 images of N = 577 random bf16 tokens, a stage-I index of their embeddings, captions of L = 32.

Points Q in {1, 4, 16, 64} x K in {50, 100}; the candidates of a point are the stage-I top-K of its queries (a device tensor),
every point runs as one stage-II chunk / call (max_triplets = 16,384).  Arms, alternated round by round in this order, each timed
with the host clock around a call that ends in a device synchronise (median and p10-p90 over --rounds):
  a_host     BLIP_NLVR.score_triplets(kv_cache=) + rerank_sort: device -> host read of the top-K, host planning, one upload, launches
  b_device   BLIP_NLVR.rerank_topk eager: plan on the device, launches from Python, no host read
  c_graph    b_device replayed from a CUDA graph
  d_chain    stage-I encode -> Stage1Index.topk -> rerank_topk (online.OnlineReranker), eager
  d_graph    d_chain replayed from a CUDA graph (CapturedQuery, new inputs copied in first)
Also per point: host_plan_ms, the numpy planning alone (plan_chunks + the three work lists) on the same candidates, and
c_graph_device_ms, the graph replay timed with CUDA events over --rounds back-to-back replays.  Scores and order of a, b and c are
compared bit for bit at every point, and the replayed chain against the eager one.  The cache (98 GB) is far larger than the L2.

    python tools/online_rerank_probe.py --out profiles/r07_online_rerank.json
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import cir_b200 as cir
from tools.stage1_index_probe import device_info
from tools.stage2_kv_cache_probe import spread, wall_ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--G", type=int, default=2297)
    ap.add_argument("--L", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--Q", type=int, nargs="+", default=[1, 4, 16, 64])
    ap.add_argument("--K", type=int, nargs="+", default=[50, 100])
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("online_rerank_probe needs a GPU")
    dev = torch.device("cuda", torch.cuda.current_device())
    syn, S = cir.synthetic, cir.schedule
    G, L, N = a.G, a.L, 577
    res = {"device": device_info(), "G": G, "N": N, "L": L, "precision": "bf16",
           "weights": "make_stage{1,2}_state_dict(0, 384, 'reference')"}
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=syn.make_stage1_state_dict(0, 384, "reference"), precision="bf16",
                                     device=dev)
    m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=syn.make_stage2_state_dict(0, 384, "reference"), precision="bf16",
                                     device=dev)
    eng = m2.engine
    eng.max_triplets = 16384
    g = torch.Generator(device=dev).manual_seed(1)
    tokens = torch.empty(G, N, 768, dtype=torch.bfloat16, device=dev)
    for g0 in range(0, G, 256):
        tokens[g0:g0 + 256] = torch.randn(tokens[g0:g0 + 256].shape, generator=g, device=dev).bfloat16()
    kv = m2.kv_cache(tokens)
    index = m1.engine.stage1_index(G).add(m1.engine.stage1_gallery_embed(m1._w, tokens))
    chain = cir.online.OnlineReranker(m1, m2, tokens, index, kv)
    torch.cuda.synchronize()

    pts = []
    for Q in a.Q:
        for K in a.K:
            hg = torch.Generator().manual_seed(1000 * Q + K)
            ref = torch.randperm(G, generator=hg)[:Q].int().to(dev)
            ids, mask = syn.make_token_ids(Q, L, seed=Q + K, min_len=12)
            ids[:, 0] = syn.ENC_TOKEN_ID
            ids, mask = ids.int().to(dev), mask.int().to(dev)
            z_t, q_emb = eng.stage1_encode(m1._w, tokens, ref, ids, mask)
            _, cand = index.topk(q_emb, K, exclude=ref)
            out = (torch.empty(Q, K, device=dev), torch.empty(Q, K, dtype=torch.int32, device=dev),
                   torch.empty(Q, K, dtype=torch.int32, device=dev))

            def arm_a():
                s = m2.score_triplets(z_t, ids, mask, tokens, cand, kv_cache=kv)
                return s, eng.rerank_sort(s)

            def arm_b():
                return m2.rerank_topk(z_t, ids, mask, cand, kv, out=out)

            (sa, oa), _ = wall_ms(arm_a)
            plan_a = dict(eng.last_plan)
            wall_ms(arm_b)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                arm_b()
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                arm_b()
            cap = chain.capture(Q, L, K)
            eq = {}
            (sb, ob, _), _ = wall_ms(arm_b)
            eq["b"] = bool(torch.equal(sa, sb) and torch.equal(oa, ob))
            sb, ob = sb.clone(), ob.clone()
            out[0].zero_(), out[1].zero_()
            wall_ms(graph.replay)
            eq["c"] = bool(torch.equal(sa, out[0]) and torch.equal(oa, out[1]))
            (r_eager, s_eager, d_eager), _ = wall_ms(lambda: chain(ref, ids, mask, K))
            (r_graph, s_graph, d_graph), _ = wall_ms(lambda: cap(ref, ids, mask))
            eq["d_graph_vs_d_chain"] = bool(torch.equal(r_eager, r_graph) and torch.equal(s_eager, s_graph) and torch.equal(d_eager, d_graph))
            eq["d_chain_vs_a"] = bool(torch.equal(s_eager, sa))

            cand_np = cand.cpu().numpy()
            t0 = time.perf_counter()
            for _ in range(a.rounds):
                for ch in S.plan_chunks(cand_np, None, eng.max_triplets, max(1, Q * K)):
                    S.build_attn_work(ch.trip_slot, L), S.build_attn_tiles(ch.trip_slot, L), S.build_attn_tiles(ch.trip_slot, 1)
            host_plan_ms = (time.perf_counter() - t0) * 1e3 / a.rounds

            ms = {k: [] for k in ("a_host", "b_device", "c_graph", "d_chain", "d_graph")}
            for _ in range(a.rounds):
                ms["a_host"].append(wall_ms(arm_a)[1])
                ms["b_device"].append(wall_ms(arm_b)[1])
                ms["c_graph"].append(wall_ms(graph.replay)[1])
                ms["d_chain"].append(wall_ms(lambda: chain(ref, ids, mask, K))[1])
                ms["d_graph"].append(wall_ms(lambda: cap(ref, ids, mask))[1])
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(a.rounds):
                graph.replay()
            e1.record()
            e1.synchronize()
            pt = {"Q": Q, "K": K, "triplets": Q * K, "plan_host": {k: plan_a[k] for k in ("chunks", "candidate_loads")},
                  "bit_equal": eq, "host_plan_ms": host_plan_ms, "c_graph_device_ms": e0.elapsed_time(e1) / a.rounds}
            pt.update({k: spread(v, Q * K) for k, v in ms.items()})
            pts.append(pt)
            print(json.dumps({"Q": Q, "K": K, "bit_equal": eq, "host_plan_ms": round(host_plan_ms, 3),
                              "graph_device_ms": round(pt["c_graph_device_ms"], 3)}
                             | {k: round(pt[k]["median_ms"], 3) for k in ms}), flush=True)
            del graph, cap
    res["points"] = pts
    res["device_after"] = device_info()
    js = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(js + "\n")
    print("all bit-equal:", all(all(p["bit_equal"].values()) for p in pts))


if __name__ == "__main__":
    main()
