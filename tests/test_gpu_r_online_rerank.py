"""Re-ranking a device-resident top-K list through the K/V gallery without the host (cir_stage2_plan_topk, cir_stage2_rerank_cached,
Engine.stage2_rerank_cached, BLIP_NLVR.rerank_topk, online.OnlineReranker).

The device planner must reproduce the host planner (schedule.plan_chunks as one chunk + build_attn_tiles) entry for entry; the
re-ranked scores and order must equal the host-planned cached path of the same single chunk + rerank_sort, bit for bit; and the
whole online chain must replay from a CUDA graph with new inputs and give the eager chain's result."""
import ctypes as C

import numpy as np
import pytest
import torch

import cir_b200 as cir
from helpers import golden_images, golden_weights, load_golden

pytestmark = pytest.mark.gpu
syn = cir.synthetic
S = cir.schedule
N = cir.native
NTOK = 577
NEG = np.float32(cir.engine.NEG_FILL)


def _models(precision):
    sd1, sd2 = golden_weights(load_golden("pipeline_small.npz"))
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd1, precision=precision)
    m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision=precision)
    return m1, m2


@pytest.fixture(scope="module")
def bf16():
    m1, m2 = _models("bf16")
    g = torch.Generator().manual_seed(61)
    tokens = torch.randn(80, NTOK, 768, generator=g).cuda().bfloat16()
    return m1, m2, tokens, m2.kv_cache(tokens)


@pytest.fixture(scope="module")
def fp32():
    m1, m2 = _models("fp32")
    g = torch.Generator().manual_seed(62)
    tokens = torch.randn(12, NTOK, 768, generator=g).cuda()
    return m1, m2, tokens, m2.kv_cache(tokens)


def _queries(eng, Q, L, seed):
    g = torch.Generator().manual_seed(seed)
    ids, mask = syn.make_token_ids(Q, L, seed=seed, min_len=max(1, L // 2))
    ids[:, 0] = syn.ENC_TOKEN_ID
    z_t = torch.randn(Q, L, 768, generator=g).cuda().to(eng.act_dtype)
    return z_t, ids.int().cuda(), mask.int().cuda()


def _rand_cand(Q, K, lo, hi, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(lo, hi, (Q, K), generator=g).int().numpy()


# ---------------------------------------------------------------------------------------------------------------- planner
def _device_plan(eng, cand, L, row0, rows):
    Q, K = cand.shape
    T = Q * K
    c = torch.from_numpy(np.ascontiguousarray(cand, dtype=np.int32)).cuda()
    i32 = dict(dtype=torch.int32, device=eng.device)
    fp, kv, tq, counts = torch.full((T,), -7, **i32), torch.full((T,), -7, **i32), torch.full((T,), -7, **i32), torch.full((3,), -7, **i32)
    tiles, tiles_cls = torch.full((T, 4), -7, **i32), torch.full((T, 4), -7, **i32)
    eng._sync_stream()
    N.check(eng._lib.cir_stage2_plan_topk(eng.ctx, N.ptr(c), Q, K, L, row0, rows, N.ptr(fp), N.ptr(kv), N.ptr(tq), N.ptr(tiles),
                                          N.ptr(tiles_cls), N.ptr(counts)), "cir_stage2_plan_topk")
    torch.cuda.synchronize()
    n = counts.cpu().numpy()
    return fp.cpu().numpy(), kv.cpu().numpy(), tq.cpu().numpy(), tiles.cpu().numpy(), tiles_cls.cpu().numpy(), n


def _plan_cases():
    r = np.random.default_rng(5)
    long_run = r.integers(0, 400, (40, 20)).astype(np.int32)
    long_run[:, :10] = 7                                                     # a run of 400 triplets: longer than G and than 256
    dup = r.integers(0, 30, (12, 9)).astype(np.int32)
    dup[:, 3] = dup[:, 1]                                                    # the same candidate twice within a list
    return {
        "reuse_heavy_64x50": r.integers(0, 10, (64, 50)).astype(np.int32),
        "reuse_1": r.permutation(5000)[:30 * 40].reshape(30, 40).astype(np.int32),
        "one_candidate": np.full((9, 13), 4, np.int32),
        "dup_in_row": dup,
        "q1": r.integers(0, 60, (1, 100)).astype(np.int32),
        "long_run": long_run,
        "max_T_64x256": r.integers(0, 3000, (64, 256)).astype(np.int32),
    }


PLAN_CASES = _plan_cases()


@pytest.mark.parametrize("L", [8, 16, 24, 32, 40])
@pytest.mark.parametrize("case", list(PLAN_CASES))
def test_plan_equals_host_planner(case, L, bf16):
    eng = bf16[1].engine
    cand = PLAN_CASES[case]
    Q, K = cand.shape
    ch = S.plan_chunks(cand, None, 1 << 20, 1 << 20)
    assert len(ch) == 1
    ch = ch[0]
    row0 = 0
    fp, kv, tq, tiles, tiles_cls, n = _device_plan(eng, cand, L, row0, 5000)
    want_t, want_c = S.build_attn_tiles(ch.trip_slot, L), S.build_attn_tiles(ch.trip_slot, 1)
    assert np.array_equal(fp, ch.flat_pos)
    assert np.array_equal(kv, ch.cand_list[ch.trip_slot] - row0)
    assert np.array_equal(ch.query_list, np.arange(Q)) and np.array_equal(tq, ch.trip_query)
    assert n.tolist() == [want_t.shape[0], want_c.shape[0], 0]
    assert np.array_equal(tiles[: n[0]], want_t) and np.array_equal(tiles_cls[: n[1]], want_c)
    assert (tiles[n[0]:] == -7).all() and (tiles_cls[n[1]:] == -7).all()                  # nothing written past the counts


def test_plan_with_invalid_entries(bf16):
    eng = bf16[1].engine
    r = np.random.default_rng(9)
    Q, K, row0, rows, L = 20, 30, 100, 50, 24
    cand = r.integers(row0, row0 + rows, (Q, K)).astype(np.int32)
    bad = r.random((Q, K))
    cand[bad < 0.1] = -1                                                     # the padding of a short filtered list
    cand[(bad >= 0.1) & (bad < 0.15)] = row0 - 1 - r.integers(0, 50, int(((bad >= 0.1) & (bad < 0.15)).sum()))
    cand[(bad >= 0.15) & (bad < 0.2)] = row0 + rows + r.integers(0, 9, int(((bad >= 0.15) & (bad < 0.2)).sum()))
    valid = (cand >= row0) & (cand < row0 + rows)
    n_bad = int((~valid).sum())
    assert n_bad > 0
    fp, kv, tq, tiles, tiles_cls, n = _device_plan(eng, cand, L, row0, rows)
    flat = np.arange(Q * K)
    vflat = flat[valid.reshape(-1)]
    order = np.argsort(cand.reshape(-1)[vflat], kind="stable")
    nv = vflat.size
    assert n[2] == n_bad
    assert np.array_equal(fp[:nv], vflat[order])                             # valid prefix: the host order of the valid entries
    assert np.array_equal(kv[:nv], cand.reshape(-1)[vflat[order]] - row0)
    assert np.array_equal(np.sort(fp[nv:]), flat[~valid.reshape(-1)])        # invalid entries trail, in flat order
    assert np.array_equal(fp[nv:], np.sort(fp[nv:])) and (kv[nv:] == 0).all()
    assert np.array_equal(tq, fp // K)
    rel = np.where(valid, cand - row0, rows).reshape(-1)[fp]                 # invalid entries form one run of their own
    want_t, want_c = S.build_attn_tiles(rel, L), S.build_attn_tiles(rel, 1)
    assert n[:2].tolist() == [want_t.shape[0], want_c.shape[0]]
    assert np.array_equal(tiles[: n[0]], want_t) and np.array_equal(tiles_cls[: n[1]], want_c)


# ---------------------------------------------------------------------------------------------------------------- scores
def _with_limits(eng, max_triplets, fn):
    old = eng.max_triplets
    eng.max_triplets = max_triplets
    try:
        return fn()
    finally:
        eng.max_triplets = old


def _host(m2, tokens, kv, z_t, ids, mask, cand):
    """The host-planned cached path as one chunk, then rerank_sort."""
    eng = m2.engine
    Q, K = cand.shape
    s = _with_limits(eng, Q * K, lambda: m2.score_triplets(z_t, ids, mask, tokens, cand, kv_cache=kv))
    assert eng.last_plan["chunks"] == 1
    return s, eng.rerank_sort(s)


def _assert_rerank_equal(m2, tokens, kv, cand, z_t, ids, mask):
    eng = m2.engine
    s0, o0 = _host(m2, tokens, kv, z_t, ids, mask, cand)
    c = torch.from_numpy(cand).cuda()
    s1, o1, r1 = _with_limits(eng, cand.size, lambda: m2.rerank_topk(z_t, ids, mask, c, kv))
    torch.cuda.synchronize()
    assert torch.isfinite(s0).all()
    assert torch.equal(s0, s1), (s0 - s1).abs().max()
    assert torch.equal(o0, o1)
    assert torch.equal(r1, torch.gather(c, 1, o1.long()))
    return s1, o1


@pytest.mark.parametrize("L", [8, 16, 24, 32, 40])
def test_rerank_equals_host_path_over_lengths(L, bf16):
    _, m2, tokens, kv = bf16
    Q, K = 6, 7
    z_t, ids, mask = _queries(m2.engine, Q, L, seed=L)
    _assert_rerank_equal(m2, tokens, kv, _rand_cand(Q, K, 0, 9, 100 + L), z_t, ids, mask)


@pytest.mark.parametrize("option", ["prune_off", "dedup_off", "fuse_off", "attn_cuda_core", "attn_mma"])
def test_rerank_equals_host_path_with_pipeline_options(option, bf16):
    _, m2, tokens, kv = bf16
    eng = m2.engine
    set_, undo = {"prune_off": (lambda: eng.set_prune_last_layer(False), lambda: eng.set_prune_last_layer(True)),
                  "dedup_off": (lambda: eng.set_dedup_first_layer(False), lambda: eng.set_dedup_first_layer(True)),
                  "fuse_off": (lambda: eng.set_fuse_qkv_attention(False), lambda: eng.set_fuse_qkv_attention(True)),
                  "attn_cuda_core": (lambda: eng.set_attention_impl(1), lambda: eng.set_attention_impl(0)),
                  "attn_mma": (lambda: eng.set_attention_impl(2), lambda: eng.set_attention_impl(0))}[option]
    Q, K = 5, 6
    z_t, ids, mask = _queries(eng, Q, 24, seed=3)
    set_()
    try:
        _assert_rerank_equal(m2, tokens, kv, _rand_cand(Q, K, 0, 12, 7), z_t, ids, mask)
    finally:
        undo()


def test_rerank_equals_host_path_fp32(fp32):
    _, m2, tokens, kv = fp32
    z_t, ids, mask = _queries(m2.engine, 5, 16, seed=4)
    _assert_rerank_equal(m2, tokens, kv, _rand_cand(5, 6, 0, 12, 9), z_t, ids, mask)


def test_rerank_row_range_cache_few_tiles_and_blocks(bf16):
    _, m2, tokens, kv = bf16
    eng = m2.engine
    ranged = m2.kv_cache(tokens, row0=30, rows=20)
    z_t, ids, mask = _queries(eng, 8, 32, seed=11)
    _assert_rerank_equal(m2, tokens, ranged, _rand_cand(8, 9, 30, 50, 12), z_t, ids, mask)
    # 16 x 50 triplets on 3 candidates: 102 tiles and 6 CLS tiles for T = 800 -- most CTAs of the counted kernel have no item
    z_t, ids, mask = _queries(eng, 16, 32, seed=13)
    cand = _rand_cand(16, 50, 40, 43, 14)
    s, o = _assert_rerank_equal(m2, tokens, kv, cand, z_t, ids, mask)
    # several calls of max_triplets // K = 3 queries each: every block is the host path of its own queries
    c = torch.from_numpy(cand).cuda()
    s2, o2, r2 = _with_limits(eng, 150, lambda: m2.rerank_topk(z_t, ids, mask, c, kv))
    for q0 in range(0, 16, 3):
        sl = slice(q0, min(q0 + 3, 16))
        sb, ob = _host(m2, tokens, kv, z_t[sl].contiguous(), ids[sl], mask[sl], cand[sl])
        assert torch.equal(s2[sl], sb) and torch.equal(o2[sl], ob)
    assert torch.equal(r2, torch.gather(c, 1, o2.long()))


def test_invalid_entries_score_neg_fill_and_rank_last(bf16):
    _, m2, tokens, kv = bf16
    eng = m2.engine
    ranged = m2.kv_cache(tokens, row0=20, rows=40)
    Q, K = 6, 10
    z_t, ids, mask = _queries(eng, Q, 16, seed=21)
    cand = _rand_cand(Q, K, 20, 60, 22)
    cand[0, 3] = cand[2, 9] = cand[4, 0] = -1
    cand[1, 5], cand[3, 2] = 19, 60                                          # just outside the cache's rows
    bad = (cand < 20) | (cand >= 60)
    s, o, r = m2.rerank_topk(z_t, ids, mask, torch.from_numpy(cand).cuda(), ranged)
    s, o = s.cpu().numpy(), o.cpu().numpy()
    assert (s[bad] == NEG).all() and (s[~bad] != NEG).all()
    for q in range(Q):
        nb = int(bad[q].sum())
        assert bad[q][o[q][K - nb:]].all()                                   # invalid entries rank last
    # the valid entries score what they score next to valid neighbours: replace the invalid ones by a cached row
    fixed = np.where(bad, 20, cand).astype(np.int32)
    s0, _ = _host(m2, tokens, ranged, z_t, ids, mask, fixed)
    assert np.array_equal(s[~bad], s0.cpu().numpy()[~bad])


def test_launch_count(bf16):
    _, m2, tokens, kv = bf16
    eng = m2.engine
    Q, K = 4, 9
    z_t, ids, mask = _queries(eng, Q, 32, seed=31)
    cand = _rand_cand(Q, K, 0, 20, 32)
    _host(m2, tokens, kv, z_t, ids, mask, cand)
    torch.cuda.synchronize()
    eng.launch_count(reset=True)
    _host(m2, tokens, kv, z_t, ids, mask, cand)
    n_host = eng.launch_count(reset=True)                                    # one cir_stage2_score_cached call + rerank_sort
    m2.rerank_topk(z_t, ids, mask, torch.from_numpy(cand).cuda(), kv)
    n_dev = eng.launch_count(reset=True)
    # the planner replaces the cache-row kernel; the scatter and the ranked-id gather are added
    assert n_dev == n_host + 2, (n_host, n_dev)


# ---------------------------------------------------------------------------------------------------------------- CUDA graphs
def test_rerank_replays_from_a_graph(bf16):
    _, m2, tokens, kv = bf16
    eng = m2.engine
    Q, K, L = 4, 12, 32
    z_t, ids, mask = _queries(eng, Q, L, seed=41)
    cand = torch.from_numpy(_rand_cand(Q, K, 0, 80, 42)).cuda()
    out = (torch.empty(Q, K, device="cuda"), torch.empty(Q, K, dtype=torch.int32, device="cuda"),
           torch.empty(Q, K, dtype=torch.int32, device="cuda"))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        m2.rerank_topk(z_t, ids, mask, cand, kv, out=out)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        m2.rerank_topk(z_t, ids, mask, cand, kv, out=out)
    z2, ids2, mask2 = _queries(eng, Q, L, seed=43)
    cand2 = torch.from_numpy(_rand_cand(Q, K, 0, 80, 44)).cuda()
    cand2[1, 3] = -1
    z_t.copy_(z2), ids.copy_(ids2), mask.copy_(mask2), cand.copy_(cand2)
    graph.replay()
    torch.cuda.synchronize()
    want = m2.rerank_topk(z2, ids2, mask2, cand2, kv)
    for a, b in zip(out, want):
        assert torch.equal(a, b)
    assert out[0][1, 3].item() == NEG


def _online(bf16):
    m1, m2, tokens, kv = bf16
    eng = m1.engine
    g_emb = eng.stage1_gallery_embed(m1._w, tokens)
    tags = np.array([1 << (i % 3) for i in range(tokens.shape[0])], np.uint32)
    index = eng.stage1_index(tokens.shape[0]).add(g_emb, tags=tags)
    return m1, m2, tokens, kv, index, cir.online.OnlineReranker(m1, m2, tokens, index, kv)


def test_online_chain_eager_equals_host_path(bf16):
    m1, m2, tokens, kv, index, chain = _online(bf16)
    eng = m1.engine
    Q, L, k = 5, 24, 20
    ref = torch.tensor([3, 17, 40, 41, 79], dtype=torch.int32).cuda()
    _, ids, mask = _queries(eng, Q, L, seed=51)
    masks = torch.tensor([1, 3, 7, 2, -1], dtype=torch.int32).cuda()
    for tags in (None, masks):
        ranked, scores, dist = chain(ref, ids, mask, k, tags=tags)
        torch.cuda.synchronize()
        z_t, q_emb = eng.stage1_encode(m1._w, tokens, ref, ids, mask)
        d0, i0 = index.topk(q_emb, k, exclude=ref, tags=tags)
        assert torch.equal(dist, d0)
        s0, o0 = _host(m2, tokens, kv, z_t, ids, mask, i0.cpu().numpy())
        assert torch.equal(scores, s0)
        assert torch.equal(ranked, torch.gather(i0, 1, o0.long()))


@pytest.mark.parametrize("tags", [False, True])
def test_online_chain_replays_from_a_graph(tags, bf16):
    m1, m2, tokens, kv, index, chain = _online(bf16)
    Q, L, k = 4, 32, 30
    cap = chain.capture(Q, L, k, tags=tags)
    for seed in (61, 62):
        g = torch.Generator().manual_seed(seed)
        ref = torch.randperm(tokens.shape[0], generator=g)[:Q].int()
        _, ids, mask = _queries(m1.engine, Q, L, seed=seed)
        masks = torch.tensor([1, 2, 4, 5], dtype=torch.int32) if tags else None
        got = [t.clone() for t in cap(ref, ids, mask, tags=masks)]
        want = chain(ref.cuda(), ids, mask, k, tags=None if masks is None else masks.cuda())
        torch.cuda.synchronize()
        for a, b in zip(got, want):
            assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------- golden
def test_config1_golden_from_a_device_topk():
    g = load_golden("config1_8x50.npz")
    sd1, sd2 = golden_weights(g)
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd1, precision="bf16")
    m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision="bf16")
    tokens2 = m2.img_embed(golden_images(g))
    kv = m2.kv_cache(tokens2)
    ids, mask = torch.tensor(g["ids"]).int().cuda(), torch.tensor(g["mask"]).int().cuda()
    z_t, _ = m1.encode_queries(tokens2, torch.tensor(g["ref_idx"]).int(), ids, mask, want_z=True, want_emb=False)
    cand = torch.from_numpy(g["cand_idx"]).cuda()
    s, order, _ = m2.rerank_topk(z_t, ids, mask, cand, kv)
    s0, _ = _host(m2, tokens2, kv, z_t, ids, mask, g["cand_idx"])
    assert torch.equal(s, s0)
    assert np.abs(s.cpu().numpy() - g["scores"]).max() <= 2e-2
    hits = m2.engine.recall_counts(torch.from_numpy(g["k_labels"]), order, (1, 5, 10, 50))
    assert [100.0 * h / int(g["Q"]) for h in hits] == g["recalls"].tolist()


# ---------------------------------------------------------------------------------------------------------------- rejected input
def test_rejected_input_launches_nothing(bf16, fp32):
    _, m2, tokens, kv = bf16
    eng = m2.engine
    _, m32, _, kv32 = fp32
    lib = eng._lib
    ws = torch.empty(1 << 20, dtype=torch.uint8, device=eng.device)
    big = torch.zeros(65, 256, dtype=torch.int32, device=eng.device)
    z_t, ids, mask = _queries(eng, 65, 8, seed=71)
    out = torch.empty(65 * 256, device=eng.device)
    huge = N.Stage2KVCache(row0=0, rows=1 << 18, num_tokens=NTOK, dtype=N.DTYPE_BF16, kv=kv._s.kv)

    def call(cache, Q, K, L, z=z_t, i=ids, m=mask):
        eng._sync_stream()
        N.check(lib.cir_stage2_rerank_cached(eng.ctx, C.byref(m2._w), C.byref(cache), N.ptr(big), Q, K, N.ptr(z), N.ptr(i), N.ptr(m), L,
                                             N.ptr(out), N.ptr(big), None, None, N.ptr(ws), ws.numel()), "rerank")
    z1, ids1, mask1 = _queries(eng, 1, 257, seed=72)
    cases = [
        ("T > 16,384", lambda: call(kv._s, 65, 256, 8)),
        ("K > 2048", lambda: call(kv._s, 1, 4096, 8)),
        ("L > 256", lambda: m2.rerank_topk(z1, ids1, mask1, big[:1, :5], kv)),
        ("dtype", lambda: call(kv32._s, 2, 5, 8)),
        ("no z_t", lambda: call(kv._s, 2, 5, 8, z=None)),
        ("no ids", lambda: call(kv._s, 2, 5, 8, i=None)),
        ("no mask", lambda: call(kv._s, 2, 5, 8, m=None)),
        ("cache too large", lambda: call(huge, 2, 5, 8)),
        ("planner T", lambda: N.check(lib.cir_stage2_plan_topk(eng.ctx, N.ptr(big), 65, 256, 8, 0, 80, *([N.ptr(big)] * 6)))),
        ("planner L", lambda: N.check(lib.cir_stage2_plan_topk(eng.ctx, N.ptr(big), 2, 5, 257, 0, 80, *([N.ptr(big)] * 6)))),
        ("other weights", lambda: eng.stage2_rerank_cached(m32._w, kv, z_t[:2], ids[:2], mask[:2], big[:2, :5])),
    ]
    for what, fn in cases:
        eng.launch_count(reset=True)
        with pytest.raises(N.CirError):
            fn()
        assert eng.launch_count() == 0, what
