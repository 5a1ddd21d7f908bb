"""MXFP8 K/V gallery (CIR_KV_MXFP8: cir_stage2_kv_cache_*_mxfp8, Stage2KVCache(fp8=True)).

The fill must store exactly the torch restatement of the format (test_stage2_kv_fp8_abi) applied to the bf16 K/V a bf16 cache holds;
scoring through it must equal scoring through a bf16 cache whose layers hold the dequantised K/V, bit for bit, on the host-planned
and the device-planned path; and on config 1 it must keep the reference recalls."""
import ctypes as C

import numpy as np
import pytest
import torch

import cir_b200 as cir
from helpers import golden_images, golden_weights, load_golden
from test_stage2_kv_fp8_abi import mxfp8_dequantize, mxfp8_quantize

pytestmark = pytest.mark.gpu
syn = cir.synthetic
S = cir.schedule
N = cir.native
NTOK = 577
NEG = np.float32(cir.engine.NEG_FILL)
ROWS = 24


def _models(precision):
    sd1, sd2 = golden_weights(load_golden("pipeline_small.npz"))
    return (cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd1, precision=precision),
            cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision=precision))


def _dequantised_bf16_cache(m2, fp8, tokens):
    """A bf16 cache of fp8's rows whose layers are overwritten with the torch dequantisation of fp8's bytes."""
    c = cir.engine.Stage2KVCache(m2.engine, m2._w, fp8.rows, NTOK, row0=fp8.row0)
    for i in range(12):
        e, s = fp8.layer(i)
        c.layer(i).copy_(mxfp8_dequantize(e.view(torch.uint8), s))
    torch.cuda.synchronize()
    return c


@pytest.fixture(scope="module")
def env():
    m1, m2 = _models("bf16")
    g = torch.Generator().manual_seed(81)
    tokens = torch.randn(ROWS, NTOK, 768, generator=g).cuda().bfloat16()
    fp8 = m2.kv_cache(tokens, fp8=True)
    return m1, m2, tokens, fp8, _dequantised_bf16_cache(m2, fp8, tokens)


def _queries(eng, Q, L, seed):
    g = torch.Generator().manual_seed(seed)
    ids, mask = syn.make_token_ids(Q, L, seed=seed, min_len=max(1, L // 2))
    ids[:, 0] = syn.ENC_TOKEN_ID
    z_t = torch.randn(Q, L, 768, generator=g).cuda().to(eng.act_dtype)
    return z_t, ids.int().cuda(), mask.int().cuda()


def _rand_cand(Q, K, lo, hi, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(lo, hi, (Q, K), generator=g).int().numpy()


# ---------------------------------------------------------------------------------------------------------------- bytes
def test_fill_equals_the_torch_quantiser(env):
    m1, m2, tokens, fp8, _ = env
    bf = m2.kv_cache(tokens)
    assert fp8.fp8 and fp8.rows == ROWS and fp8.nbytes == -(-12 * ROWS * NTOK * 3168 // 256) * 256
    assert fp8.nbytes * 6144 <= bf.nbytes * 3168 + 6144 * 256                # 3,168 bytes per token row against 6,144
    for i in range(12):
        e, s = fp8.layer(i)
        assert e.dtype == torch.float8_e4m3fn and e.shape == (ROWS * NTOK, 3072) and s.dtype == torch.uint8 and s.shape == (ROWS * NTOK, 96)
        we, ws = mxfp8_quantize(bf.layer(i))
        assert torch.equal(e.view(torch.uint8), we), i
        assert torch.equal(s, ws), i


@pytest.mark.parametrize("slice_rows", [1, 5])
def test_slice_fills_are_byte_identical(slice_rows, env, monkeypatch):
    m1, m2, tokens, fp8, _ = env
    monkeypatch.setattr(cir.engine, "KV_FILL_SLICE_ROWS", slice_rows)
    a = cir.engine.Stage2KVCache(m2.engine, m2._w, ROWS, NTOK, fp8=True)
    a.fill(tokens[7:], 7).fill(tokens[:7], 0)                                  # out of order, uneven slices
    b = cir.engine.Stage2KVCache(m2.engine, m2._w, ROWS, NTOK, fp8=True)
    for r in range(0, ROWS, 3):
        b.fill(tokens[r:r + 3], r)
    torch.cuda.synchronize()
    n = fp8.nbytes
    assert torch.equal(a._blob[:n], fp8._blob[:n]) and torch.equal(b._blob[:n], fp8._blob[:n])


# ---------------------------------------------------------------------------------------------------------------- scores
def _chunk(m2, cache, cand, z_t, ids, mask, prefix=None):
    eng = m2.engine
    ch = S.plan_chunks(cand, None, 1 << 20, 1 << 20)
    assert len(ch) == 1
    ch = ch[0]
    L = ids.shape[1]
    lists = dict(attn_work=S.build_attn_work(ch.trip_slot, L), attn_tiles=S.build_attn_tiles(ch.trip_slot, L),
                 attn_tiles_cls=S.build_attn_tiles(ch.trip_slot, 1))
    ql = torch.from_numpy(ch.query_list.astype(np.int64)).cuda()
    if prefix is None:
        args = (z_t[ql].contiguous(), ids[ql].contiguous(), mask[ql].contiguous(), ch.trip_query, ch.trip_slot)
    else:
        args = (None, ids, mask, ch.query_list[ch.trip_query], ch.trip_slot)
    eng.launch_count(reset=True)
    s, f = eng.stage2_score_chunk(m2._w, None, ch.cand_list, *args, want_feats=True, prefix=prefix, kv_cache=cache, **lists)
    torch.cuda.synchronize()
    return s, f, eng.launch_count(reset=True)


def _assert_chunk_equal(env, cand, z_t, ids, mask, prefix=None, caches=None):
    m2 = env[1]
    fp8, deq = caches or env[3:]
    s0, f0, n0 = _chunk(m2, deq, cand, z_t, ids, mask, prefix)
    s1, f1, n1 = _chunk(m2, fp8, cand, z_t, ids, mask, prefix)
    assert torch.isfinite(s0).all()
    assert torch.equal(s0, s1), (s0 - s1).abs().max()
    assert torch.equal(f0, f1), (f0 - f1).abs().max()
    assert n1 == n0 + 11, (n0, n1)           # 12 dequant kernels instead of the one cache-row kernel


@pytest.mark.parametrize("L", [8, 16, 24, 32, 40])
def test_chunk_equal_over_lengths(L, env):
    Q, K = 6, 7
    z_t, ids, mask = _queries(env[1].engine, Q, L, seed=L)
    _assert_chunk_equal(env, _rand_cand(Q, K, 0, 9, 100 + L), z_t, ids, mask)


@pytest.mark.parametrize("option", ["prune_off", "dedup_off", "fuse_off", "attn_cuda_core", "attn_mma"])
def test_chunk_equal_with_pipeline_options(option, env):
    eng = env[1].engine
    set_, undo = {"prune_off": (lambda: eng.set_prune_last_layer(False), lambda: eng.set_prune_last_layer(True)),
                  "dedup_off": (lambda: eng.set_dedup_first_layer(False), lambda: eng.set_dedup_first_layer(True)),
                  "fuse_off": (lambda: eng.set_fuse_qkv_attention(False), lambda: eng.set_fuse_qkv_attention(True)),
                  "attn_cuda_core": (lambda: eng.set_attention_impl(1), lambda: eng.set_attention_impl(0)),
                  "attn_mma": (lambda: eng.set_attention_impl(2), lambda: eng.set_attention_impl(0))}[option]
    z_t, ids, mask = _queries(eng, 5, 24, seed=3)
    set_()
    try:
        _assert_chunk_equal(env, _rand_cand(5, 6, 0, 12, 7), z_t, ids, mask)
    finally:
        undo()


def test_chunk_equal_prefixed_reuse_1_and_a_row_range(env):
    m1, m2, tokens, fp8, deq = env
    eng = m2.engine
    Q, K, L = 4, 5, 32
    z_t, ids, mask = _queries(eng, Q, L, seed=5)
    prefix = eng.stage2_prefix(m2._w, z_t, ids, mask)
    _assert_chunk_equal(env, _rand_cand(Q, K, 0, 20, 8), z_t, ids, mask, prefix=prefix)
    disjoint = torch.randperm(ROWS, generator=torch.Generator().manual_seed(9))[:Q * K].view(Q, K).int().numpy()   # reuse 1
    _assert_chunk_equal(env, disjoint, z_t, ids, mask)
    _assert_chunk_equal(env, disjoint, z_t, ids, mask, prefix=prefix)
    ranged = m2.kv_cache(tokens, row0=10, rows=12, fp8=True)
    assert ranged.nbytes == -(-12 * 12 * NTOK * 3168 // 256) * 256
    for i in range(12):                                                        # the same bytes as the whole cache's rows
        assert torch.equal(ranged.layer(i)[1], fp8.layer(i)[1][10 * NTOK:22 * NTOK])
    caches = (ranged, _dequantised_bf16_cache(m2, ranged, tokens))
    _assert_chunk_equal(env, _rand_cand(Q, K, 10, 22, 10), z_t, ids, mask, caches=caches)


def test_matrix_equal_over_chunks_with_inactive_rows(env):
    m1, m2, tokens, fp8, deq = env
    eng = m2.engine
    Q, K, L = 12, 8, 32
    z_t, ids, mask = _queries(eng, Q, L, seed=11)
    cand = _rand_cand(Q, K, 0, ROWS, 12)
    active = np.ones(Q, bool)
    active[[2, 7]] = False
    old = eng.max_triplets
    eng.max_triplets = 24
    try:
        a = m2.score_triplets(z_t, ids, mask, tokens, cand, active, kv_cache=deq)
        plan = dict(eng.last_plan)
        b = m2.score_triplets(z_t, ids, mask, tokens, cand, active, kv_cache=fp8)
        assert eng.last_plan == plan and plan["chunks"] > 3                  # the same chunk plan (24 triplets < 64 candidates)
    finally:
        eng.max_triplets = old
    assert torch.equal(a, b), (a - b).abs().max()
    assert (b[torch.from_numpy(~active).cuda()] == cir.engine.NEG_FILL).all()


def test_chunks_bounded_by_max_candidates(env):
    m1, m2, tokens, fp8, deq = env
    eng = m2.engine
    Q, K, L = 6, 10, 16
    z_t, ids, mask = _queries(eng, Q, L, seed=13)
    cand = _rand_cand(Q, K, 0, ROWS, 14)
    old = eng.max_candidates
    eng.max_candidates = 5
    try:
        got = m2.score_triplets(z_t, ids, mask, tokens, cand, kv_cache=fp8)
        assert eng.last_plan["chunks"] >= -(-np.unique(cand).size // 5)
        want = m2.score_triplets(z_t, ids, mask, tokens, cand, kv_cache=deq)
    finally:
        eng.max_candidates = old
    assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------------------------- device-planned
def _host(env, kv, z_t, ids, mask, cand):
    """The host-planned path as one chunk, then rerank_sort."""
    m2, tokens = env[1], env[2]
    eng = m2.engine
    Q, K = cand.shape
    old = eng.max_triplets, eng.max_candidates
    eng.max_triplets, eng.max_candidates = Q * K, 1 << 20
    try:
        s = m2.score_triplets(z_t, ids, mask, tokens, cand, kv_cache=kv)
        assert eng.last_plan["chunks"] == 1
    finally:
        eng.max_triplets, eng.max_candidates = old
    return s, eng.rerank_sort(s)


def _assert_rerank_equal(env, cand, z_t, ids, mask):
    m2, kv = env[1], env[3]
    s0, o0 = _host(env, kv, z_t, ids, mask, cand)
    c = torch.from_numpy(cand).cuda()
    s1, o1, r1 = m2.rerank_topk(z_t, ids, mask, c, kv)
    torch.cuda.synchronize()
    assert torch.isfinite(s0).all()
    assert torch.equal(s0, s1), (s0 - s1).abs().max()
    assert torch.equal(o0, o1)
    assert torch.equal(r1, torch.gather(c, 1, o1.long()))
    return s1, o1


@pytest.mark.parametrize("case", ["duplicates", "q1", "long_run", "few_unique"])
def test_rerank_equals_the_host_planned_call(case, env):
    eng = env[1].engine
    r = np.random.default_rng(3)
    if case == "duplicates":
        cand = r.integers(0, ROWS, (7, 9)).astype(np.int32)
        cand[:, 4] = cand[:, 2]
    elif case == "q1":
        cand = r.integers(0, ROWS, (1, 40)).astype(np.int32)
    elif case == "long_run":
        cand = r.integers(0, ROWS, (40, 20)).astype(np.int32)
        cand[:, :10] = 7                                                       # a run of 400 triplets
    else:
        cand = r.integers(5, 8, (16, 50)).astype(np.int32)                     # 3 unique candidates, T = 800
    Q = cand.shape[0]
    z_t, ids, mask = _queries(eng, Q, 32, seed=20 + Q)
    _assert_rerank_equal(env, cand, z_t, ids, mask)


def test_rerank_invalid_entries_and_launches(env):
    m1, m2, tokens, fp8, deq = env
    eng = m2.engine
    ranged = m2.kv_cache(tokens, row0=4, rows=16, fp8=True)
    Q, K = 6, 10
    z_t, ids, mask = _queries(eng, Q, 16, seed=21)
    cand = _rand_cand(Q, K, 4, 20, 22)
    cand[0, 3] = cand[2, 9] = cand[4, 0] = -1
    cand[1, 5], cand[3, 2] = 3, 20                                           # just outside the cache's rows
    bad = (cand < 4) | (cand >= 20)
    s, o, r = m2.rerank_topk(z_t, ids, mask, torch.from_numpy(cand).cuda(), ranged)
    s, o = s.cpu().numpy(), o.cpu().numpy()
    assert (s[bad] == NEG).all() and (s[~bad] != NEG).all()
    for q in range(Q):
        nb = int(bad[q].sum())
        assert bad[q][o[q][K - nb:]].all()
    fixed = np.where(bad, 4, cand).astype(np.int32)
    s0, _ = _host(env, ranged, z_t, ids, mask, fixed)
    assert np.array_equal(s[~bad], s0.cpu().numpy()[~bad])
    # every entry invalid: nothing to score, nothing faults
    s, o, r = m2.rerank_topk(z_t, ids, mask, torch.full((Q, K), -1, dtype=torch.int32, device="cuda"), ranged)
    assert (s.cpu().numpy() == NEG).all()
    # launches: the bf16 cache's call + the run kernel + 12 dequant kernels
    c = torch.from_numpy(fixed).cuda()
    m2.rerank_topk(z_t, ids, mask, c, deq)
    torch.cuda.synchronize()
    eng.launch_count(reset=True)
    m2.rerank_topk(z_t, ids, mask, c, deq)
    n_bf = eng.launch_count(reset=True)
    m2.rerank_topk(z_t, ids, mask, c, fp8)
    assert eng.launch_count(reset=True) == n_bf + 13


def test_query_blocks_stay_within_the_triplet_budget(env):
    m1, m2, tokens, fp8, deq = env
    eng = m2.engine
    Q, K, L = 45, 50, 8                                                      # 2,250 triplets: two calls of 40 and 5 queries
    z_t, ids, mask = _queries(eng, Q, L, seed=31)
    cand = _rand_cand(Q, K, 0, ROWS, 32)
    assert cir.engine.RERANK_FP8_MAX_TRIPLETS // K == 40
    s, o, r = m2.rerank_topk(z_t, ids, mask, torch.from_numpy(cand).cuda(), fp8)
    for sl in (slice(0, 40), slice(40, 45)):
        s0, o0 = _host(env, fp8, z_t[sl].contiguous(), ids[sl], mask[sl], cand[sl])
        assert torch.equal(s[sl], s0) and torch.equal(o[sl], o0)


def test_workspace_sizes(env):
    m1, m2, tokens, fp8, deq = env
    eng = m2.engine
    lib = eng._lib
    for T, Cn, Q, L in ((8, 3, 2, 32), (300, 64, 6, 16), (2048, 2048, 41, 40)):
        bf = lib.cir_stage2_kv_score_workspace_bytes(eng.ctx, C.byref(deq._s), T, Cn, Q, L)
        assert bf == lib.cir_stage2_score_cached_workspace_bytes(eng.ctx, T, Q, L, NTOK)
        f8 = lib.cir_stage2_kv_score_workspace_bytes(eng.ctx, C.byref(fp8._s), T, Cn, Q, L)
        assert abs((f8 - bf) - (Cn * NTOK * 3072 * 2 - 4 * T)) <= 512       # + dequantised K/V, - the cache-row list
    for Q, K, L in ((1, 50, 32), (40, 50, 8)):
        bf = lib.cir_stage2_kv_rerank_workspace_bytes(eng.ctx, C.byref(deq._s), Q, K, L)
        assert bf == lib.cir_stage2_rerank_cached_workspace_bytes(eng.ctx, Q, K, L, NTOK)
        assert lib.cir_stage2_kv_rerank_workspace_bytes(eng.ctx, C.byref(fp8._s), Q, K, L) > bf + Q * K * NTOK * 3072 * 2


# ---------------------------------------------------------------------------------------------------------------- CUDA graphs
def test_rerank_replays_from_a_graph(env):
    m1, m2, tokens, fp8, deq = env
    eng = m2.engine
    Q, K, L = 4, 12, 32
    z_t, ids, mask = _queries(eng, Q, L, seed=41)
    cand = torch.from_numpy(_rand_cand(Q, K, 0, ROWS, 42)).cuda()
    out = (torch.empty(Q, K, device="cuda"), torch.empty(Q, K, dtype=torch.int32, device="cuda"),
           torch.empty(Q, K, dtype=torch.int32, device="cuda"))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        m2.rerank_topk(z_t, ids, mask, cand, fp8, out=out)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        m2.rerank_topk(z_t, ids, mask, cand, fp8, out=out)
    z2, ids2, mask2 = _queries(eng, Q, L, seed=43)
    cand2 = torch.from_numpy(_rand_cand(Q, K, 0, 3, 44)).cuda()            # far fewer unique candidates than at capture
    cand2[1, 3] = -1
    z_t.copy_(z2), ids.copy_(ids2), mask.copy_(mask2), cand.copy_(cand2)
    graph.replay()
    torch.cuda.synchronize()
    want = m2.rerank_topk(z2, ids2, mask2, cand2, fp8)
    for a, b in zip(out, want):
        assert torch.equal(a, b)
    assert out[0][1, 3].item() == NEG


def test_online_chain_with_an_fp8_cache(env):
    m1, m2, tokens, fp8, deq = env
    eng = m1.engine
    g_emb = eng.stage1_gallery_embed(m1._w, tokens)
    index = eng.stage1_index(ROWS).add(g_emb)
    chain = cir.online.OnlineReranker(m1, m2, tokens, index, fp8)
    Q, L, k = 4, 24, 10
    ref = torch.tensor([3, 17, 5, 20], dtype=torch.int32).cuda()
    _, ids, mask = _queries(eng, Q, L, seed=51)
    ranked, scores, dist = chain(ref, ids, mask, k)
    z_t, q_emb = eng.stage1_encode(m1._w, tokens, ref, ids, mask)
    d0, i0 = index.topk(q_emb, k, exclude=ref)
    s0, o0 = _host(env, fp8, z_t, ids, mask, i0.cpu().numpy())
    assert torch.equal(dist, d0) and torch.equal(scores, s0) and torch.equal(ranked, torch.gather(i0, 1, o0.long()))
    cap = chain.capture(Q, L, k)
    for seed in (61, 62):
        gg = torch.Generator().manual_seed(seed)
        ref = torch.randperm(ROWS, generator=gg)[:Q].int()
        _, ids, mask = _queries(eng, Q, L, seed=seed)
        got = [t.clone() for t in cap(ref, ids, mask)]
        want = chain(ref.cuda(), ids, mask, k)
        torch.cuda.synchronize()
        for a, b in zip(got, want):
            assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------- accuracy
def test_config1_recalls_through_an_fp8_cache():
    g = load_golden("config1_8x50.npz")
    sd1, sd2 = golden_weights(g)
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd1, precision="bf16")
    m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision="bf16")
    tokens2 = m2.img_embed(golden_images(g))
    kv = m2.kv_cache(tokens2, fp8=True)
    ids, mask = torch.tensor(g["ids"]).int().cuda(), torch.tensor(g["mask"]).int().cuda()
    z_t, _ = m1.encode_queries(tokens2, torch.tensor(g["ref_idx"]).int(), ids, mask, want_z=True, want_emb=False)
    s = m2.score_triplets(z_t, ids, mask, tokens2, g["cand_idx"], kv_cache=kv)
    err = np.abs(s.cpu().numpy() - g["scores"])
    assert err.max() <= 2e-2, err.max()
    order = m2.engine.rerank_sort(s)
    hits = m2.engine.recall_counts(torch.from_numpy(g["k_labels"]), order, (1, 5, 10, 50))
    assert [100.0 * h / int(g["Q"]) for h in hits] == g["recalls"].tolist()
    s2, order2, _ = m2.rerank_topk(z_t, ids, mask, torch.from_numpy(g["cand_idx"]).cuda(), kv)
    assert np.abs(s2.cpu().numpy() - g["scores"]).max() <= 2e-2
    hits = m2.engine.recall_counts(torch.from_numpy(g["k_labels"]), order2, (1, 5, 10, 50))
    assert [100.0 * h / int(g["Q"]) for h in hits] == g["recalls"].tolist()


# ---------------------------------------------------------------------------------------------------------------- rejected input
def test_rejected_input_launches_nothing(env):
    m1, m2, tokens, fp8, deq = env
    eng = m2.engine
    lib = eng._lib
    _, m32 = _models("fp32")
    e32 = m32.engine
    Q, K, L = 2, 5, 16
    z_t, ids, mask = _queries(eng, Q, L, seed=71)
    z32, ids32, mask32 = _queries(e32, Q, L, seed=71)
    cand = torch.from_numpy(_rand_cand(Q, K, 0, ROWS, 72)).cuda()
    ch = S.plan_chunks(cand.cpu().numpy(), None, 1 << 20, 1 << 20)[0]
    cl, tq, ts = (torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).cuda() for a in (ch.cand_list, ch.trip_query, ch.trip_slot))
    T, Cn = tq.numel(), cl.numel()
    out = torch.empty(Q * K, device="cuda")
    order = torch.empty(Q * K, dtype=torch.int32, device="cuda")
    blob = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    need_score = lib.cir_stage2_kv_score_workspace_bytes(eng.ctx, C.byref(fp8._s), T, Cn, Q, L)
    need_rerank = lib.cir_stage2_kv_rerank_workspace_bytes(eng.ctx, C.byref(fp8._s), Q, K, L)
    ws = torch.empty(max(need_score, need_rerank), dtype=torch.uint8, device="cuda")

    def score(e, w, cache, z, i, m, nbytes):
        e._sync_stream()
        return lib.cir_stage2_score_cached(e.ctx, C.byref(w), C.byref(cache._s), N.ptr(cl), Cn, N.ptr(z), N.ptr(i), None, None, N.ptr(m),
                                           Q, L, N.ptr(tq), N.ptr(ts), T, None, 0, None, 0, None, 0, N.ptr(out), None, N.ptr(ws), nbytes)

    def rerank(e, w, cache, z, i, m, nbytes):
        e._sync_stream()
        return lib.cir_stage2_rerank_cached(e.ctx, C.byref(w), C.byref(cache._s), N.ptr(cand), Q, K, N.ptr(z), N.ptr(i), N.ptr(m), L,
                                            N.ptr(out), N.ptr(order), None, None, N.ptr(ws), nbytes)

    def fill(fn, cache, *extra):
        eng._sync_stream()
        return fn(eng.ctx, C.byref(m2._w), C.byref(cache._s), N.ptr(tokens), 0, 2, *extra)

    s32 = N.Stage2KVCache()
    one_row = lib.cir_stage2_kv_cache_fill_mxfp8_workspace_bytes(eng.ctx, C.byref(fp8._s), 1)
    cases = [
        ("fp8 cache, fp32 context: score", e32, lambda: score(e32, m32._w, fp8, z32, ids32, mask32, ws.numel()), -1),
        ("fp8 cache, fp32 context: rerank", e32, lambda: rerank(e32, m32._w, fp8, z32, ids32, mask32, ws.numel()), -1),
        ("fp8 init in an fp32 context", e32,
         lambda: lib.cir_stage2_kv_cache_init_mxfp8(e32.ctx, N.ptr(blob), blob.numel(), 0, 1, 8, C.byref(s32)), -1),
        ("short score workspace", eng, lambda: score(eng, m2._w, fp8, z_t, ids, mask, need_score - 256), -3),
        ("bf16-sized score workspace", eng,
         lambda: score(eng, m2._w, fp8, z_t, ids, mask, lib.cir_stage2_score_cached_workspace_bytes(eng.ctx, T, Q, L, NTOK)), -3),
        ("short rerank workspace", eng, lambda: rerank(eng, m2._w, fp8, z_t, ids, mask, need_rerank - 256), -3),
        ("bf16 fill of an fp8 cache", eng, lambda: fill(lib.cir_stage2_kv_cache_fill, fp8), -1),
        ("fp8 fill of a bf16 cache", eng, lambda: fill(lib.cir_stage2_kv_cache_fill_mxfp8, deq, N.ptr(ws), ws.numel()), -1),
        ("fp8 fill, workspace under one row", eng,
         lambda: fill(lib.cir_stage2_kv_cache_fill_mxfp8, fp8, N.ptr(ws), one_row - 256), -3),
    ]
    for what, e, fn, rc in cases:
        e.launch_count(reset=True)
        assert fn() == rc, what
        assert e.launch_count() == 0, what
    with pytest.raises(N.CirError):
        cir.engine.Stage2KVCache(e32, m32._w, 2, NTOK, fp8=True)
