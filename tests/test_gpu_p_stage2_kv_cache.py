"""Resident stage-II cross-attention K/V gallery (cir_stage2_kv_cache_*, cir_stage2_score_cached, engine.Stage2KVCache).

The cache is filled once with the cross_kv_w GEMM of every layer; scoring through it must return what the per-chunk projection
returns, bit for bit, in bf16 and in the fp32 check mode.  The per-chunk K/V GEMM of a chunk with C >= 3 candidates takes the
cta_group::2 pair tile, as the fill always does; chunks of C <= 2 candidates take a single-CTA tile (see
test_pair_and_single_cta_tiles_give_the_same_kv_bits), so every bit-equality case below uses C >= 3."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import cir_b200 as cir
from helpers import golden_images, golden_weights, load_golden

pytestmark = pytest.mark.gpu
syn = cir.synthetic
S = cir.schedule
NTOK = 577


def _model(precision):
    sd1, sd2 = golden_weights(load_golden("pipeline_small.npz"))
    return cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision=precision)


@pytest.fixture(scope="module")
def bf16():
    m2 = _model("bf16")
    g = torch.Generator().manual_seed(31)
    tokens = torch.randn(80, NTOK, 768, generator=g).cuda().bfloat16()
    return m2, tokens, m2.kv_cache(tokens)


@pytest.fixture(scope="module")
def fp32():
    m2 = _model("fp32")
    g = torch.Generator().manual_seed(32)
    tokens = torch.randn(12, NTOK, 768, generator=g).cuda()
    return m2, tokens, m2.kv_cache(tokens)


def _kv_weight(m2, i):
    """(W act [3072, 768], bias fp32 [3072]) of layer i as views of the packed blob."""
    eng, w = m2.engine, m2._w
    blob = m2._keep[1][0]
    es = 2 if eng.act_dtype == torch.bfloat16 else 4
    off_w, off_b = int(w.cross_kv_w[i]) - blob.data_ptr(), int(w.cross_kv_b[i]) - blob.data_ptr()
    W = blob[off_w:off_w + 3072 * 768 * es].view(eng.act_dtype).view(3072, 768)
    b = blob[off_b:off_b + 3072 * 4].view(torch.float32)
    return W, b


def _queries(eng, Q, L, seed):
    g = torch.Generator().manual_seed(seed)
    ids, mask = syn.make_token_ids(Q, L, seed=seed, min_len=max(1, L // 2))
    ids[:, 0] = syn.ENC_TOKEN_ID
    z_t = torch.randn(Q, L, 768, generator=g).cuda().to(eng.act_dtype)
    return z_t, ids.int().cuda(), mask.int().cuda()


def _chunk_both(m2, tokens, cache, cand, z_t, ids, mask, prefix=None):
    """One chunk (every triplet of cand [Q,K]) through cir_stage2_score and cir_stage2_score_cached -> (uncached, cached, launches)."""
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
    out = []
    for kv in (None, cache):
        eng.launch_count(reset=True)
        s, f = eng.stage2_score_chunk(m2._w, tokens, ch.cand_list, *args, want_feats=True, prefix=prefix, kv_cache=kv, **lists)
        torch.cuda.synchronize()
        out.append((s, f, eng.launch_count(reset=True)))
    return out[0], out[1], ch


def _assert_chunk_equal(m2, tokens, cache, cand, z_t, ids, mask, prefix=None):
    (s0, f0, n0), (s1, f1, n1), ch = _chunk_both(m2, tokens, cache, cand, z_t, ids, mask, prefix)
    assert ch.cand_list.size >= 3
    assert torch.isfinite(s0).all()
    assert torch.equal(s0, s1), (s0 - s1).abs().max()
    assert torch.equal(f0, f1), (f0 - f1).abs().max()
    # the cached call skips the token gather and the 12 K/V GEMMs and adds the one cache-row kernel
    assert n1 == n0 - 12, (n0, n1)


# ---------------------------------------------------------------------------------------------------------------- cache contents
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_cache_equals_the_kv_gemm(precision, bf16, fp32):
    m2, tokens, cache = bf16 if precision == "bf16" else fp32
    eng = m2.engine
    tok = tokens[:12]
    c = m2.kv_cache(tok)
    assert c.rows == 12 and c.row0 == 0 and c.num_tokens == NTOK and c.nbytes == 12 * 12 * NTOK * 3072 * tok.element_size()
    for i in range(12):
        W, b = _kv_weight(m2, i)
        want = eng.gemm(tok.reshape(-1, 768), W, bias=b)
        assert torch.equal(c.layer(i), want), i
        assert torch.equal(cache.layer(i)[: 12 * NTOK], want), i
    # slices of any size, in any order: the same bytes (the 1-row slice would take a single-CTA tile without the forced pair)
    s = cir.engine.Stage2KVCache(eng, m2._w, 12, NTOK)
    s.fill(tok[1:12], 1).fill(tok[0:1], 0)
    t = cir.engine.Stage2KVCache(eng, m2._w, 12, NTOK)
    t.fill(tok[:5]).fill(tok[5:], 5)
    torch.cuda.synchronize()
    assert torch.equal(s._blob[: c.nbytes], c._blob[: c.nbytes]) and torch.equal(t._blob[: c.nbytes], c._blob[: c.nbytes])


def test_pair_and_single_cta_tiles_give_the_same_kv_bits(bf16):
    """The finding DESIGN.md section 5 records: the cta_group::2 pair tile (the fill, chunks of >= 3 candidates) and the single-CTA
    tiles (128 columns: chunks of <= 2 candidates; 256 columns: CIR_GEMM_TCGEN05_1CTA) accumulate every K/V element in the same
    order, so they store the same bits."""
    m2, tokens, cache = bf16
    eng = m2.engine
    W, b = _kv_weight(m2, 5)
    want = cache.layer(5)
    assert torch.equal(eng.gemm(tokens[:2].reshape(-1, 768), W, bias=b), want[: 2 * NTOK])
    eng.set_gemm_impl(cir.native.GEMM_TCGEN05_1CTA)
    try:
        single = eng.gemm(tokens[:8].reshape(-1, 768), W, bias=b)
    finally:
        eng.set_gemm_impl(cir.native.GEMM_AUTO)
    assert torch.equal(single, want[: 8 * NTOK]), (single.float() - want[: 8 * NTOK].float()).abs().max()


# ---------------------------------------------------------------------------------------------------------------- chunk level
@pytest.mark.parametrize("L", [8, 16, 24, 32, 40])
def test_chunk_equal_over_lengths(L, bf16):
    m2, tokens, cache = bf16
    g = torch.Generator().manual_seed(100 + L)
    Q, K = 6, 7
    cand = torch.stack([torch.randint(0, 9, (K,), generator=g) for _ in range(Q)]).int().numpy()       # repeated candidates
    z_t, ids, mask = _queries(m2.engine, Q, L, seed=L)
    _assert_chunk_equal(m2, tokens, cache, cand, z_t, ids, mask)


@pytest.mark.parametrize("option", ["prune_off", "dedup_off", "fuse_off", "attn_cuda_core", "attn_mma"])
def test_chunk_equal_with_pipeline_options(option, bf16):
    m2, tokens, cache = bf16
    eng = m2.engine
    set_, undo = {"prune_off": (lambda: eng.set_prune_last_layer(False), lambda: eng.set_prune_last_layer(True)),
                  "dedup_off": (lambda: eng.set_dedup_first_layer(False), lambda: eng.set_dedup_first_layer(True)),
                  "fuse_off": (lambda: eng.set_fuse_qkv_attention(False), lambda: eng.set_fuse_qkv_attention(True)),
                  "attn_cuda_core": (lambda: eng.set_attention_impl(1), lambda: eng.set_attention_impl(0)),
                  "attn_mma": (lambda: eng.set_attention_impl(2), lambda: eng.set_attention_impl(0))}[option]
    g = torch.Generator().manual_seed(7)
    Q, K = 5, 6
    cand = torch.stack([torch.randint(0, 12, (K,), generator=g) for _ in range(Q)]).int().numpy()
    z_t, ids, mask = _queries(eng, Q, 24, seed=3)
    set_()
    try:
        _assert_chunk_equal(m2, tokens, cache, cand, z_t, ids, mask)
    finally:
        undo()


def test_chunk_equal_prefixed_and_reuse_1(bf16):
    m2, tokens, cache = bf16
    eng = m2.engine
    Q, K, L = 4, 9, 32
    z_t, ids, mask = _queries(eng, Q, L, seed=5)
    prefix = eng.stage2_prefix(m2._w, z_t, ids, mask)
    g = torch.Generator().manual_seed(8)
    cand = torch.stack([torch.randint(10, 30, (K,), generator=g) for _ in range(Q)]).int().numpy()
    _assert_chunk_equal(m2, tokens, cache, cand, z_t, ids, mask, prefix=prefix)
    disjoint = torch.randperm(80, generator=g)[: Q * K].view(Q, K).int().numpy()                      # every candidate once
    _assert_chunk_equal(m2, tokens, cache, disjoint, z_t, ids, mask)
    _assert_chunk_equal(m2, tokens, cache, disjoint, z_t, ids, mask, prefix=prefix)


def test_chunk_equal_fp32(fp32):
    m2, tokens, cache = fp32
    g = torch.Generator().manual_seed(9)
    Q, K = 5, 6
    cand = torch.stack([torch.randint(0, 12, (K,), generator=g) for _ in range(Q)]).int().numpy()
    z_t, ids, mask = _queries(m2.engine, Q, 16, seed=4)
    _assert_chunk_equal(m2, tokens, cache, cand, z_t, ids, mask)


# ---------------------------------------------------------------------------------------------------------------- matrix level
def _with_limits(eng, max_triplets, max_candidates, fn):
    old = (eng.max_triplets, eng.max_candidates)
    eng.max_triplets, eng.max_candidates = max_triplets, max_candidates
    try:
        return fn()
    finally:
        eng.max_triplets, eng.max_candidates = old


def test_matrix_equal_over_chunks_inactive_rows_and_a_row_range(bf16):
    m2, tokens, cache = bf16
    eng = m2.engine
    Q, K, L = 12, 8, 32
    z_t, ids, mask = _queries(eng, Q, L, seed=11)
    g = torch.Generator().manual_seed(12)
    cand = torch.stack([torch.randperm(20, generator=g)[:K] for _ in range(Q)]).int().numpy() + 30       # rows 30..49
    active = np.ones(Q, bool)
    active[[2, 7]] = False
    ranged = m2.kv_cache(tokens, row0=30, rows=20)
    assert ranged.row0 == 30 and ranged.rows == 20
    base = _with_limits(eng, 24, 64, lambda: m2.score_triplets(z_t, ids, mask, tokens, cand, active))
    assert eng.last_plan["chunks"] > 3
    for kv in (cache, ranged):
        got = _with_limits(eng, 24, 64, lambda: m2.score_triplets(z_t, ids, mask, tokens, cand, active, kv_cache=kv))
        assert torch.equal(base, got), (base - got).abs().max()
    assert (got[torch.from_numpy(~active).cuda()] == cir.engine.NEG_FILL).all()


def test_matrix_more_than_64_candidates_in_one_chunk(bf16):
    m2, tokens, cache = bf16
    eng = m2.engine
    Q, K, L = 10, 30, 16
    z_t, ids, mask = _queries(eng, Q, L, seed=13)
    g = torch.Generator().manual_seed(14)
    cand = torch.stack([torch.randperm(80, generator=g)[:K] for _ in range(Q)]).int().numpy()
    assert np.unique(cand).size > 64
    got = m2.score_triplets(z_t, ids, mask, tokens, cand, kv_cache=cache)       # default limits: one chunk without max_candidates
    assert eng.last_plan["chunks"] == 1 and eng.last_plan["candidate_loads"] > 64
    base = _with_limits(eng, eng.max_triplets, 1 << 20, lambda: m2.score_triplets(z_t, ids, mask, tokens, cand))
    assert eng.last_plan["chunks"] == 1
    assert torch.equal(base, got), (base - got).abs().max()


# ---------------------------------------------------------------------------------------------------------------- golden
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_config1_golden_through_the_cache(precision):
    g = load_golden("config1_8x50.npz")
    sd1, sd2 = golden_weights(g)
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd1, precision=precision)
    m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision=precision)
    tokens2 = m2.img_embed(golden_images(g))
    kv = m2.kv_cache(tokens2)
    ids, mask = torch.tensor(g["ids"]), torch.tensor(g["mask"])
    z_t, _ = m1.encode_queries(tokens2, torch.tensor(g["ref_idx"]).int(), ids, mask, want_z=True, want_emb=False)
    s = m2.score_triplets(z_t, ids, mask, tokens2, g["cand_idx"], kv_cache=kv)
    assert torch.equal(s, m2.score_triplets(z_t, ids, mask, tokens2, g["cand_idx"]))
    err = np.abs(s.cpu().numpy() - g["scores"])
    assert err.max() <= (2e-2 if precision == "bf16" else 1e-4), err.max()
    if precision == "bf16":
        G, Q = int(g["G"]), int(g["Q"])
        names = syn.index_names_for(G)
        tb = syn.TokenBatch(input_ids=ids, attention_mask=mask)
        ds = syn.SyntheticRelativeDataset(names, g["ref_idx"], g["target_idx"], ["x"] * Q, g["cand_idx"], kind="cirr",
                                          group_idx=syn.make_group_members(torch.tensor(g["ref_idx"]), torch.tensor(g["target_idx"]),
                                                                           G, seed=11).numpy(), token_batch=tb)
        got = cir.validate_stage2.compute_cirr_val_metrics(ds, m2, m1, tokens2, names, kv_cache=kv)
        assert list(got[3:]) == g["recalls"].tolist(), (got, g["recalls"])


# ---------------------------------------------------------------------------------------------------------------- drivers
def test_drivers_with_the_cache(bf16):
    m2, _, _ = bf16
    sd1, _ = golden_weights(load_golden("pipeline_small.npz"))
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd1, precision="bf16")
    G = 10
    tokens = m2.img_embed(syn.make_images(G, 384, seed=1))
    kv = m2.kv_cache(tokens)
    names = syn.index_names_for(G)
    Q, K = 6, 5
    ref, tgt, ids, mask = syn.make_queries(Q, G, 12, seed=9, min_len=6)
    cand, labels = syn.make_random_topk(Q, G, K, ref, tgt, seed=10, hit_rate=0.8)
    groups = syn.make_group_members(ref, tgt, G, seed=11)
    tb = syn.TokenBatch(input_ids=ids, attention_mask=mask)
    ds = syn.SyntheticRelativeDataset(names, ref, tgt, ["x"] * Q, cand.numpy(), kind="cirr", group_idx=groups.numpy(), token_batch=tb)
    V2 = cir.validate_stage2
    a = V2.compute_fiq_val_metrics(ds, m2, m1, tokens, names, return_order=True)
    b = V2.compute_fiq_val_metrics(ds, m2, m1, tokens, names, return_order=True, kv_cache=kv)
    assert a[:2] == b[:2] and np.array_equal(a[2], b[2])
    assert V2.compute_cirr_val_metrics(ds, m2, m1, tokens, names) == V2.compute_cirr_val_metrics(ds, m2, m1, tokens, names, kv_cache=kv)
    pa = V2.generate_cirr_val_predictions(m2, m1, ds, names, tokens)
    pb = V2.generate_cirr_val_predictions(m2, m1, ds, names, tokens, kv_cache=kv)
    assert torch.equal(pa[0], pb[0]) and torch.equal(pa[1], pb[1])


# ---------------------------------------------------------------------------------------------------------------- multi-GPU
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, ws, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=torch.device("cuda", rank))
    try:
        dev = torch.device("cuda", rank)
        sd2 = syn.make_stage2_state_dict(0, 384, "dense")
        m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision="bf16", device=dev)
        g = torch.Generator().manual_seed(40)
        G, Q, K, L = 16, 7, 6, 16
        tokens = torch.randn(G, NTOK, 768, generator=g).to(dev).bfloat16()
        kv = m2.kv_cache(tokens)                                               # replicated on every rank
        z_t, ids, mask = (t.to(dev) for t in _queries(m2.engine, Q, L, seed=41))
        cand = torch.stack([torch.randperm(G, generator=g)[:K] for _ in range(Q)]).int().numpy()
        sharded = cir.distributed.score_matrix_sharded(m2, tokens, z_t, ids, mask, cand, kv_cache=kv)
        single = m2.engine.stage2_score_matrix(m2._w, tokens, z_t, ids, mask, cand, kv_cache=kv)
        assert torch.equal(sharded, single), (sharded - single).abs().max()
        ret[rank] = "ok"
    except Exception as e:  # pragma: no cover
        ret[rank] = f"{type(e).__name__}: {e}"
        raise
    finally:
        dist.destroy_process_group()


def test_two_gpu_replicated_caches_match_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    assert dict(ret) == {0: "ok", 1: "ok"}


# ---------------------------------------------------------------------------------------------------------------- rejected input
def test_rejected_input_launches_nothing(bf16, fp32):
    m2, tokens, cache = bf16
    eng = m2.engine
    Q, K, L = 3, 4, 16
    z_t, ids, mask = _queries(eng, Q, L, seed=50)
    cand = np.array([[0, 1, 2, 3], [4, 5, 6, 7], [8, 9, 10, 11]], np.int32)
    ranged = m2.kv_cache(tokens, row0=2, rows=10)
    other_w, other_keep = eng.pack_stage2(golden_weights(load_golden("pipeline_small.npz"))[1])     # same values, other blob
    short = tokens[:, :401].contiguous()
    m32, tok32, _ = fp32
    ch = S.plan_chunks(cand, None, 1 << 20, 1 << 20)[0]
    z32, ids32, mask32 = _queries(m32.engine, Q, L, seed=50)
    cases = [
        ("outside the cache range", eng, lambda: m2.score_triplets(z_t, ids, mask, tokens, cand, kv_cache=ranged)),
        ("other weights", eng, lambda: eng.stage2_score_matrix(other_w, tokens, z_t, ids, mask, cand, kv_cache=cache)),
        ("token count", eng, lambda: m2.score_triplets(z_t, ids, mask, short, cand, kv_cache=cache)),
        ("dtype", m32.engine, lambda: m32.engine.stage2_score_chunk(m32._w, None, ch.cand_list, z32[ch.query_list.astype(np.int64)],
                                                                    ids32, mask32, ch.trip_query, ch.trip_slot, kv_cache=cache)),
        ("blob too small", eng, lambda: cir.engine.Stage2KVCache(eng, m2._w, 4, NTOK, blob=torch.empty(4096, dtype=torch.uint8,
                                                                                                        device=eng.device))),
        ("fill past rows", eng, lambda: ranged.fill(tokens[10:13], 10)),
    ]
    for what, e, fn in cases:
        e.launch_count(reset=True)
        with pytest.raises(cir.native.CirError):
            fn()
        assert e.launch_count() == 0, what
    del other_keep
