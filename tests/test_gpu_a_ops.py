"""GPU parity of the primitive ops through the C-ABI (fp32 check mode + CUDA-core bf16 GEMM).
Runs before the tcgen05 tests so that a tensor-core failure cannot mask these."""
import numpy as np
import pytest
import torch

import cir_b200 as cir
from attn_bound import check_attention, ref_attention64
from oracle import cir_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def e32():
    return cir.engine.get_engine(precision="fp32")


@pytest.fixture(scope="module")
def e16():
    return cir.engine.get_engine(precision="bf16")


def _rand(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).cuda()


@pytest.mark.parametrize("M,N,K,batch", [(70, 100, 96, 1), (256, 768, 768, 2), (33, 2304, 768, 1)])
def test_gemm_fp32_simt(e32, M, N, K, batch):
    N_ = cir.native
    A, W = _rand(batch, M, K, seed=1), _rand(batch, N, K, seed=2, scale=0.05)
    bias, res = _rand(batch, N, seed=3), _rand(batch, M, N, seed=4)
    ref = torch.einsum("bmk,bnk->bmn", A.double(), W.double()) + bias.double()[:, None, :]
    out = e32.gemm(A, W, bias)
    assert (out.double() - ref).abs().max() < 1e-4
    out = e32.gemm(A, W, bias, residual=res, act=N_.ACT_GELU)
    ref2 = torch.nn.functional.gelu(ref) + res.double()
    assert (out.double() - ref2).abs().max() < 1e-4
    out = e32.gemm(A, W, bias, act=N_.ACT_RELU)
    assert (out.double() - ref.clamp_min(0)).abs().max() < 1e-4


def test_gemm_bf16_simt_matches_torch(e16):
    N_ = cir.native
    e16.set_gemm_impl(N_.GEMM_SIMT)
    try:
        A, W = _rand(2, 100, 128, seed=1).bfloat16(), _rand(2, 72, 128, seed=2, scale=0.05).bfloat16()
        bias = _rand(2, 72, seed=3)
        ref = torch.einsum("bmk,bnk->bmn", A.double(), W.double()) + bias.double()[:, None, :]
        out = e16.gemm(A, W, bias, out_f32=True)
        assert (out.double() - ref).abs().max() < 1e-4
        out = e16.gemm(A, W, bias)
        assert out.dtype == torch.bfloat16 and (out.double() - ref).abs().max() < 2e-2
    finally:
        e16.set_gemm_impl(N_.GEMM_AUTO)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_add_layernorm_twin(prec):
    e = cir.engine.get_engine(precision=prec)
    M = 70
    m = _rand(M, 768, seed=1)
    a = _rand(2 * M, 768, seed=2).to(e.act_dtype)
    gamma, beta = 1 + 0.1 * _rand(2, 768, seed=3), 0.1 * _rand(2, 768, seed=4)
    y = e.add_layernorm(m, gamma, beta, res=a, x_rows=M, rows_per_group=M, eps=1e-12)
    x = m.repeat(2, 1) + a.float()
    ref = torch.cat([torch.nn.functional.layer_norm(x[:M], (768,), gamma[0], beta[0], 1e-12),
                     torch.nn.functional.layer_norm(x[M:], (768,), gamma[1], beta[1], 1e-12)])
    tol = 1e-5 if prec == "fp32" else 3e-2
    assert y.dtype == e.act_dtype and (y.float() - ref).abs().max() < tol


@pytest.mark.parametrize("prec,B,Lq,Lk,masked", [("fp32", 3, 12, 12, True), ("fp32", 2, 12, 577, False),
                                                   ("fp32", 1, 577, 577, False), ("bf16", 3, 32, 577, False),
                                                   ("bf16", 2, 32, 32, True)])
def test_attention_simt(prec, B, Lq, Lk, masked):
    e = cir.engine.get_engine(precision=prec)
    q = _rand(B, Lq, 768, seed=1).to(e.act_dtype)
    nkv = 2
    k = _rand(nkv, Lk, 768, seed=2).to(e.act_dtype)
    v = _rand(nkv, Lk, 768, seed=3).to(e.act_dtype)
    kv_index = torch.tensor([i % nkv for i in range(B)], dtype=torch.int32).cuda()
    mask = None
    if masked:
        mask = torch.ones(B, Lk, dtype=torch.int32)
        for b in range(B):
            mask[b, Lk - 1 - b:] = 0
        mask = mask.cuda()
    o = e.attention(q, k, v, key_mask=mask, kv_index=kv_index)
    ref = ref_attention64(q, k, v, mask, kv_index)
    ratio, where = check_attention(o, ref, prec)
    assert ratio <= 1.0, (ratio, where)
    if prec == "fp32":
        assert (o.double() - ref.o).abs().max() < 2e-5


def test_rerank_sort_bit_exact_with_ties(e32):
    g = torch.Generator().manual_seed(0)
    for K in (1, 5, 50, 100, 200, 777):
        s = torch.randn(64, K, generator=g)
        s[:, ::3] = s[:, :1].clone()         # plant ties
        s[0, :] = 0.0
        s[1, : K // 2] = -0.0
        order = e32.rerank_sort(s.cuda()).cpu()
        want = O.rerank_order(s)
        assert torch.equal(order.long(), want)


def test_topk_from_dist_bit_exact(e32):
    g = torch.Generator().manual_seed(1)
    for (Q, G, K) in ((7, 50, 50), (33, 2297, 100), (5, 5000, 200), (3, 3, 2)):
        q = torch.nn.functional.normalize(torch.randn(Q, 256, generator=g), dim=-1)
        gal = torch.nn.functional.normalize(torch.randn(G, 256, generator=g), dim=-1)
        gal[G // 2] = gal[0]                 # exact duplicate -> tie broken by index
        dist = 1 - q @ gal.T
        excl = torch.randint(0, G, (Q,), generator=g)
        K_eff = min(K, G - 1)
        td, ti = e32.topk_from_dist(dist.cuda(), K_eff, exclude=excl)
        wd, wi = O.stage1_topk(q, gal, excl, K_eff)
        # oracle recomputes dist with the same CPU matmul -> identical matrix
        assert torch.equal(ti.cpu().long(), wi)
        assert torch.equal(td.cpu(), wd)
        td2, ti2 = e32.topk_from_dist(dist.cuda(), K_eff, exclude=None)
        wd2, wi2 = O.stage1_topk(q, gal, None, K_eff)
        assert torch.equal(ti2.cpu().long(), wi2)


def test_stage1_topk_fused_and_sharded_merge(e32):
    g = torch.Generator().manual_seed(2)
    Q, G, K = 19, 20000, 100
    q = torch.nn.functional.normalize(torch.randn(Q, 256, generator=g), dim=-1)
    gal = torch.nn.functional.normalize(torch.randn(G, 256, generator=g), dim=-1)
    excl = torch.randint(0, G, (Q,), generator=g)
    td, ti = e32.stage1_topk(q, gal, K, exclude=excl)
    wd, wi = O.stage1_topk(q, gal, excl, K)
    # GPU fp32 dot products may differ from the CPU's in the last bit: compare sets/values with tolerance,
    # and exactness against the GPU's own distance matrix below
    assert (td.cpu() - wd).abs().max() < 1e-6
    assert (ti.cpu().long() == wi).float().mean() > 0.99
    for r in range(Q):
        assert int(excl[r]) not in ti[r].tolist()
    # sharded: 3 uneven gallery shards + merge == unsharded, bit for bit
    parts_d, parts_i = [], []
    bounds = [0, 7000, 7001, G]
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        d, i = e32.stage1_topk(q, gal[lo:hi], K, exclude=excl, col_offset=lo)
        parts_d.append(d); parts_i.append(i)
    md, mi = e32.topk_merge(torch.stack(parts_d), torch.stack(parts_i))
    assert torch.equal(mi, ti) and torch.equal(md, td)


def test_recall_counts(e32):
    g = torch.Generator().manual_seed(3)
    Q, K = 101, 50
    scores = torch.randn(Q, K, generator=g)
    labels = torch.zeros(Q, K, dtype=torch.bool)
    for r in range(Q):
        if r % 7:
            labels[r, int(torch.randint(0, K, (1,), generator=g))] = True
    order = e32.rerank_sort(scores.cuda())
    hits = e32.recall_counts(labels, order, (1, 5, 10, 50))
    lab = O.sorted_labels(scores, labels.numpy())
    want = [int(lab[:, :k].sum()) for k in (1, 5, 10, 50)]
    assert hits == want


def test_embeddings_and_normalize(e32):
    import ctypes as C
    N_ = cir.native
    g = torch.Generator().manual_seed(4)
    word, pos = torch.randn(500, 768, generator=g).cuda(), torch.randn(512, 768, generator=g).cuda()
    gamma, beta = (1 + 0.1 * torch.randn(768, generator=g)).cuda(), (0.1 * torch.randn(768, generator=g)).cuda()
    ids = torch.randint(0, 500, (5, 9), generator=g).int().cuda()
    out = torch.empty(5, 9, 768, device="cuda")
    e32._sync_stream()
    N_.check(e32._lib.cir_bert_embeddings(e32.ctx, N_.ptr(ids), 5, 9, N_.ptr(word), N_.ptr(pos), N_.ptr(gamma), N_.ptr(beta), N_.ptr(out)))
    ref = torch.nn.functional.layer_norm(word[ids.long()] + pos[:9][None], (768,), gamma, beta, 1e-12)
    assert (out - ref).abs().max() < 1e-5
    x = torch.randn(11, 256, generator=g).cuda()
    y = torch.empty_like(x)
    N_.check(e32._lib.cir_l2_normalize(e32.ctx, N_.ptr(x), N_.ptr(y), 11, 256))
    assert (y - torch.nn.functional.normalize(x, dim=-1)).abs().max() < 1e-6


@pytest.mark.parametrize("B,Lq,Lk,masked", [(5, 32, 577, False), (7, 12, 577, False), (3, 40, 577, False), (6, 32, 32, True),
                                            (4, 12, 12, True), (2, 577, 577, False), (9, 32, 100, True)])
def test_attention_mma_vs_reference(e16, B, Lq, Lk, masked):
    q = _rand(B, Lq, 768, seed=1).bfloat16()
    nkv = 3
    k = _rand(nkv, Lk, 768, seed=2).bfloat16()
    v = _rand(nkv, Lk, 768, seed=3).bfloat16()
    kv_index = torch.tensor(sorted(i % nkv for i in range(B)), dtype=torch.int32).cuda()
    mask = None
    if masked:
        mask = torch.ones(B, Lk, dtype=torch.int32)
        for b in range(B):
            mask[b, Lk - 1 - (b % 5):] = 0
        mask = mask.cuda()
    ref = ref_attention64(q, k, v, mask, kv_index)
    o = e16.attention(q, k, v, key_mask=mask, kv_index=kv_index)              # tensor cores, one run per batch
    assert check_attention(o, ref, "bf16")[0] <= 1.0
    work = cir.schedule.build_attn_work(kv_index.cpu().numpy(), Lq)            # K/V shared inside candidate runs
    o2 = e16.attention(q, k, v, key_mask=mask, kv_index=kv_index, work=work)
    assert check_attention(o2, ref, "bf16")[0] <= 1.0
    e16.set_attention_impl(1)
    try:
        o3 = e16.attention(q, k, v, key_mask=mask, kv_index=kv_index)          # CUDA-core kernel on the same inputs
    finally:
        e16.set_attention_impl(0)
    assert (o.float() - o3.float()).abs().max() < 2.5e-2


@pytest.mark.parametrize("B,Lq,Lk", [(9, 32, 577), (5, 12, 577), (6, 40, 577), (3, 577, 577), (7, 32, 128), (4, 32, 200), (2, 130, 65)])
def test_attention_tcgen05_vs_reference(e16, B, Lq, Lk):
    q = _rand(B, Lq, 768, seed=1).bfloat16()
    nkv = 3
    k = _rand(nkv, Lk, 768, seed=2).bfloat16()
    v = _rand(nkv, Lk, 768, seed=3).bfloat16()
    kv_index = torch.tensor(sorted(i % nkv for i in range(B)), dtype=torch.int32).cuda()
    ref = ref_attention64(q, k, v, None, kv_index)
    tiles = cir.schedule.build_attn_tiles(kv_index.cpu().numpy(), Lq)
    o = e16.attention(q, k, v, kv_index=kv_index, tiles=tiles)                 # tcgen05 kernel
    ratio, where = check_attention(o, ref, "bf16")
    assert ratio <= 1.0, (ratio, where)
    e16.set_attention_impl(2)
    try:
        o2 = e16.attention(q, k, v, kv_index=kv_index, work=cir.schedule.build_attn_work(kv_index.cpu().numpy(), Lq))
    finally:
        e16.set_attention_impl(0)
    assert (o.float() - o2.float()).abs().max() < 2.5e-2


def test_attention_tcgen05_lazy_rescale_path(e16):
    """Keys whose scores dwarf everything seen before force the reference max to move (the O accumulator is rescaled
    in TMEM through tcgen05.ld / tcgen05.st); the first chunks then contribute ~0, exactly as in an exact softmax."""
    B, Lq, Lk = 8, 32, 577
    q = _rand(B, Lq, 768, seed=1).bfloat16()
    k = _rand(2, Lk, 768, seed=2)
    k[:, 200:260] *= 6.0                                       # a burst in chunk 3
    k[:, 500:] *= 12.0                                         # and a bigger one in the last chunks
    k = k.bfloat16()
    v = _rand(2, Lk, 768, seed=3).bfloat16()
    kv_index = torch.tensor([0, 0, 0, 0, 1, 1, 1, 1], dtype=torch.int32).cuda()
    ref = ref_attention64(q, k, v, None, kv_index)
    o = e16.attention(q, k, v, kv_index=kv_index, tiles=cir.schedule.build_attn_tiles(kv_index.cpu().numpy(), Lq))
    assert torch.isfinite(o).all()
    ratio, where = check_attention(o, ref, "bf16")             # outputs are near one-hot mixtures of |v| ~ 3 rows
    assert ratio <= 1.0, (ratio, where)
    e16.set_attention_impl(2)
    try:
        o2 = e16.attention(q, k, v, kv_index=kv_index, work=cir.schedule.build_attn_work(kv_index.cpu().numpy(), Lq))
    finally:
        e16.set_attention_impl(0)
    assert (o.float() - o2.float()).abs().max() < 4e-2


@pytest.mark.parametrize("B,Lq,Lk,nkv", [
    (700, 32, 577, 9),      # ~90 double tiles x 12 heads: every persistent CTA walks several items, runs end in half-empty tiles
    (1500, 1, 577, 5),      # CLS rows only (RB = 1, 256 triplets per double tile)
    (640, 32, 64, 7),       # one K/V chunk per item: the Q prefetch trails the ring (drain path of the loader)
    (300, 24, 100, 4),      # two chunks per item, ragged rows per triplet (RB = 32 > Lq)
    (40, 200, 130, 3),      # RB = 256: one triplet per double tile
    (33, 300, 16, 2),       # row slices of a long query (L > 256), minimum key count
])
def test_attention_tcgen05_persistent_items(e16, B, Lq, Lk, nkv):
    """The persistent double-tile kernel with more work items than CTAs, against the fp64 reference."""
    q = _rand(B, Lq, 768, seed=4).bfloat16()
    k = _rand(nkv, Lk, 768, seed=5).bfloat16()
    v = _rand(nkv, Lk, 768, seed=6).bfloat16()
    kv_index = torch.tensor(sorted(i % nkv for i in range(B)), dtype=torch.int32).cuda()
    tiles = cir.schedule.build_attn_tiles(kv_index.cpu().numpy(), Lq)
    o = e16.attention(q, k, v, kv_index=kv_index, tiles=tiles)
    ref = ref_attention64(q, k, v, None, kv_index)
    ratio, where = check_attention(o, ref, "bf16")
    assert ratio <= 1.0, (ratio, where)
    o_again = e16.attention(q, k, v, kv_index=kv_index, tiles=tiles)           # deterministic: no atomics, fixed schedule
    assert torch.equal(o, o_again)
