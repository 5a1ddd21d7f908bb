"""Every attention kernel behind cir_attention, and cir_qkv_attention, against the fp64 reference of attn_bound.py
under its rounding-error bound (error / bound <= 1), at the key and query tails of the kernels' tiling, the layouts
the pipelines pass (QKV rows of 2304, K0|V0|K1|V1 rows of 3072, K|V rows of 1536, two streams writing the halves of
1536-wide output rows, CLS rows), masks shared through mask_index, score ranges that move the lazy max, and an fp32
context.  The C-ABI is called directly so strides, mask_index, kv_batches, work and tiles are the test's own.
Outputs land in buffers pre-filled with a NaN sentinel: everything a call must not write is checked bit for bit,
and a second launch on the same inputs must reproduce the output bit for bit.

Kernels (selected by impl and shape; the tcgen05 and small kernels are confirmed through their profile counters):
  tc     fatc::attention_tc_kernel    impl 0, bf16, no mask, tile list
  small  attention_small_kernel       impl 0, bf16, 1 < Lq <= 32, Lk <= 32, no work list
  mma    attention_mma_kernel<8>      impl 2 with a work list;  mma2: <2/4/8> by Lq without one
  simt   attention_simt_kernel<bf16>  impl 1;  simt32: <float> in an fp32 context"""
import ctypes as C

import numpy as np
import pytest
import torch

import cir_b200 as cir
from attn_bound import check_attention, qkv_attention_ref64, ref_attention64

pytestmark = pytest.mark.gpu
N = cir.native
SENT = 0x7FAB                         # a bf16 quiet NaN; fp32 buffers hold it in both halves


@pytest.fixture(scope="module")
def engines():
    """Private contexts: their profile counters tell which kernel ran."""
    return {"bf16": cir.engine.Engine(precision="bf16"), "fp32": cir.engine.Engine(precision="fp32")}


MODES = {"tc": ("bf16", 0), "small": ("bf16", 0), "mma": ("bf16", 2), "mma2": ("bf16", 2), "simt": ("bf16", 1),
         "simt32": ("fp32", 1)}


def _rand(g, *shape, scale=1.0):
    return torch.randn(*shape, generator=g) * scale


def _buffer(n, dtype, fill=None):
    """Device buffer of n elements; fill=None: the sentinel bits."""
    if fill is not None:
        return fill.to(dtype).reshape(-1).cuda()
    b = torch.empty(n, dtype=dtype, device="cuda")
    b.view(torch.int16).fill_(SENT)
    return b


def _bits(t):
    """The raw bits of a bf16 or fp32 tensor, one integer per element."""
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def _view(buf, shape, bs, rs, off):
    return buf.as_strided(shape, (bs, rs, 1), off)


def _launch(e, q, k, v, o, Lk, kv_index=None, key_mask=None, mask_index=None, work=None, tiles=None):
    """cir_attention on strided [B, L, H*64] views; kv_batches = the K/V batches behind k."""
    B, Lq, HD = q.shape
    a = N.AttnArgs()
    a.q, a.k, a.v, a.o = N.ptr(q), N.ptr(k), N.ptr(v), N.ptr(o)
    a.q_bs, a.q_rs, a.k_bs, a.k_rs = q.stride(0), q.stride(1), k.stride(0), k.stride(1)
    a.v_bs, a.v_rs, a.o_bs, a.o_rs = v.stride(0), v.stride(1), o.stride(0), o.stride(1)
    a.kv_index, a.key_mask, a.mask_index = N.ptr(kv_index), N.ptr(key_mask), N.ptr(mask_index)
    a.work, a.num_work = N.ptr(work), (0 if work is None else work.shape[0])
    a.tiles, a.num_tiles, a.kv_batches = N.ptr(tiles), (0 if tiles is None else tiles.shape[0]), k.shape[0]
    a.B, a.H, a.Lq, a.Lk, a.scale = B, HD // 64, Lq, Lk, 0.125
    e._sync_stream()
    N.check(e._lib.cir_attention(e.ctx, C.byref(a)), "cir_attention")


def _counts(e):
    return e.profile_read(N.PROF_ATTN_TC)[2], e.profile_read(N.PROF_ATTN_SELF)[2]


def _i32(a):
    return None if a is None else torch.as_tensor(np.asarray(a), dtype=torch.int32).cuda()


def run_checked(engines, mode, q, k, v, o, obuf, kv_index=None, key_mask=None, mask_index=None, tag=""):
    """One launch in `mode` writing the view o of obuf; asserts the kernel, the bound, finiteness, that nothing
    outside o changed, and a bit-identical second launch.  -> error / bound."""
    prec, impl = MODES[mode]
    e = engines[prec]
    Lq, Lk = q.shape[1], k.shape[1]
    kvi = kv_index.cpu().numpy() if kv_index is not None else np.arange(q.shape[0])
    work = _i32(cir.schedule.build_attn_work(kvi, Lq)) if mode == "mma" else None
    tiles = _i32(cir.schedule.build_attn_tiles(kvi, Lq)) if mode == "tc" else None
    before = obuf.clone()
    written = torch.zeros(obuf.shape, dtype=torch.bool, device="cuda")
    _view(written, o.shape, o.stride(0), o.stride(1), o.storage_offset()).fill_(True)
    e.set_attention_impl(impl)
    e.profile_gemm(True)                                     # restarts the counters
    try:
        _launch(e, q, k, v, o, Lk, kv_index, key_mask, mask_index, work, tiles)
        ran = _counts(e)
        e.profile_gemm(False)
        first = o.clone()
        _launch(e, q, k, v, o, Lk, kv_index, key_mask, mask_index, work, tiles)
    finally:
        e.set_attention_impl(0)
        e.profile_gemm(False)
    torch.cuda.synchronize()
    assert ran == {"tc": (1, 0), "small": (0, 1)}.get(mode, (0, 0)), (mode, ran)
    assert torch.equal(_bits(first), _bits(o.contiguous())), "second launch differs"
    assert torch.isfinite(first).all()
    assert torch.equal(_bits(obuf)[~written], _bits(before)[~written]), "write outside the output"
    ref = ref_attention64(q, k, v, key_mask=key_mask, kv_index=kv_index, mask_index=mask_index)
    ratio, where = check_attention(first, ref, prec)
    print(f"[{mode}] {tag} B={q.shape[0]} Lq={Lq} Lk={Lk}: error/bound {ratio:.3f} at {where}")
    assert ratio <= 1.0, (mode, tag, ratio, where)
    return ratio


def _runs(Lq, runs_extra=2):
    """Sorted kv_index with a run of length 1 at both ends and one run that crosses a 256-row double tile."""
    RB = 256 if Lq > 256 else 1 << max(0, (Lq - 1).bit_length())
    G = max(1, 256 // RB)
    lens = [1, G + 1, runs_extra, 1]
    return np.repeat(np.arange(len(lens)), lens).astype(np.int32)


def _simple(engines, mode, Lq, Lk, H=2, seed=0, kv_extra=2, qfun=None, kfun=None, mask=None,
            mask_index=None, kv=None):
    """Contiguous-row case: q [B, Lq, H*64], k/v with kv_extra unused K/V batches behind the used ones."""
    g = torch.Generator().manual_seed(seed)
    prec = MODES[mode][0]
    dt = torch.bfloat16 if prec == "bf16" else torch.float32
    kvi = _runs(Lq) if kv is None else kv
    B, nkv = kvi.size, int(kvi.max()) + 1 + kv_extra
    HD = H * 64
    qh = _rand(g, B, Lq, HD)
    kh = _rand(g, nkv, Lk, HD)
    if qfun:
        qh = qfun(qh)
    if kfun:
        kh = kfun(kh)
    qb = _buffer(0, dt, qh)
    kb = _buffer(0, dt, kh)
    vb = _buffer(0, dt, _rand(g, nkv, Lk, HD))
    ob = _buffer(B * Lq * HD + 1024, dt)
    q = _view(qb, (B, Lq, HD), Lq * HD, HD, 0)
    k = _view(kb, (nkv, Lk, HD), Lk * HD, HD, 0)
    v = _view(vb, (nkv, Lk, HD), Lk * HD, HD, 0)
    o = _view(ob, (B, Lq, HD), Lq * HD, HD, 0)
    return run_checked(engines, mode, q, k, v, o, ob, kv_index=_i32(kvi), key_mask=_i32(mask), mask_index=_i32(mask_index),
                       tag=f"seed={seed}")


LK_TAILS = [16, 17, 31, 32, 33, 63, 64, 65, 127, 129, 200, 577, 1024]
LQ_TAILS = [1, 2, 15, 16, 17, 31, 32, 33, 255, 256, 257, 577]


@pytest.mark.parametrize("mode", ["tc", "mma", "mma2", "simt", "simt32"])
@pytest.mark.parametrize("Lk", LK_TAILS)
def test_key_and_query_tails(engines, mode, Lk):
    """Every edge of the 64-key chunk and of its 32-column halves, crossed with the query tails of the 16-row mma
    tiles, the 32-row simt tiles and the RB = 1 .. 256 rows of the tcgen05 double tiles."""
    for i, Lq in enumerate(LQ_TAILS):
        if Lq * Lk > 577 * 577 and mode.startswith("simt"):
            continue                                         # one CTA per 32 rows re-reads all keys: keep the sweep short
        _simple(engines, mode, Lq, Lk, seed=Lk * 1000 + i)


@pytest.mark.parametrize("mode", ["small", "mma", "mma2", "simt", "simt32"])
@pytest.mark.parametrize("Lq,Lk", [(32, 32), (16, 16), (2, 8), (24, 24), (17, 31), (1, 32), (40, 100), (32, 577)])
def test_masks_shared_through_mask_index(engines, mode, Lq, Lk):
    """Mask rows of length 1, 2, Lk - 1 and Lk, each shared by several batches in a non-monotone mask_index (as
    trip_query shares a query's caption mask among its triplets)."""
    if mode == "small" and not (1 < Lq <= 32 and Lk <= 32):
        pytest.skip("the small kernel takes 1 < Lq <= 32, Lk <= 32")
    lens = torch.tensor([Lk, 1, 2, max(1, Lk - 1)])
    mask = (torch.arange(Lk)[None, :] < lens[:, None]).int()
    kv = np.array([0, 0, 0, 1, 1, 2, 2, 2, 2], np.int32)
    mask_index = np.array([2, 0, 3, 1, 3, 0, 2, 1, 0], np.int32)
    _simple(engines, mode, Lq, Lk, H=12, seed=Lq * 7 + Lk, mask=mask, mask_index=mask_index, kv=kv)


def _burst(k):
    k[:, 200:260] *= 6.0                                     # moves the lazy max in chunk 3 ...
    k[:, 500:] *= 12.0                                       # ... and again in the last chunks
    return k


def _onehot(k):
    k[:, ::37] *= 12.0                                       # a few keys dominate every row
    return k


def _first_chunk_max(k):
    k[:, 3] *= 4.0                                           # the max is in chunk 0: the reference never moves
    return k


def _burst32(k):
    k[:, 20:] *= 12.0                                        # 32 keys: the burst sits in the only chunk
    return k


SCORES = {"burst": dict(kfun=_burst), "onehot": dict(kfun=_onehot), "first_chunk_max": dict(kfun=_first_chunk_max),
          "all_negative": dict(qfun=lambda q: q.abs(), kfun=lambda k: -k.abs())}


@pytest.mark.parametrize("mode", ["tc", "mma", "simt", "simt32"])
@pytest.mark.parametrize("scores", list(SCORES))
@pytest.mark.parametrize("Lq", [1, 32])
def test_score_ranges(engines, mode, scores, Lq):
    _simple(engines, mode, Lq, 577, H=12, seed=Lq, **SCORES[scores])


@pytest.mark.parametrize("scores", list(SCORES))
def test_score_ranges_small(engines, scores):
    kw = dict(SCORES[scores])
    if scores == "burst":
        kw["kfun"] = _burst32
    mask = torch.ones(1, 32, dtype=torch.int32)
    _simple(engines, "small", 32, 32, H=12, seed=5, mask=mask, mask_index=np.zeros(5, np.int32),
            kv=np.array([0, 0, 1, 2, 2], np.int32), **kw)


# ------------------------------------------------------------------------------------ production layouts

def _cross_layout(engines, mode, L, kv_row, pad_rows, seed, cls=False):
    """Stage-II cross-attention: q of both streams [2][T, L, 768]; K/V rows of kv_row elements (3072 = K0|V0|K1|V1,
    1536 = K|V of one stream, used by both); o rows of 1536 (ctx0 | ctx1) with o_bs = (L + pad_rows) * 1536, both
    streams written by two calls.  kv_index names a few of many cached K/V batches.  cls: Lq = 1 with q_bs = 768
    and o_bs = 1536 (the last layer's CLS rows)."""
    g = torch.Generator().manual_seed(seed)
    D, Nk = 768, 577
    kvi = np.array([1, 1, 1, 4, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6], np.int32)           # runs of 3, 1 and 10 (> 8 per tile)
    T, kv_batches = kvi.size, 9
    Lq = 1 if cls else L
    prec = MODES[mode][0]
    dt = torch.bfloat16 if prec == "bf16" else torch.float32
    qb = _buffer(0, dt, _rand(g, 2, T, Lq, D))
    kvb = _buffer(0, dt, _rand(g, kv_batches, Nk, kv_row))
    rows = Lq + pad_rows
    ob = _buffer(T * rows * 2 * D + 4096, dt)
    ratios = []
    for s in range(2):
        q = _view(qb, (T, Lq, D), Lq * D, D, s * T * Lq * D)
        koff = (s * 2 * D) if kv_row == 4 * D else 0
        k = _view(kvb, (kv_batches, Nk, D), Nk * kv_row, kv_row, koff)
        v = _view(kvb, (kv_batches, Nk, D), Nk * kv_row, kv_row, koff + D)
        o = _view(ob, (T, Lq, D), rows * 2 * D, 2 * D, s * D)
        ratios.append(run_checked(engines, mode, q, k, v, o, ob, kv_index=_i32(kvi), tag=f"cross s={s} kv_row={kv_row} pad={pad_rows}"))
    return max(ratios)


@pytest.mark.parametrize("mode", ["tc", "mma", "mma2", "simt", "simt32"])
@pytest.mark.parametrize("kv_row,pad_rows", [(3072, 0), (3072, 2), (1536, 0)])
def test_cross_attention_layout(engines, mode, kv_row, pad_rows):
    _cross_layout(engines, mode, 32, kv_row, pad_rows, seed=kv_row + pad_rows)


@pytest.mark.parametrize("mode", ["tc", "mma", "mma2", "simt", "simt32"])
def test_cross_attention_cls_rows(engines, mode):
    _cross_layout(engines, mode, 32, 3072, 0, seed=11, cls=True)


def _self_layout(engines, mode, L, cls, seed):
    """Text self-attention on the QKV GEMM output: rows of 2304 (q | k | v), q/k/v batch stride L * 2304, the mask
    of query trip_query[b] for triplet b; o [T, L, 768], or for the CLS rows Lq = 1 with o_bs = 768."""
    g = torch.Generator().manual_seed(seed)
    D = 768
    T = 11
    prec = MODES[mode][0]
    dt = torch.bfloat16 if prec == "bf16" else torch.float32
    qkv = _buffer(0, dt, _rand(g, T, L, 3 * D))
    lens = torch.tensor([L, 1, 2, L - 1, 5])
    mask = (torch.arange(L)[None, :] < lens[:, None]).int()
    trip_query = np.array([0, 0, 1, 1, 1, 4, 2, 3, 3, 0, 4], np.int32)
    Lq = 1 if cls else L
    ob = _buffer(T * Lq * D + 4096, dt)
    q = _view(qkv, (T, Lq, D), L * 3 * D, 3 * D, 0)
    k = _view(qkv, (T, L, D), L * 3 * D, 3 * D, D)
    v = _view(qkv, (T, L, D), L * 3 * D, 3 * D, 2 * D)
    o = _view(ob, (T, Lq, D), Lq * D, D, 0)
    return run_checked(engines, mode, q, k, v, o, ob, key_mask=_i32(mask), mask_index=_i32(trip_query),
                       tag=f"self L={L} cls={cls}")


@pytest.mark.parametrize("mode", ["small", "mma", "mma2", "simt", "simt32"])
@pytest.mark.parametrize("L", [8, 17, 32, 40])
def test_self_attention_layout(engines, mode, L):
    if mode == "small" and L > 32:
        pytest.skip("the small kernel takes Lk <= 32")
    _self_layout(engines, mode, L, False, seed=L)


@pytest.mark.parametrize("mode", ["mma2", "mma", "simt", "simt32"])
@pytest.mark.parametrize("L", [8, 32])
def test_self_attention_cls_rows(engines, mode, L):
    _self_layout(engines, mode, L, True, seed=100 + L)


# ------------------------------------------------------------------------------------ fused QKV + self-attention

def _qkv_inputs(batch, caps, L, seed, min_len=3, share=None):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(batch, caps, L, 768, generator=g).cuda().bfloat16()
    w = (torch.randn(batch, 2304, 768, generator=g) * 0.04).cuda().bfloat16()
    bias = (torch.randn(batch, 2304, generator=g) * 0.2).cuda()
    nq = max(1, caps // 3) if share is None else share
    lens = torch.randint(min_len, L + 1, (nq,), generator=g)
    lens[0] = L
    if min_len == 1:
        lens[1 % nq] = 1
        lens[2 % nq] = 2
    mask = (torch.arange(L)[None, :] < lens[:, None]).int().cuda()
    mask_index = torch.randint(0, nq, (caps,), generator=g).int().cuda()
    return x, w, bias, mask, mask_index


def check_fused(e, x, w, bias, mask, mask_index):
    """cir_qkv_attention against qkv_attention_ref64; the projection flips are read off the tcgen05 GEMM."""
    batch, caps, L, _ = x.shape
    fused = e.qkv_attention(x, w, bias, key_mask=mask, mask_index=mask_index)
    again = e.qkv_attention(x, w, bias, key_mask=mask, mask_index=mask_index)
    proj = e.gemm(x.reshape(batch, caps * L, 768), w, bias)
    torch.cuda.synchronize()
    assert torch.equal(fused, again)
    assert torch.isfinite(fused.float()).all()
    worst = 0.0
    for s, ref in enumerate(qkv_attention_ref64(x, w, bias, mask, mask_index, proj)):
        ratio, where = check_attention(fused[s], ref, "bf16")
        print(f"[qkv] batch={batch} caps={caps} L={L} stream {s}: error/bound {ratio:.3f} at {where}")
        assert ratio <= 1.0, (s, ratio, where)
        worst = max(worst, ratio)
    return worst


@pytest.fixture(scope="module")
def e16():
    return cir.engine.get_engine(precision="bf16")


@pytest.mark.parametrize("L", [8, 16, 24, 32])
@pytest.mark.parametrize("caps,share", [(37, None), (300, 1), (300, 2)])
def test_fused_qkv_short_captions_and_shared_masks(e16, L, caps, share):
    """Caption lengths 1 and 2 (rows where only CLS, or CLS and one token, attend) and many captions sharing one or
    two mask rows; the fused kernel must also match the unfused path bit for bit here."""
    x, w, bias, mask, mask_index = _qkv_inputs(2, caps, L, seed=caps + L, min_len=1, share=share)
    check_fused(e16, x, w, bias, mask, mask_index)
    qkv = e16.gemm(x.reshape(2, caps * L, 768), w, bias)
    km = mask[mask_index.long()]
    want = torch.stack([e16.attention(*(qkv[s].reshape(caps, L, 2304)[..., i * 768:(i + 1) * 768] for i in range(3)), key_mask=km)
                        for s in range(2)])
    assert torch.equal(e16.qkv_attention(x, w, bias, key_mask=mask, mask_index=mask_index), want)
