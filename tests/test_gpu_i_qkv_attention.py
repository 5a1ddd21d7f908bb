"""cir_qkv_attention: the fused QKV projection + masked text self-attention kernel (tcgen05 pair tile of one head's
Q|K|V, attention finished in the epilogue) against (1) the unfused path -- tcgen05 GEMM into HBM + attention kernel -- which it
must reproduce BIT FOR BIT (same bf16 rounding point, same operation order), (2) an fp64 restatement of
BertSelfAttention.forward (src/nlvr_encoder.py:140-222) under the rounding-error bound of attn_bound.py, and (3) end to
end: stage-I / stage-II results with the fusion on and off are identical."""
import numpy as np
import pytest
import torch

import cir_b200 as cir
from attn_bound import check_attention, qkv_attention_ref64
from helpers import golden_weights, load_golden

pytestmark = pytest.mark.gpu
syn = cir.synthetic


@pytest.fixture(scope="module")
def e16():
    return cir.engine.get_engine(precision="bf16")


def _inputs(batch, caps, L, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(batch, caps, L, 768, generator=g).cuda().bfloat16()
    w = (torch.randn(batch, 2304, 768, generator=g) * 0.04).cuda().bfloat16()
    bias = (torch.randn(batch, 2304, generator=g) * 0.2).cuda()
    nq = max(1, caps // 3)
    lens = torch.randint(3, L + 1, (nq,), generator=g)
    lens[0] = L
    mask = (torch.arange(L)[None, :] < lens[:, None]).int().cuda()
    mask_index = torch.randint(0, nq, (caps,), generator=g).int().cuda()
    return x, w, bias, mask, mask_index


def _unfused(e, x, w, bias, mask, mask_index):
    batch, caps, L, _ = x.shape
    qkv = e.gemm(x.reshape(batch, caps * L, 768), w, bias)                    # [batch, caps*L, 2304] bf16 in HBM
    km = mask[mask_index.long()]
    out = []
    for s in range(batch):
        t = qkv[s].reshape(caps, L, 2304)
        out.append(e.attention(t[..., :768], t[..., 768:1536], t[..., 1536:], key_mask=km))
    return torch.stack(out)


@pytest.mark.parametrize("batch,caps,L", [(2, 8, 32), (2, 37, 32), (1, 5, 32), (2, 16, 16), (1, 43, 16), (2, 1200, 32), (2, 4096, 32),
                                          (2, 10, 24), (1, 23, 24), (2, 700, 24), (2, 16, 8), (1, 45, 8), (2, 900, 8)])
def test_fused_equals_unfused_bit_for_bit(e16, batch, caps, L):
    x, w, bias, mask, mask_index = _inputs(batch, caps, L, seed=caps + L)
    fused = e16.qkv_attention(x, w, bias, key_mask=mask, mask_index=mask_index)
    torch.cuda.synchronize()
    assert torch.isfinite(fused.float()).all()
    want = _unfused(e16, x, w, bias, mask, mask_index)
    assert torch.equal(fused, want), (fused.float() - want.float()).abs().max().item()
    proj = e16.gemm(x.reshape(batch, caps * L, 768), w, bias)                  # the kernel's bf16 projection: 1-ulp flips vs fp64
    for s, ref in enumerate(qkv_attention_ref64(x, w, bias, mask, mask_index, proj)):
        ratio, where = check_attention(fused[s], ref, "bf16")
        assert ratio <= 1.0, (s, ratio, where)


def test_fused_without_mask_and_bias(e16):
    x, w, _, _, _ = _inputs(2, 24, 32, seed=5)
    fused = e16.qkv_attention(x, w)
    qkv = e16.gemm(x.reshape(2, 24 * 32, 768), w)
    want = torch.stack([e16.attention(*(qkv[s].reshape(24, 32, 2304)[..., i * 768:(i + 1) * 768] for i in range(3))) for s in range(2)])
    assert torch.equal(fused, want)


def test_unsupported_length_is_refused(e16):
    x, w, bias, mask, mask_index = _inputs(1, 4, 40, seed=1)
    with pytest.raises(cir.native.CirError):
        e16.qkv_attention(x, w, bias, key_mask=mask, mask_index=mask_index)


@pytest.mark.parametrize("L", [8, 16, 24, 32])
def test_pipelines_identical_with_and_without_the_fusion(L):
    """Stage I (z_t, q_emb) and stage II (scores over several chunks incl. the per-query prefix) with cir_set_fuse_qkv_attention
    on (default) and off: identical bits."""
    sd1, sd2 = golden_weights(load_golden("pipeline_small.npz"))
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd1, precision="bf16")
    m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision="bf16")
    eng = m2.engine
    g = torch.Generator().manual_seed(3)
    G, Q, K = 7, 21, 6
    tokens = torch.randn(G, 577, 768, generator=g).cuda().bfloat16()
    ids, mask = syn.make_token_ids(Q, L, seed=7, min_len=min(5, L))
    ids[:, 0] = syn.ENC_TOKEN_ID
    ref = torch.randint(0, G, (Q,), generator=g).int()
    cand = torch.stack([torch.randperm(G, generator=g)[:K] for _ in range(Q)]).int().numpy()
    old = eng.max_triplets

    def run():
        z, qe = m1.encode_queries(tokens, ref, ids, mask, want_z=True, want_emb=True)
        eng.max_triplets = 40                                                # several chunks -> the query-prefix path
        try:
            s = m2.score_triplets(z, ids, mask, tokens, cand)
        finally:
            eng.max_triplets = old
        return z, qe, s
    z_on, qe_on, s_on = run()
    for e in {m1.engine, m2.engine}:
        e.set_fuse_qkv_attention(False)
    try:
        z_off, qe_off, s_off = run()
    finally:
        for e in {m1.engine, m2.engine}:
            e.set_fuse_qkv_attention(True)
    assert torch.isfinite(s_on).all()
    assert torch.equal(z_on, z_off) and torch.equal(qe_on, qe_off)
    assert torch.equal(s_on, s_off), (s_on - s_off).abs().max().item()
