"""The attention error bound of tests/attn_bound.py, checked on the CPU against a simulated kernel.

``simulate`` restates the bf16 tensor-core attention the way the kernels compute it: 64-key chunks, a lazy
reference max that moves only when the row max grew by more than 2^8 (in the log2 domain), P = exp2(.) rounded to
bf16 for the PV product, fp32 row sums and accumulators, output rounded to bf16.  The bound must accept it
(ratio <= 1 on every shape) without being loose (the largest ratio over the shapes >= 0.5), and reject each of the
mutants below by more than a factor 2 (ratio > 2), each a plausible slip in a kernel edit:

  1 tail chunk's padded keys counted in the row sum      6 one run reads the neighbouring kv_index batch
  2 last key dropped                                      7 last valid query row written with its neighbour's values
  3 a one-key tail chunk skipped                          8 a lazy-max move rescales O but not l
  4 one masked key left unmasked                          9 P rounded to 7 instead of 8 significant bits
  5 mask_index ignored for one batch

On random inputs the simulated kernel sits at 0.35-0.5.  Rows dominated by one or two keys come closer to 1 (0.7
with a two-key mask, 0.8 where the lazy max sits below a dominant key so that its P = 2^j > 1 is rounded): those
are the rows where the worst case of the derivation is reached, so a bound that kept them below 0.7 would fail a
correct kernel elsewhere.

Mutant 9 is a factor-2 precision loss; no bound that accepts every correct kernel can put it above 2 (see the
attn_bound docstring), so it is checked at > 1 on an input whose P is exact in bf16 but not in 7 bits."""
import math

import pytest
import torch

from attn_bound import check_attention, ref_attention64

LOG2E = 1.4426950408889634


def _round7(x):
    m, e = torch.frexp(x)
    return torch.ldexp(torch.round(m * 128.0) / 128.0, e)


def simulate(q, k, v, key_mask=None, kv_index=None, mask_index=None, scale=0.125, mutant=0):
    """A correct bf16 flash-attention kernel (mutant 0) or one of the mutants above, in fp32 torch on the CPU."""
    B, Lq, HD = q.shape
    Bk, Lk = k.shape[0], k.shape[1]
    H = HD // 64
    kvi = torch.arange(B) if kv_index is None else kv_index.long().clone()
    mi = torch.arange(B) if mask_index is None else mask_index.long().clone()
    if mutant == 6:
        kvi[kvi == kvi[0]] = (kvi[0] + 1) % Bk
    if mutant == 5:
        b = int(torch.nonzero(mi != torch.arange(B))[0])
        mi[b] = b
    qh = q.float().reshape(B, Lq, H, 64).transpose(1, 2)
    kh = k.float()[kvi].reshape(B, Lk, H, 64).transpose(1, 2)
    vh = v.float()[kvi].reshape(B, Lk, H, 64).transpose(1, 2)
    sl2 = scale * LOG2E
    x = (qh @ kh.transpose(-1, -2)) * sl2
    if key_mask is not None:
        km = key_mask[mi].clone()
        if mutant == 4:
            row = km[0]
            row[int(torch.nonzero(row == 0)[0])] = 1
        x = x + torch.where(km == 0, MASK_L2, 0.0)[:, None, None, :]
    keys = Lk - 1 if mutant == 2 else Lk
    nch = (keys + 63) // 64
    if mutant == 3:
        assert keys % 64 == 1
        nch -= 1
    o = torch.zeros(B, H, Lq, 64)
    l = torch.zeros(B, H, Lq, 1)
    m = None
    for c in range(nch):
        xs = x[..., c * 64:min(keys, (c + 1) * 64)]
        vs = vh[:, :, c * 64:min(keys, (c + 1) * 64)]
        cmax = xs.amax(-1, keepdim=True)
        if m is None:
            m = cmax
        else:
            m_new = torch.where(cmax > m + 8.0, cmax, m)
            alpha = torch.exp2(m - m_new)
            o = o * alpha
            if mutant != 8:
                l = l * alpha
            m = m_new
        e = torch.exp2(xs - m)
        l = l + e.sum(-1, keepdim=True)
        if mutant == 1 and xs.shape[-1] < 64:
            l = l + (64 - xs.shape[-1]) * torch.exp2(-m)          # padded keys read as score 0, not zero-filled
        pb = _round7(e) if mutant == 9 else e.bfloat16().float()
        o = o + pb @ vs
    out = (o / l).transpose(1, 2).reshape(B, Lq, HD).bfloat16()
    if mutant == 7:
        out[:, Lq - 1] = out[:, Lq - 2]
    return out


MASK_L2 = -10000.0 * LOG2E


def _case(name):
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    rnd = lambda *s: torch.randn(*s, generator=g)
    if name == "lk16_masked":            # masked text self-attention, shared mask rows (trip_query), lengths 1 .. L
        B, Lq, Lk, H, nkv = 6, 32, 16, 2, 3
        lens = torch.tensor([Lk, 1, 2, Lk - 1])
        mask = (torch.arange(Lk)[None, :] < lens[:, None]).int()
        mask_index = torch.tensor([1, 0, 3, 2, 0, 1], dtype=torch.int32)
    elif name == "lk65_cls":             # one query row, one-key tail chunk
        B, Lq, Lk, H, nkv, mask, mask_index = 40, 1, 65, 4, 5, None, None
    elif name == "lk577_vit_cross":      # the cross-attention shape: 32 text rows x 577 image tokens
        B, Lq, Lk, H, nkv, mask, mask_index = 9, 32, 577, 12, 3, None, None
    elif name == "lq300_lk65_masked":    # long query, tail chunk and masks
        B, Lq, Lk, H, nkv = 3, 300, 65, 2, 2
        lens = torch.tensor([Lk, 40, 64])
        mask = (torch.arange(Lk)[None, :] < lens[:, None]).int()
        mask_index = torch.tensor([1, 2, 0], dtype=torch.int32)
    elif name == "lazy_burst":           # the lazy max moves twice (bursts in chunk 3 and in the last chunks)
        B, Lq, Lk, H, nkv, mask, mask_index = 8, 32, 577, 12, 2, None, None
    else:
        raise KeyError(name)
    q = rnd(B, Lq, H * 64).bfloat16()
    k = rnd(nkv, Lk, H * 64)
    if name == "lazy_burst":
        k[:, 200:260] *= 6.0
        k[:, 500:] *= 12.0
    k = k.bfloat16()
    v = rnd(nkv, Lk, H * 64).bfloat16()
    kv_index = torch.tensor(sorted(i % nkv for i in range(B)), dtype=torch.int32)
    return dict(q=q, k=k, v=v, key_mask=mask, kv_index=kv_index, mask_index=mask_index)


CASES = ["lk16_masked", "lk65_cls", "lk577_vit_cross", "lq300_lk65_masked", "lazy_burst"]


def _applies(mutant, name, a):
    Lq, Lk = a["q"].shape[1], a["k"].shape[1]
    masked = a["key_mask"] is not None
    return {1: Lk % 64 != 0 and name != "lazy_burst",      # exp2(-m) vanishes once the burst sets m
            2: True, 3: Lk % 64 == 1, 4: masked, 5: masked and a["mask_index"] is not None,
            6: a["k"].shape[0] > 1, 7: Lq >= 2, 8: name == "lazy_burst"}[mutant]


@pytest.fixture(scope="module")
def cases():
    out = {}
    for name in CASES:
        a = _case(name)
        out[name] = (a, ref_attention64(**a))
    return out


def test_simulated_kernel_within_bound(cases):
    worst = 0.0
    for name in CASES:
        a, ref = cases[name]
        ratio, where = check_attention(simulate(**a), ref, "bf16")
        print(f"{name}: correct kernel error/bound = {ratio:.3f} at {where}")
        assert ratio <= 1.0, (name, ratio, where)
        worst = max(worst, ratio)
    assert worst >= 0.5, worst


@pytest.mark.parametrize("mutant", range(1, 9))
def test_mutant_rejected(cases, mutant):
    seen = []
    for name in CASES:
        a, ref = cases[name]
        if not _applies(mutant, name, a):
            continue
        ratio, where = check_attention(simulate(**a, mutant=mutant), ref, "bf16")
        print(f"mutant {mutant} on {name}: error/bound = {ratio:.3g} at {where}")
        seen.append(name)
        assert ratio > 2, (name, ratio, where)
    assert seen


def test_seven_bit_p_flagged():
    """One key with score 0 (P = 1, v = 0) sets the max; n keys have P just above and n just below
    0.5 * (1 + 2^-7), which bf16 holds exactly and the 7-bit grid has as a midpoint.  v = +1 on the first group
    and -1 on the second: the output is ~0 and every 7-bit rounding error (up on +1, down on -1) adds up."""
    n, Lq = 20, 2
    mid = 0.5 * (1 + 2 ** -7)
    q = torch.zeros(1, Lq, 64)
    q[..., 0] = 8.0                                          # scale 1/8 -> score = k[:, 0]
    k = torch.zeros(1, 1 + 2 * n, 64)
    k[0, 1:1 + n, 0] = math.log(mid * (1 + 2 ** -13))
    k[0, 1 + n:, 0] = math.log(mid * (1 - 2 ** -13))
    v = torch.zeros(1, 1 + 2 * n, 64)
    v[0, 1:1 + n] = 1.0
    v[0, 1 + n:] = -1.0
    a = dict(q=q, k=k, v=v)
    ref = ref_attention64(**a)
    good, _ = check_attention(simulate(q.bfloat16(), k, v.bfloat16()), ref, "bf16")
    bad, where = check_attention(simulate(q.bfloat16(), k, v.bfloat16(), mutant=9), ref, "bf16")
    print(f"7-bit P: correct {good:.3f}, mutant {bad:.3f} at {where}")
    assert good <= 0.7 and bad > 1, (good, bad)
