"""fp64 reference of cir_attention / cir_qkv_attention and the rounding-error bound their outputs must meet.

The reference is softmax(Q K^T * scale + (1 - mask) * -10000) V evaluated in fp64 from the same (bf16 or fp32)
inputs the kernel read, so the only difference left is the kernel's own rounding.  ``check_attention`` divides the
elementwise error by a bound built from the kernels' rounding points and returns the largest ratio; a correct kernel
stays <= 1 on every input, and the test suite asserts exactly that.

Derivation.  Write p_k for the exact softmax weights of one output row (sum 1), o = sum_k p_k v_k for the exact
output, A = sum_k p_k |v_k| (>= |o|) and u = 2^-8 for the unit roundoff of bf16 (8 significant bits: round to
nearest is within 2^-8 of the value, relative).  The bf16 kernels (tcgen05, mma.sync, small, simt<bf16>, fused QKV)
compute:

1. P = exp2(S * scale * log2(e) - m) in fp32 against a reference max m.  m is the exact running max (mma.sync,
   small), or a lazy one that moves only when the row max grew by more than 2^8 (tcgen05), so P <= 256 and fp32
   holds it without overflow or meaningful underflow.  A common factor 2^-m cancels in O / l.
2. P rounded to bf16 for the PV product (tensor-core kernels): P_k (1 + e_k), |e_k| <= u.  The row sum l adds the
   unrounded fp32 P, so the numerator error is sum_k p_k e_k v_k: at most u * A.  (Had l summed the rounded P too,
   the error would be sum_k p_k e_k (v_k - o): at most u * (A + |o|).  The bound covers both.)  simt<bf16> keeps P
   in fp32 and skips this step.
3. The output rounded to bf16: at most u * |o| (plus u times the error above, second order).

   First order that is u * (A + |o|) -- in the notation c * 2^-9 * (A + |o|), c = 2.  It is reached: a row with
   one dominant key (p_max = 1 exactly, |o| = A) whose output lies near a bf16 rounding midpoint has an error
   close to u * |o| = 2^-9 * (A + |o|); c = 1 would fail a correct kernel there.

4. fp32 arithmetic, all orders of summation, and 2 u per addition to allow for truncating tensor-core accumulators:
   the row sum l (Lk additions), the PV accumulation (2 Lk u A), the O / l rescales of an online or lazy max
   (two roundings per 64-key chunk, at most 16 chunks) and the final reciprocal and product:
   u32 * (3 Lk + 48) * (A + |o|), u32 = 2^-24.
5. Score errors.  A perturbation d_k of score k (in the natural-log domain) changes p_k by p_k (e^d_k - 1) and the
   output, after renormalisation, by at most sum_k p_k (e^|d_k| - 1) (|v_k| + |o|).  The kernels' scores carry
   - the fp32 dot product of 64 head dimensions, 2 u32 per step: scale * 132 u32 * sum_d |q_d k_d|,
   - rounding of scale * log2(e), the FMA with it and the subtraction of m: 3 u32 (|s| + |x| + 6), where s is
     the scaled score, x = s - max and 6 > 8 ln 2 covers a lazy max that sits up to 2^8 below the row max,
   - exp2 itself (MUFU.EX2 or exp2f/expf): relative 2^-21 at most.
   Masked keys (-10000) have p = 0 in fp64 and in the kernels, so they add nothing.
6. Perturbed inputs.  ``dq``/``dk``/``dv`` are elementwise bounds of how far the kernel's q/k/v may be from the
   reference's.  cir_qkv_attention projects Q|K|V with an fp32 accumulator and rounds to bf16; the fp64
   projection rounded to bf16 can land one bf16 ulp away where the exact value sits next to a rounding midpoint
   (or, for values that cancel to near zero, as far as the fp32 accumulation error).
   A q flip moves the scores of its row by scale * dq_d |k_d|, a k flip the scores of its key by scale * |q_d| dk_d,
   both handled like 5; a v flip moves the output by sum_k p_k dv_k.

The fp32 form (simt<float>, every fp32-context attention) drops steps 2 and 3 and rounds the output to fp32
(inside the 48 of step 4).  A floor of 2^-60 absorbs flushed denormals; nothing else is absolute.

What the bound cannot see: a kernel that rounds P to 7 instead of 8 significant bits errs by at most 2^-7 * A,
twice the largest error step 2 allows, so such a kernel stays below ratio 2.  tests/test_attention_bound.py shows
it is still flagged (ratio > 1) on an input whose P is exact in bf16 but not in 7 bits.
"""
from __future__ import annotations

from typing import NamedTuple

import torch

U_BF16 = 2.0 ** -8
U_F32 = 2.0 ** -24
EXP2_REL = 2.0 ** -21
FLOOR = 2.0 ** -60
MASK_ADD = -10000.0


class AttnRef(NamedTuple):
    o: torch.Tensor          # fp64 [B, Lq, H*64]
    absv: torch.Tensor       # fp64 sum_k p_k |v_k|, same shape
    es: torch.Tensor         # fp64 absolute error allowed for score and input perturbations (steps 5 and 6)
    Lk: int


def _heads(t, H):
    return t.reshape(t.shape[0], t.shape[1], H, 64).transpose(1, 2)


def ref_attention64(q, k, v, key_mask=None, kv_index=None, mask_index=None, scale=0.125, dq=None, dk=None, dv=None,
                    max_elems=1 << 25) -> AttnRef:
    """q [B,Lq,H*64], k/v [Bk,Lk,H*64] (any dtype, any strides, one device) -> AttnRef in fp64.  key_mask int
    [*, Lk] (1 = attend), row mask_index[b] (default b) for batch b; kv_index[b] (default b) names the K/V batch.
    dq/dk/dv: optional elementwise bounds of input perturbations, shaped like q/k/v."""
    B, Lq, HD = q.shape
    Lk = k.shape[1]
    H = HD // 64
    dev = q.device
    kvi = torch.arange(B, device=dev) if kv_index is None else kv_index.to(dev).long()
    mi = torch.arange(B, device=dev) if mask_index is None else mask_index.to(dev).long()
    step = max(1, max_elems // max(1, H * Lq * Lk))
    outs, absvs, ess = [], [], []
    for b0 in range(0, B, step):
        sl = slice(b0, min(B, b0 + step))
        qh = _heads(q[sl].double(), H)
        kh = _heads(k[kvi[sl]].double(), H)
        vh = _heads(v[kvi[sl]].double(), H)
        s = (qh @ kh.transpose(-1, -2)) * scale
        if key_mask is not None:
            s = s + (1.0 - key_mask.to(dev)[mi[sl]].double())[:, None, None, :] * MASK_ADD
        mx = s.amax(-1, keepdim=True)
        x = s - mx
        p = torch.exp(x)
        p = p / p.sum(-1, keepdim=True)
        o = p @ vh
        av = vh.abs()
        absv = p @ av
        d = scale * 132 * U_F32 * (qh.abs() @ kh.abs().transpose(-1, -2)) + 3 * U_F32 * (s.abs() + x.abs() + 6.0) + EXP2_REL
        if dq is not None:
            d = d + scale * (_heads(dq[sl].double(), H) @ kh.abs().transpose(-1, -2))
        if dk is not None:
            d = d + scale * (qh.abs() @ _heads(dk[kvi[sl]].double(), H).transpose(-1, -2))
        pd = torch.where(p > 0, p * torch.expm1(d), torch.zeros_like(p))     # masked keys: p = 0 (x ~ -10000)
        es = pd @ av + pd.sum(-1, keepdim=True) * o.abs()
        if dv is not None:
            es = es + p @ _heads(dv[kvi[sl]].double(), H)
        back = lambda t: t.transpose(1, 2).reshape(t.shape[0], Lq, HD)
        outs.append(back(o)); absvs.append(back(absv)); ess.append(back(es))
    return AttnRef(torch.cat(outs), torch.cat(absvs), torch.cat(ess), Lk)


def bf16_ulp(t):
    """Spacing of the bf16 grid at |t| (normal range)."""
    _, e = torch.frexp(t.double().abs().clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(e, dtype=torch.float64), e - 8)


def qkv_attention_ref64(x, w, bias, mask, mask_index, qkv_kernel, scale=0.125):
    """fp64 restatement of cir_qkv_attention over x [batch, caps, L, 768]: Q|K|V = x w^T + bias in fp64, rounded to
    bf16 as the kernel rounds its projection, then ref_attention64 per stream.  ``qkv_kernel`` [batch, caps*L, 2304]
    is the bf16 projection a GPU GEMM produced from the same operands: it may differ from the rounded fp64 one by
    one bf16 ulp next to rounding midpoints, or by the fp32 accumulation error where the sum cancels to near zero
    (asserted here); those differences enter the bound through dq/dk/dv.
    -> list of AttnRef, one per stream."""
    batch, caps, L, HD = x.shape
    proj = torch.einsum("bmk,bnk->bmn", x.reshape(batch, caps * L, HD).double(), w.double())
    if bias is not None:
        proj = proj + bias.double()[:, None, :]
    acc = torch.einsum("bmk,bnk->bmn", x.reshape(batch, caps * L, HD).double().abs(), w.double().abs())
    if bias is not None:
        acc = acc + bias.double().abs()[:, None, :]
    qkv = proj.bfloat16()
    flip = (qkv_kernel.double() - qkv.double()).abs()
    # one bf16 ulp, or where the sum cancels to near zero the fp32 accumulation error (2 u32 per step of K = 768)
    assert bool((flip <= bf16_ulp(proj) + 2 * (HD + 1) * U_F32 * acc).all()), "projection differs by more than rounding"
    km = None if mask is None else mask[mask_index.long()] if mask_index is not None else mask
    refs = []
    for s in range(batch):
        t, d = qkv[s].reshape(caps, L, 3 * HD), flip[s].reshape(caps, L, 3 * HD)
        part = lambda u, i: u[..., i * HD:(i + 1) * HD]
        refs.append(ref_attention64(part(t, 0), part(t, 1), part(t, 2), key_mask=km, scale=scale,
                                    dq=part(d, 0), dk=part(d, 1), dv=part(d, 2)))
    return refs


def attention_bound(ref: AttnRef, kind: str) -> torch.Tensor:
    """Elementwise bound of |out - ref.o|.  kind: "bf16" (bf16 output, bf16 P or fp32 P) or "fp32" (fp32 context)."""
    assert kind in ("bf16", "fp32"), kind
    mag = ref.absv + ref.o.abs()
    rel = U_F32 * (3 * ref.Lk + 48) + (U_BF16 if kind == "bf16" else 0.0)
    return rel * mag + ref.es + FLOOR


def check_attention(out, ref: AttnRef, kind: str):
    """-> (max |out - ref| / bound, index of the worst element).  Non-finite outputs count as infinitely wrong."""
    err = (out.to(ref.o.device).double() - ref.o).abs()
    err = torch.where(torch.isfinite(err), err, torch.full_like(err, float("inf")))
    r = err / attention_bound(ref, kind)
    flat = int(torch.argmax(r).item())
    return r.reshape(-1)[flat].item(), tuple(int(i) for i in torch.unravel_index(torch.tensor(flat), r.shape))
