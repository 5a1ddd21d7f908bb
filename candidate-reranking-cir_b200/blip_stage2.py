"""Stage-II model wrapper: same surface as the reference's ``BLIP_NLVR`` (src/blip_stage2.py:19-145),
all math in the sm_100a library."""
from __future__ import annotations

from typing import Dict, Optional

import torch
from torch import nn

from . import native as N
from .blip import EncoderOutput, check_vit, init_tokenizer, tokenize
from .engine import Engine, get_engine


class BLIP_NLVR(nn.Module):
    def __init__(self, med_config="configs/med_config.json", image_size=480, vit="base", vit_grad_ckpt=False,
                 vit_ckpt_layer=0, *, state_dict: Optional[Dict[str, torch.Tensor]] = None, precision: str = "bf16",
                 device=None, engine: Optional[Engine] = None,
                 synthetic_tokenizer: bool = False):
        """Signature of src/blip_stage2.py:20-26 plus keyword-only extras: ``state_dict`` (reference
        key names, SURVEY 8b), ``precision`` ("bf16" | "fp32" check mode), ``device``/``engine``.
        ``med_config`` is accepted for compatibility; the dims are the fixed BERT-base/ViT-B ones of
        configs/med_config.json."""
        super().__init__()
        check_vit(vit)
        self.image_size = image_size
        self.engine = engine or get_engine(device, precision)
        self.tokenizer = init_tokenizer(synthetic_tokenizer)
        self._from_checkpoint = False
        self._vit = self._w = None
        self._keep = []
        if state_dict is not None:
            self.load_state_dict(state_dict)

    # nn.Module compatibility used by the reference drivers (validate_stage2.py:288)
    def float(self):
        return self

    def load_state_dict(self, state_dict, strict: bool = True):
        e = self.engine
        self._vit, k1, n_tok = e.pack_vit(state_dict)
        assert n_tok == (self.image_size // 16) ** 2 + 1, "pos_embed does not match image_size"
        self._w, k2 = e.pack_stage2(state_dict)
        self._keep = [k1, k2]
        return self

    def _need_weights(self):
        if self._w is None:
            raise N.CirError("BLIP_NLVR has no weights: pass state_dict= or call load_state_dict()")

    def img_embed(self, image, train=True, atts=False):
        """src/blip_stage2.py:57-63: ViT tokens [B,577,768] (activation dtype)."""
        self._need_weights()
        image_embeds = self.engine.vit_forward(self._vit, image)
        if atts:
            return image_embeds, torch.ones(image_embeds.size()[:-1], dtype=torch.long, device=image_embeds.device)
        return image_embeds

    def img_txt_fusion_val(self, r_image_embeds, t_image_embeds, text):
        """src/blip_stage2.py:101-136: one query (z_t) against K candidate token tensors -> [K] logits."""
        self._need_weights()
        e = self.engine
        z = r_image_embeds.last_hidden_state
        assert z.shape[0] == 1                                                  # :108
        K = t_image_embeds.shape[0]
        ids, mask = tokenize(self.tokenizer, text, e.device)
        assert tuple(z.shape[:2]) == tuple(ids.shape), "left and right inputs shall be the same shape"   # nlvr_encoder.py:891
        cand = e.to_act(t_image_embeds)
        ar = torch.arange(K, dtype=torch.int32, device=e.device)
        scores, _ = e.stage2_score_chunk(self._w, cand, ar, e.to_act(z), ids, mask, torch.zeros_like(ar), ar)
        return scores

    def img_txt_fusion(self, r_image_embeds, t_image_embeds, text, train=True):
        """src/blip_stage2.py:65-99: row i scores query i against all B targets -> [B,B] logits.
        (Forward only; one shared candidate set -> K/V computed once for all B rows.)"""
        self._need_weights()
        e = self.engine
        z = e.to_act(r_image_embeds.last_hidden_state)
        B = z.shape[0]
        ids, mask = tokenize(self.tokenizer, text, e.device)
        cand = e.to_act(t_image_embeds)
        Bt = cand.shape[0]
        cand_idx = torch.arange(Bt, dtype=torch.int32).expand(B, Bt).numpy()
        return e.stage2_score_matrix(self._w, cand, z, ids, mask, cand_idx)

    # ---- batched fast path used by validate_stage2 (candidate-major, gallery-resident)
    def score_triplets(self, z_t, ids, mask, gallery_tokens, cand_idx, row_active=None, kv_cache=None):
        """z_t act [Q,L,768]; ids/mask [Q,L]; gallery_tokens act [G,N,768]; cand_idx [Q,K] -> fp32 [Q,K].
        ``kv_cache``: optional :meth:`kv_cache` of this model covering the candidates (same scores, no per-chunk K/V work)."""
        self._need_weights()
        return self.engine.stage2_score_matrix(self._w, gallery_tokens, z_t, ids, mask, cand_idx, row_active, kv_cache=kv_cache)

    def rerank_topk(self, z_t, ids, mask, cand_idx, kv_cache, out=None):
        """Re-rank a device-resident top-K list cand_idx int32 [Q,K] (e.g. the idx of engine.Stage1Index.topk) through ``kv_cache``
        without the host (engine.Engine.stage2_rerank_cached) -> (scores fp32 [Q,K], order int32 [Q,K], ranked int32 [Q,K]).
        The scores are those of :meth:`score_triplets` with ``kv_cache``; capturable in a CUDA graph."""
        self._need_weights()
        return self.engine.stage2_rerank_cached(self._w, kv_cache, z_t, ids, mask, cand_idx, out=out)

    def kv_cache(self, gallery_tokens, row0: int = 0, rows: Optional[int] = None):
        """The cross-attention K/V of gallery rows [row0, row0 + rows) under this model's weights, computed once
        (engine.Stage2KVCache): 42.5 MB per 384 px image in bf16.  Pass it as ``kv_cache=`` to score_triplets / the drivers."""
        self._need_weights()
        return self.engine.stage2_kv_cache(self._w, gallery_tokens, row0, rows)

    def forward(self, *a, **k):
        raise NotImplementedError("use img_embed / img_txt_fusion_val / img_txt_fusion (the reference defines no forward())")


def blip_stage2(pretrained="", **kwargs):
    """src/blip_stage2.py:139-145.  ``pretrained`` may be a checkpoint path holding
    {'BLIP_NLVR': state_dict} (src/validate_stage2.py:359-360) or {'model': state_dict}."""
    model = BLIP_NLVR(**kwargs)
    if pretrained:
        from .checkpoint import load_state_dict
        from .synthetic import SyntheticTokenizer
        if isinstance(model.tokenizer, SyntheticTokenizer):
            raise N.CirError("a real checkpoint needs the real BERT WordPiece tokenizer: the synthetic hash tokenizer is for "
                             "synthetic weights only (assign model.tokenizer or pass pre-tokenised batches)")
        model.load_state_dict(load_state_dict(pretrained, "BLIP_NLVR", kwargs.get("image_size", model.image_size)))
        model._from_checkpoint = True
    return model
