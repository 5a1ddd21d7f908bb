"""Host-side engine: owns the native context, packs reference ``state_dict``s into the layouts
``include/cir_b200.h`` documents, manages the workspace and drives the C-ABI pipelines.

torch is used for device memory, streams and one-off weight layout preparation only; every
arithmetic step of the hot path is a kernel in ``csrc/``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import native as N
from .schedule import build_attn_tiles, build_attn_work, plan_chunks

HIDDEN, FFN, LAYERS, EMBED = 768, 3072, 12, 256
NEG_FILL = -99999.99          # src/validate_stage2.py:123,258
RERANK_MAX_TRIPLETS = 16384   # triplets per cir_stage2_rerank_cached call (one planning CTA)


class Engine:
    """One engine per (device, precision).  precision: "bf16" (tcgen05 tensor cores) or "fp32"
    (the fp32 check mode of BASELINE.json: CUDA-core fp32 everywhere)."""

    def __init__(self, device: Optional[torch.device | int | str] = None, precision: str = "bf16"):
        if not torch.cuda.is_available():
            raise N.CirError("no CUDA device: the B200 path has no CPU fallback")
        assert precision in ("bf16", "fp32")
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        self.precision = precision
        self.act_dtype = torch.bfloat16 if precision == "bf16" else torch.float32
        self._lib = N.lib()
        h = N.vp()
        N.check(self._lib.cir_create(C.byref(h), dev.index, N.DTYPE_BF16 if precision == "bf16" else N.DTYPE_F32), "cir_create")
        self.ctx = h
        self._ws: Optional[torch.Tensor] = None
        # stage-II chunk limits (triplets / unique candidates per cir_stage2_score call); environment overrides for sweeps
        self.max_triplets = int(os.environ.get("CIR_MAX_TRIPLETS", 4096))
        self.max_candidates = int(os.environ.get("CIR_MAX_CANDIDATES", 64))
        self.query_prefix = True       # stage2_score_matrix: layer 0's query-only part once per query set (cir_stage2_prefix)
        self.prefix_batch = 8192       # queries per cir_stage2_prefix call (bounds its workspace: ~0.7 MB per query at L = 32)
        self._rr_ws: Optional[torch.Tensor] = None    # stage2_rerank_cached's own workspace (never Engine.workspace: see there)
        self._rr_retired: List[torch.Tensor] = []     # outgrown workspaces stay alive: a captured graph may still point at one

    # ------------------------------------------------------------------ plumbing
    def _sync_stream(self):
        N.check(self._lib.cir_set_stream(self.ctx, N.vp(torch.cuda.current_stream(self.device).cuda_stream)))

    def set_gemm_impl(self, impl: int):
        N.check(self._lib.cir_set_gemm_impl(self.ctx, impl), "cir_set_gemm_impl")

    def set_attention_impl(self, impl: int):
        """0 = auto (tcgen05 where eligible, else mma.sync), 1 = CUDA-core kernel, 2 = mma.sync only."""
        N.check(self._lib.cir_set_attention_impl(self.ctx, impl), "cir_set_attention_impl")

    def set_prune_last_layer(self, enable: bool):
        """Stage II: layer 11 for the CLS rows only (default) or for all rows (cross-check)."""
        N.check(self._lib.cir_set_prune_last_layer(self.ctx, 1 if enable else 0))

    def set_gemm_tma_store(self, enable: bool):
        """bf16 GEMM outputs through TMA bulk tensor stores (default on) or per-lane 16 B stores."""
        N.check(self._lib.cir_set_gemm_tma_store(self.ctx, 1 if enable else 0))

    def set_dedup_first_layer(self, enable: bool):
        """stage II: layer 0's query-only part once per unique query of a chunk (default on; exact)."""
        N.check(self._lib.cir_set_dedup_first_layer(self.ctx, 1 if enable else 0))

    def set_fuse_qkv_attention(self, enable: bool):
        """bf16, L in {8, 16, 24, 32}: QKV projection + masked text self-attention as one kernel (default on; bit-equal to the unfused path)."""
        N.check(self._lib.cir_set_fuse_qkv_attention(self.ctx, 1 if enable else 0))

    def set_stage1_tensor_cores(self, enable: bool):
        """bf16, G >= 16,384: stage-I top-K filters candidates on the tensor cores and re-checks them in fp32 (default on; bit-equal)."""
        N.check(self._lib.cir_set_stage1_tensor_cores(self.ctx, 1 if enable else 0))

    def profile_gemm(self, enable: bool):
        N.check(self._lib.cir_profile_gemm(self.ctx, 1 if enable else 0))

    def profile_gemm_read(self):
        """-> (summed GEMM ms, summed algorithmic FLOPs, launches) since profile_gemm(True)."""
        ms, fl, n = C.c_double(), C.c_double(), N.i64()
        N.check(self._lib.cir_profile_gemm_read(self.ctx, C.byref(ms), C.byref(fl), C.byref(n)))
        return ms.value, fl.value, n.value

    def profile_read(self, kind: int):
        """-> (summed ms, summed algorithmic work, launches) of the kernels of ``kind`` (native.PROF_*) since profile_gemm(True)."""
        ms, wk, n = C.c_double(), C.c_double(), N.i64()
        N.check(self._lib.cir_profile_read(self.ctx, kind, C.byref(ms), C.byref(wk), C.byref(n)))
        return ms.value, wk.value, n.value

    def launch_count(self, reset: bool = False) -> int:
        return int(self._lib.cir_launch_count(self.ctx, 1 if reset else 0))

    def workspace(self, nbytes: int) -> torch.Tensor:
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = None
            self._ws = torch.empty(int(nbytes * 1.05) + 4096, dtype=torch.uint8, device=self.device)
        return self._ws

    def dev(self, t: torch.Tensor, dtype=None) -> torch.Tensor:
        return t.to(device=self.device, dtype=dtype or t.dtype).contiguous()

    def to_act(self, t: torch.Tensor) -> torch.Tensor:
        """any float tensor -> contiguous device tensor in the activation dtype (cast by our kernel)."""
        t = t.to(self.device)
        if t.dtype == self.act_dtype:
            return t.contiguous()
        t = t.to(torch.float32).contiguous()
        out = torch.empty(t.shape, dtype=self.act_dtype, device=self.device)
        self._sync_stream()
        N.check(self._lib.cir_cast_f32_to_act(self.ctx, N.ptr(t), N.ptr(out), t.numel()), "cast")
        return out

    def to_f32(self, t: torch.Tensor) -> torch.Tensor:
        if t.dtype == torch.float32:
            return t
        out = torch.empty(t.shape, dtype=torch.float32, device=self.device)
        self._sync_stream()
        N.check(self._lib.cir_cast_act_to_f32(self.ctx, N.ptr(t.contiguous()), N.ptr(out), t.numel()), "cast")
        return out

    def _check_range(self, a, hi: int, what: str):
        """Host-resident index arrays are range-checked before they reach a device gather (the kernels trust them);
        device-resident ones only with ``CIR_CHECK_INDICES=1`` (it costs a stream synchronisation)."""
        if hi is None:
            return
        if isinstance(a, torch.Tensor):
            if a.is_cuda and os.environ.get("CIR_CHECK_INDICES") != "1":
                return
            if a.numel() == 0:
                return
            lo_v, hi_v = int(a.min()), int(a.max())
        else:
            a = np.asarray(a)
            if a.size == 0:
                return
            lo_v, hi_v = int(a.min()), int(a.max())
        if lo_v < 0 or hi_v >= hi:
            raise N.CirError(f"{what}: index range [{lo_v}, {hi_v}] outside [0, {hi}) -- stale top-K file, wrong gallery or wrong tokenizer?")

    def _i32(self, a) -> torch.Tensor:
        if isinstance(a, torch.Tensor):
            return a.to(device=self.device, dtype=torch.int32).contiguous()
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(self.device, non_blocking=True)

    # ------------------------------------------------------------------ weight packing
    def _w(self, t: torch.Tensor) -> torch.Tensor:        # GEMM weight: activation dtype
        return t.detach().to(device=self.device, dtype=torch.float32).to(self.act_dtype).contiguous()

    def _p(self, t: torch.Tensor) -> torch.Tensor:        # bias / LN / tables: fp32
        return t.detach().to(device=self.device, dtype=torch.float32).contiguous()

    def _upload(self, sd, key, hold):
        """One state_dict tensor -> fp32 device pointer for a cir_*_state (None when the key is absent)."""
        if key not in sd:
            return N.vp(0)
        t = self._p(sd[key])
        hold.append(t)
        return N.ptr(t)

    def pack_vit(self, sd: Dict[str, torch.Tensor], prefix: str = "visual_encoder."):
        """visual_encoder.* -> cir_vit_weights through the C-ABI packer (cir_pack_vit_weights): -> (struct, [blob], tokens)."""
        hold: List[torch.Tensor] = []
        st = N.VitState()
        U = lambda name: self._upload(sd, prefix + name, hold)
        st.patch_w, st.patch_b, st.cls_token, st.pos_embed = U("patch_embed.proj.weight"), U("patch_embed.proj.bias"), U("cls_token"), U("pos_embed")
        n_tok = int(sd[prefix + "pos_embed"].reshape(-1, HIDDEN).shape[0])
        st.num_tokens = n_tok
        for i in range(LAYERS):
            b = f"blocks.{i}."
            st.norm1_g[i], st.norm1_b[i] = U(b + "norm1.weight"), U(b + "norm1.bias")
            st.qkv_w[i], st.qkv_b[i] = U(b + "attn.qkv.weight"), U(b + "attn.qkv.bias")
            st.proj_w[i], st.proj_b[i] = U(b + "attn.proj.weight"), U(b + "attn.proj.bias")
            st.norm2_g[i], st.norm2_b[i] = U(b + "norm2.weight"), U(b + "norm2.bias")
            st.fc1_w[i], st.fc1_b[i] = U(b + "mlp.fc1.weight"), U(b + "mlp.fc1.bias")
            st.fc2_w[i], st.fc2_b[i] = U(b + "mlp.fc2.weight"), U(b + "mlp.fc2.bias")
        st.norm_g, st.norm_b = U("norm.weight"), U("norm.bias")
        blob = torch.empty(self._lib.cir_pack_vit_bytes(self.ctx, n_tok), dtype=torch.uint8, device=self.device)
        w = N.VitWeights()
        self._sync_stream()
        N.check(self._lib.cir_pack_vit_weights(self.ctx, C.byref(st), N.ptr(blob), blob.numel(), C.byref(w)), "cir_pack_vit_weights")
        torch.cuda.synchronize(self.device)          # the fp32 uploads in `hold` are released on return
        return w, [blob], n_tok

    def _embed_state(self, sd, emb, hold):
        e = "text_encoder.embeddings."
        emb.word_emb, emb.vocab_rows = self._upload(sd, e + "word_embeddings.weight", hold), int(sd[e + "word_embeddings.weight"].shape[0])
        emb.pos_emb, emb.pos_rows = self._upload(sd, e + "position_embeddings.weight", hold), int(sd[e + "position_embeddings.weight"].shape[0])
        emb.ln_g, emb.ln_b = self._upload(sd, e + "LayerNorm.weight", hold), self._upload(sd, e + "LayerNorm.bias", hold)
        self.vocab_rows = int(emb.vocab_rows)

    def pack_stage1(self, sd: Dict[str, torch.Tensor]):
        """BLIP_Retrieval text encoder + projections -> cir_stage1_weights through cir_pack_stage1_weights: -> (struct, [blob])."""
        hold: List[torch.Tensor] = []
        st = N.Stage1State()
        self._embed_state(sd, st.emb, hold)
        U = lambda name: self._upload(sd, name, hold)
        for i in range(LAYERS):
            p = f"text_encoder.encoder.layer.{i}."
            a, c = p + "attention.", p + "crossattention."
            for nm, f in (("query", "q"), ("key", "k"), ("value", "v")):
                getattr(st, f"self_{f}_w")[i], getattr(st, f"self_{f}_b")[i] = U(a + f"self.{nm}.weight"), U(a + f"self.{nm}.bias")
                getattr(st, f"cross_{f}_w")[i], getattr(st, f"cross_{f}_b")[i] = U(c + f"self.{nm}.weight"), U(c + f"self.{nm}.bias")
            st.self_out_w[i], st.self_out_b[i] = U(a + "output.dense.weight"), U(a + "output.dense.bias")
            st.self_ln_g[i], st.self_ln_b[i] = U(a + "output.LayerNorm.weight"), U(a + "output.LayerNorm.bias")
            st.cross_out_w[i], st.cross_out_b[i] = U(c + "output.dense.weight"), U(c + "output.dense.bias")
            st.cross_ln_g[i], st.cross_ln_b[i] = U(c + "output.LayerNorm.weight"), U(c + "output.LayerNorm.bias")
            st.ffn1_w[i], st.ffn1_b[i] = U(p + "intermediate.dense.weight"), U(p + "intermediate.dense.bias")
            st.ffn2_w[i], st.ffn2_b[i] = U(p + "output.dense.weight"), U(p + "output.dense.bias")
            st.ffn_ln_g[i], st.ffn_ln_b[i] = U(p + "output.LayerNorm.weight"), U(p + "output.LayerNorm.bias")
        st.text_proj_w, st.text_proj_b = U("text_proj.weight"), U("text_proj.bias")
        st.vision_proj_w, st.vision_proj_b = U("vision_proj.weight"), U("vision_proj.bias")
        blob = torch.empty(self._lib.cir_pack_stage1_bytes(self.ctx, st.emb.vocab_rows, st.emb.pos_rows), dtype=torch.uint8, device=self.device)
        w = N.Stage1Weights()
        self._sync_stream()
        N.check(self._lib.cir_pack_stage1_weights(self.ctx, C.byref(st), N.ptr(blob), blob.numel(), C.byref(w)), "cir_pack_stage1_weights")
        torch.cuda.synchronize(self.device)
        return w, [blob]

    def stage2_state(self, sd: Dict[str, torch.Tensor], hold: List[torch.Tensor]):
        """BLIP_NLVR state_dict -> cir_stage2_state (fp32 device uploads are appended to ``hold``)."""
        st = N.Stage2State()
        self._embed_state(sd, st.emb, hold)
        U = lambda name: self._upload(sd, name, hold)
        for i in range(LAYERS):
            p = f"text_encoder.encoder.layer.{i}."
            a, c = p + "attention.", p + "crossattention."
            for s_, ab in ((0, "A"), (1, "B")):
                for nm, f in (("query", "q"), ("key", "k"), ("value", "v")):
                    getattr(st, f"self_{f}_w")[s_][i], getattr(st, f"self_{f}_b")[s_][i] = U(a + f"self{s_}.{nm}.weight"), U(a + f"self{s_}.{nm}.bias")
                    getattr(st, f"cross_{f}_w")[s_][i], getattr(st, f"cross_{f}_b")[s_][i] = U(c + f"self{s_}.{nm}.weight"), U(c + f"self{s_}.{nm}.bias")
                st.self_out_w[s_][i], st.self_out_b[s_][i] = U(a + f"output.dense{s_}.weight"), U(a + f"output.dense{s_}.bias")
                st.self_ln_g[s_][i], st.self_ln_b[s_][i] = U(a + f"output.LayerNorm{ab}.weight"), U(a + f"output.LayerNorm{ab}.bias")
                st.cross_out_w[s_][i], st.cross_out_b[s_][i] = U(c + f"output.dense{s_}.weight"), U(c + f"output.dense{s_}.bias")
                st.cross_ln_g[s_][i], st.cross_ln_b[s_][i] = U(c + f"output.LayerNorm{ab}.weight"), U(c + f"output.LayerNorm{ab}.bias")
            st.merge_w[i], st.merge_b[i] = U(c + "output.merge_layer.weight"), U(c + "output.merge_layer.bias")     # layers 6..11 (src/nlvr_encoder.py:286)
            st.ffn1_w[i], st.ffn1_b[i] = U(p + "intermediate.dense.weight"), U(p + "intermediate.dense.bias")
            st.ffn2_w[i], st.ffn2_b[i] = U(p + "output.dense.weight"), U(p + "output.dense.bias")
            st.ffn_ln_g[i], st.ffn_ln_b[i] = U(p + "output.LayerNorm.weight"), U(p + "output.LayerNorm.bias")
        st.cls0_w, st.cls0_b, st.cls2_w, st.cls2_b = U("cls_head.0.weight"), U("cls_head.0.bias"), U("cls_head.2.weight"), U("cls_head.2.bias")
        return st

    def pack_stage2(self, sd: Dict[str, torch.Tensor]):
        """Twin-stream packing through cir_pack_stage2_weights: stacks the stream tensors and folds the avg / Linear merge of the
        cross-attention output into one [768,1536] matrix per layer (src/nlvr_encoder.py:250-258, composed in fp64 on the device).
        -> (struct, keep-alive list)."""
        hold: List[torch.Tensor] = []
        st = self.stage2_state(sd, hold)
        blob = torch.empty(self._lib.cir_pack_stage2_bytes(self.ctx, st.emb.vocab_rows, st.emb.pos_rows), dtype=torch.uint8, device=self.device)
        w = N.Stage2Weights()
        self._sync_stream()
        N.check(self._lib.cir_pack_stage2_weights(self.ctx, C.byref(st), N.ptr(blob), blob.numel(), C.byref(w)), "cir_pack_stage2_weights")
        torch.cuda.synchronize(self.device)
        return w, [blob]

    # ------------------------------------------------------------------ pipelines
    def vit_forward(self, w, images: torch.Tensor, batch: int = 32) -> torch.Tensor:
        """images fp32 [B,3,S,S] (host or device) -> tokens act [B,N,768]."""
        assert images.dim() == 4 and images.shape[1] == 3 and images.shape[2] == images.shape[3]
        B, S = images.shape[0], images.shape[2]
        n_tok = (S // 16) ** 2 + 1
        out = torch.empty(B, n_tok, HIDDEN, dtype=self.act_dtype, device=self.device)
        self._sync_stream()
        for b0 in range(0, B, batch):
            img = images[b0:b0 + batch].to(self.device, torch.float32, non_blocking=True).contiguous()
            nb = img.shape[0]
            need = self._lib.cir_vit_workspace_bytes(self.ctx, nb, S)
            ws = self.workspace(need)
            N.check(self._lib.cir_vit_forward(self.ctx, C.byref(w), N.ptr(img), nb, S, N.ptr(out[b0:b0 + nb]),
                                              N.ptr(ws), ws.numel()), "cir_vit_forward")
        return out

    def stage1_encode(self, w, gallery_tokens: torch.Tensor, ref_index, ids, mask, want_z=True, want_emb=True,
                      normalize_twice=False, batch: int = 256, workspace: Optional[torch.Tensor] = None):
        """-> (z_t act [Q,L,768] | None, q_emb fp32 [Q,256] | None).  ``workspace``: optional caller-owned uint8 device tensor of at
        least cir_stage1_workspace_bytes for one batch (default: :meth:`workspace`)."""
        self._check_range(ref_index, gallery_tokens.shape[0], "stage1_encode ref_index")
        self._check_range(ids, getattr(self, "vocab_rows", None), "stage1_encode token ids")
        ref_index, ids, mask = self._i32(ref_index), self._i32(ids), self._i32(mask)
        Q, L = ids.shape
        n_tok = gallery_tokens.shape[1]
        assert gallery_tokens.dtype == self.act_dtype and gallery_tokens.is_contiguous()
        z = torch.empty(Q, L, HIDDEN, dtype=self.act_dtype, device=self.device) if want_z else None
        emb = torch.empty(Q, EMBED, dtype=torch.float32, device=self.device) if want_emb else None
        self._sync_stream()
        for q0 in range(0, Q, batch):
            nq = min(batch, Q - q0)
            need = self._lib.cir_stage1_workspace_bytes(self.ctx, nq, L, n_tok)
            ws = self.workspace(need) if workspace is None else workspace
            N.check(self._lib.cir_stage1_encode(
                self.ctx, C.byref(w), N.ptr(gallery_tokens), N.ptr(ref_index[q0:q0 + nq]), N.ptr(ids[q0:q0 + nq]),
                N.ptr(mask[q0:q0 + nq]), nq, L, n_tok, N.ptr(z[q0:q0 + nq]) if want_z else N.vp(0),
                N.ptr(emb[q0:q0 + nq]) if want_emb else N.vp(0), 1 if normalize_twice else 0, N.ptr(ws), ws.numel()),
                "cir_stage1_encode")
        return z, emb

    def stage1_gallery_embed(self, w, tokens: torch.Tensor) -> torch.Tensor:
        G, n_tok = tokens.shape[0], tokens.shape[1]
        out = torch.empty(G, EMBED, dtype=torch.float32, device=self.device)
        ws = self.workspace(G * EMBED * 4 + 512)
        self._sync_stream()
        N.check(self._lib.cir_stage1_gallery_embed(self.ctx, C.byref(w), N.ptr(tokens), G, n_tok, N.ptr(out), N.ptr(ws), ws.numel()),
                "cir_stage1_gallery_embed")
        return out

    def stage2_score_chunk(self, w, gallery_tokens, cand_list, z_t, ids, mask, trip_query, trip_slot, want_feats=False,
                           attn_work=None, attn_tiles=None, attn_tiles_cls=None, prefix=None, out=None, kv_cache=None):
        """One C-ABI call: T triplets sharing C candidates -> (scores fp32 [T], feats fp32 [T,1536] | None).
        ``attn_work``: optional int32 [W,4] K/V-sharing work list (schedule.build_attn_work).
        ``prefix``: optional (a0, qc0) from :meth:`stage2_prefix` for the same Q queries as ids/mask (z_t is then unused).
        ``kv_cache``: optional :class:`Stage2KVCache` holding every candidate of ``cand_list`` (cir_stage2_score_cached; not checked
        here -- :meth:`stage2_score_pairs` checks it); ``gallery_tokens`` is then unused and may be None."""
        cand_list, ids, mask = self._i32(cand_list), self._i32(ids), self._i32(mask)
        trip_query, trip_slot = self._i32(trip_query), self._i32(trip_slot)
        T, Cn, (Q, L) = trip_query.numel(), cand_list.numel(), ids.shape
        if prefix is None:
            assert z_t.shape == (Q, L, HIDDEN) and z_t.dtype == self.act_dtype and z_t.is_contiguous()
        if kv_cache is None:
            n_tok = gallery_tokens.shape[1]
            assert gallery_tokens.dtype == self.act_dtype and gallery_tokens.is_contiguous()
            need = self._lib.cir_stage2_workspace_bytes(self.ctx, T, Cn, Q, L, n_tok)
        else:
            need = self._lib.cir_stage2_score_cached_workspace_bytes(self.ctx, T, Q, L, kv_cache.num_tokens)
        scores = torch.empty(T, dtype=torch.float32, device=self.device) if out is None else out
        assert scores.is_contiguous() and scores.numel() == T and scores.dtype == torch.float32
        feats = torch.empty(T, 2 * HIDDEN, dtype=torch.float32, device=self.device) if want_feats else None
        ws = self.workspace(need)
        aw = None if attn_work is None or len(attn_work) == 0 else self._i32(attn_work)
        at = None if attn_tiles is None or len(attn_tiles) == 0 else self._i32(attn_tiles)
        ac = None if attn_tiles_cls is None or len(attn_tiles_cls) == 0 else self._i32(attn_tiles_cls)
        self._sync_stream()
        if kv_cache is not None:
            a0, qc0 = (None, None) if prefix is None else prefix
            if prefix is not None:
                assert a0.shape == (2, Q * L, HIDDEN) and qc0.shape == a0.shape and a0.dtype == self.act_dtype
            N.check(self._lib.cir_stage2_score_cached(
                self.ctx, C.byref(w), C.byref(kv_cache._s), N.ptr(cand_list), Cn, N.ptr(z_t if prefix is None else None), N.ptr(ids),
                N.ptr(a0), N.ptr(qc0), N.ptr(mask), Q, L, N.ptr(trip_query), N.ptr(trip_slot), T, N.ptr(aw),
                0 if aw is None else aw.shape[0], N.ptr(at), 0 if at is None else at.shape[0], N.ptr(ac), 0 if ac is None else ac.shape[0],
                N.ptr(scores), N.ptr(feats), N.ptr(ws), ws.numel()), "cir_stage2_score_cached")
            return scores, feats
        tail = (Q, L, n_tok, N.ptr(trip_query), N.ptr(trip_slot), T, N.ptr(aw), 0 if aw is None else aw.shape[0],
                N.ptr(at), 0 if at is None else at.shape[0], N.ptr(ac), 0 if ac is None else ac.shape[0], N.ptr(scores), N.ptr(feats),
                N.ptr(ws), ws.numel())
        if prefix is None:
            N.check(self._lib.cir_stage2_score(self.ctx, C.byref(w), N.ptr(gallery_tokens), N.ptr(cand_list), Cn, N.ptr(z_t), N.ptr(ids),
                                               N.ptr(mask), *tail), "cir_stage2_score")
        else:
            a0, qc0 = prefix
            assert a0.shape == (2, Q * L, HIDDEN) and qc0.shape == a0.shape and a0.dtype == self.act_dtype
            N.check(self._lib.cir_stage2_score_prefixed(self.ctx, C.byref(w), N.ptr(gallery_tokens), N.ptr(cand_list), Cn, N.ptr(a0),
                                                        N.ptr(qc0), N.ptr(mask), *tail), "cir_stage2_score_prefixed")
        return scores, feats

    def stage2_prefix(self, w, z_t, ids, mask, batch: Optional[int] = None):
        """Layer 0's query-only part for a whole query set (cir_stage2_prefix) -> (a0, qc0), each act [2, Q*L, 768].
        Query sets larger than ``batch`` (default ``self.prefix_batch``) go through several calls to bound the workspace."""
        ids, mask = self._i32(ids), self._i32(mask)
        Q, L = ids.shape
        assert z_t.shape == (Q, L, HIDDEN) and z_t.dtype == self.act_dtype and z_t.is_contiguous()
        batch = self.prefix_batch if batch is None else batch
        a0 = torch.empty(2, Q * L, HIDDEN, dtype=self.act_dtype, device=self.device)
        qc0 = torch.empty_like(a0)
        self._sync_stream()
        for q0 in range(0, Q, batch):
            nb = min(batch, Q - q0)
            whole = nb == Q
            a_b = a0 if whole else torch.empty(2, nb * L, HIDDEN, dtype=self.act_dtype, device=self.device)
            q_b = qc0 if whole else torch.empty_like(a_b)
            ws = self.workspace(self._lib.cir_stage2_prefix_workspace_bytes(self.ctx, nb, L))
            N.check(self._lib.cir_stage2_prefix(self.ctx, C.byref(w), N.ptr(z_t[q0:q0 + nb]), N.ptr(ids[q0:q0 + nb]), N.ptr(mask[q0:q0 + nb]),
                                                nb, L, N.ptr(a_b), N.ptr(q_b), N.ptr(ws), ws.numel()), "cir_stage2_prefix")
            if not whole:
                a0[:, q0 * L:(q0 + nb) * L].copy_(a_b)
                qc0[:, q0 * L:(q0 + nb) * L].copy_(q_b)
        return a0, qc0

    def _upload_i32(self, arrays: List[np.ndarray]) -> List[torch.Tensor]:
        """Many small int32 host arrays -> device tensors with ONE pinned staging copy (one H2D instead of one per array;
        flat_pos arrays are int64 and travel as int32 pairs).  The staging buffer is reused: the copy that last read it is
        waited for before it is overwritten."""
        sizes = [int(a.size) * (2 if a.dtype == np.int64 else 1) for a in arrays]
        offs = np.concatenate([[0], np.cumsum([(n + 3) & ~3 for n in sizes])]).astype(np.int64)      # 16 B aligned slices
        total = int(offs[-1])
        if total == 0:
            return [torch.empty(a.shape, dtype=torch.int64 if a.dtype == np.int64 else torch.int32, device=self.device) for a in arrays]
        if getattr(self, "_stage_host", None) is None or self._stage_host.numel() < total:
            self._stage_host = torch.empty(max(total, 1 << 20), dtype=torch.int32).pin_memory()
            self._stage_event = None
        if self._stage_event is not None:
            self._stage_event.synchronize()
        host = self._stage_host.numpy()
        for a, o, n in zip(arrays, offs[:-1], sizes):
            if n:
                host[o:o + n] = np.ascontiguousarray(a).reshape(-1).view(np.int32)
        dev = self._stage_host[:total].to(self.device, non_blocking=True)
        self._stage_event = torch.cuda.Event()
        self._stage_event.record(torch.cuda.current_stream(self.device))
        self.h2d_bytes = getattr(self, "h2d_bytes", 0) + total * 4
        out = []
        for a, o, n in zip(arrays, offs[:-1], sizes):
            t = dev[o:o + n]
            out.append(t.view(torch.int64).view(a.shape) if a.dtype == np.int64 else t.view(a.shape))
        return out

    def stage2_score_pairs(self, w, gallery_tokens, z_t, ids, mask, cand_idx, row_active=None, part=None, kv_cache=None):
        """Score this process's share of the Q*K triplets, candidate-major.  ``part=(rank, world)`` restricts the work to the
        rank's contiguous candidate range (schedule.candidate_partition): every candidate's K/V projections stay on ONE rank,
        so the per-GPU K/V reuse does not fall with the number of GPUs.  z_t act [Q,L,768] / ids / mask [Q,L] cover ALL Q queries.
        ``kv_cache``: a :class:`Stage2KVCache` filled with ``w`` that holds every candidate this process scores: the chunks then
        read their K/V from it (cir_stage2_score_cached) and are bounded by ``max_triplets`` only.  It is checked against ``w``,
        the token count of ``gallery_tokens`` and the candidates before anything launches (CirError).
        -> (flat_pos int64 [n] = q*K+k of each scored triplet, scores fp32 [n]) on the device."""
        cand_np = cand_idx.cpu().numpy() if isinstance(cand_idx, torch.Tensor) else np.asarray(cand_idx)
        Q, K = cand_np.shape
        self._check_range(cand_np, gallery_tokens.shape[0], "stage2_score_matrix cand_idx")
        self._check_range(ids, getattr(self, "vocab_rows", None), "stage2_score_matrix token ids")
        act_np = None if row_active is None else np.asarray(row_active, dtype=bool)
        info: dict = {}
        if kv_cache is not None:
            kv_cache._check_use(self, w, gallery_tokens.shape[1])
        # the cached path keeps no per-chunk K/V, so nothing bounds the unique candidates of a chunk
        max_cand = self.max_candidates if kv_cache is None else max(1, Q * K)
        chunks = plan_chunks(cand_np, act_np, self.max_triplets, max_cand, part=part, info=info)
        if kv_cache is not None and chunks:
            kv_cache._check_rows(min(int(c.cand_list[0]) for c in chunks), max(int(c.cand_list[-1]) for c in chunks))
        self.last_plan = {"part_sizes": info["part_sizes"], "chunks": len(chunks), "triplets": int(sum(c.flat_pos.size for c in chunks)),
                          "candidate_loads": int(sum(c.cand_list.size for c in chunks))}
        ids_d, mask_d = self._i32(ids), self._i32(mask)
        L = ids_d.shape[1]
        if not chunks:
            return (torch.empty(0, dtype=torch.int64, device=self.device), torch.empty(0, dtype=torch.float32, device=self.device))
        use_prefix = self.query_prefix and len(chunks) > 1
        # every index array of every chunk in one upload
        host: List[np.ndarray] = []
        for ch in chunks:
            tq = ch.query_list[ch.trip_query] if use_prefix else ch.trip_query     # prefix: global query rows
            host += [ch.cand_list, tq.astype(np.int32), ch.trip_slot, build_attn_work(ch.trip_slot, L), build_attn_tiles(ch.trip_slot, L),
                     build_attn_tiles(ch.trip_slot, 1), ch.flat_pos, ch.query_list.astype(np.int64)]
        dev = self._upload_i32(host)
        prefix = self.stage2_prefix(w, z_t, ids_d, mask_d) if use_prefix else None
        scores = torch.empty(self.last_plan["triplets"], dtype=torch.float32, device=self.device)
        pos = torch.empty(self.last_plan["triplets"], dtype=torch.int64, device=self.device)
        o = 0
        for i, ch in enumerate(chunks):
            cl, tq, ts, aw, at, ac, fp, ql = dev[8 * i:8 * i + 8]
            lists = dict(attn_work=aw, attn_tiles=at, attn_tiles_cls=ac)
            n = ch.flat_pos.size
            if prefix is not None:                              # global query rows: no per-chunk selection of z_t / ids / mask
                s, _ = self.stage2_score_chunk(w, gallery_tokens, cl, None, ids_d, mask_d, tq, ts, prefix=prefix, out=scores[o:o + n],
                                               kv_cache=kv_cache, **lists)
            else:
                s, _ = self.stage2_score_chunk(w, gallery_tokens, cl, z_t.index_select(0, ql).contiguous(), ids_d.index_select(0, ql),
                                               mask_d.index_select(0, ql), tq, ts, out=scores[o:o + n], kv_cache=kv_cache, **lists)
            pos[o:o + n] = fp
            o += n
        return pos, scores

    def stage2_score_matrix(self, w, gallery_tokens, z_t, ids, mask, cand_idx, row_active=None, kv_cache=None):
        """All Q*K triplets, candidate-major.  z_t act [Q,L,768]; ids/mask [Q,L]; cand_idx [Q,K] ->
        scores fp32 [Q,K]; inactive rows are filled with -99999.99 (src/validate_stage2.py:123,258).
        With more than one chunk, layer 0's query-only part is computed once for all Q queries (stage2_prefix) instead of
        once per chunk for the chunk's unique queries.  ``kv_cache``: see :meth:`stage2_score_pairs` (same scores, bit for bit)."""
        Q, K = cand_idx.shape
        pos, s = self.stage2_score_pairs(w, gallery_tokens, z_t, ids, mask, cand_idx, row_active, kv_cache=kv_cache)
        out = torch.full((Q * K,), NEG_FILL, dtype=torch.float32, device=self.device)
        out.index_copy_(0, pos, s)
        return out.view(Q, K)

    def stage2_rerank_cached(self, w, kv_cache: "Stage2KVCache", z_t, ids, mask, cand, out=None):
        """Re-rank the candidate lists cand int [Q,K] (normally the idx of :meth:`Stage1Index.topk`, already on the device) through
        the resident K/V gallery, with no host round trip (cir_stage2_rerank_cached): the candidate-major plan is built on the
        device, so nothing is read back and the call can be captured in a CUDA graph.  z_t act [Q,L,768]; ids / mask [Q,L].
        -> (scores fp32 [Q,K], order int32 [Q,K] = rerank_sort(scores), ranked int32 [Q,K] = cand[q, order[q, r]]).

        The scores equal stage2_score_matrix(..., kv_cache=kv_cache) when that runs as one chunk, bit for bit.  Entries of -1 (the
        padding of a filtered search) or outside the cache's rows score -99999.99 and rank last.  Query sets larger than
        max(1, max_triplets // K) queries go through several calls; none synchronises.  The cache is checked against ``w`` on the
        host, the candidates are not (they stay on the device).  ``out``: optional (scores, order, ranked) to fill; with device
        int32 cand / ids / mask and ``out``, a warmed-up call allocates and uploads nothing."""
        kv_cache._check_use(self, w, kv_cache.num_tokens)
        cand, ids, mask = self._i32(cand), self._i32(ids), self._i32(mask)
        assert cand.dim() == 2 and ids.dim() == 2 and mask.shape == ids.shape
        Q, K = cand.shape
        L = ids.shape[1]
        assert ids.shape[0] == Q and z_t.shape == (Q, L, HIDDEN) and z_t.dtype == self.act_dtype and z_t.is_contiguous()
        if out is None:
            out = (torch.empty(Q, K, dtype=torch.float32, device=self.device), torch.empty(Q, K, dtype=torch.int32, device=self.device),
                   torch.empty(Q, K, dtype=torch.int32, device=self.device))
        scores, order, ranked = out
        assert scores.shape == order.shape == ranked.shape == (Q, K) and scores.dtype == torch.float32
        assert order.dtype == ranked.dtype == torch.int32 and all(t.is_contiguous() for t in out)
        qb = max(1, min(self.max_triplets, RERANK_MAX_TRIPLETS) // K)
        need = self._lib.cir_stage2_rerank_cached_workspace_bytes(self.ctx, min(qb, Q), K, L, kv_cache.num_tokens)
        if self._rr_ws is None or self._rr_ws.numel() < need:
            if self._rr_ws is not None:
                self._rr_retired.append(self._rr_ws)
            self._rr_ws = torch.empty(max(need, 256), dtype=torch.uint8, device=self.device)
        ws = self._rr_ws
        self._sync_stream()
        for q0 in range(0, Q, qb):
            n = min(qb, Q - q0)
            N.check(self._lib.cir_stage2_rerank_cached(
                self.ctx, C.byref(w), C.byref(kv_cache._s), N.ptr(cand[q0:q0 + n]), n, K, N.ptr(z_t[q0:q0 + n]), N.ptr(ids[q0:q0 + n]),
                N.ptr(mask[q0:q0 + n]), L, N.ptr(scores[q0:q0 + n]), N.ptr(order[q0:q0 + n]), N.ptr(ranked[q0:q0 + n]), None,
                N.ptr(ws), ws.numel()), "cir_stage2_rerank_cached")
        return scores, order, ranked

    # ------------------------------------------------------------------ sort / top-K / recall
    def rerank_sort(self, scores: torch.Tensor) -> torch.Tensor:
        scores = scores.to(self.device, torch.float32).contiguous()
        Q, K = scores.shape
        order = torch.empty(Q, K, dtype=torch.int32, device=self.device)
        self._sync_stream()
        N.check(self._lib.cir_rerank_sort(self.ctx, N.ptr(scores), Q, K, N.ptr(order)), "cir_rerank_sort")
        return order

    def topk_from_dist(self, dist: torch.Tensor, k: int, exclude=None, col_offset: int = 0):
        dist = dist.to(self.device, torch.float32).contiguous()
        Q, G = dist.shape
        td = torch.empty(Q, k, dtype=torch.float32, device=self.device)
        ti = torch.empty(Q, k, dtype=torch.int32, device=self.device)
        ex = None if exclude is None else self._i32(exclude)
        ws = self.workspace(self._lib.cir_topk_workspace_bytes(Q, G, k))
        self._sync_stream()
        N.check(self._lib.cir_topk_from_dist(self.ctx, N.ptr(dist), Q, G, G, N.ptr(ex), col_offset, k, N.ptr(td), N.ptr(ti),
                                             N.ptr(ws), ws.numel()), "cir_topk_from_dist")
        return td, ti

    def stage1_topk(self, q_emb: torch.Tensor, g_emb: torch.Tensor, k: int, exclude=None, col_offset: int = 0):
        q_emb = q_emb.to(self.device, torch.float32).contiguous()
        g_emb = g_emb.to(self.device, torch.float32).contiguous()
        Q, G = q_emb.shape[0], g_emb.shape[0]
        td = torch.empty(Q, k, dtype=torch.float32, device=self.device)
        ti = torch.empty(Q, k, dtype=torch.int32, device=self.device)
        ex = None if exclude is None else self._i32(exclude)
        ws = self.workspace(self._lib.cir_stage1_topk_workspace_bytes(Q, G, k))
        self._sync_stream()
        N.check(self._lib.cir_stage1_topk(self.ctx, N.ptr(q_emb), N.ptr(g_emb), Q, G, N.ptr(ex), col_offset, k, N.ptr(td),
                                          N.ptr(ti), N.ptr(ws), ws.numel()), "cir_stage1_topk")
        return td, ti

    def stage2_kv_cache(self, w, gallery_tokens: torch.Tensor, row0: int = 0, rows: Optional[int] = None) -> "Stage2KVCache":
        """A resident cross-attention K/V gallery (cir_stage2_kv_cache) of gallery rows [row0, row0 + rows) (default: to the end of
        ``gallery_tokens``, act [G,N,768]), filled with the packed stage-II weights ``w``: 42.5 MB per image in bf16 at N = 577."""
        G, n_tok = gallery_tokens.shape[0], gallery_tokens.shape[1]
        rows = G - row0 if rows is None else rows
        if row0 < 0 or rows < 0 or row0 + rows > G:
            raise N.CirError(f"stage2_kv_cache: rows [{row0}, {row0 + rows}) outside the gallery's [0, {G})")
        cache = Stage2KVCache(self, w, rows, n_tok, row0=row0)
        return cache.fill(gallery_tokens[row0:row0 + rows], row0)

    def stage1_index(self, capacity: int) -> "Stage1Index":
        """An empty resident stage-I gallery index for up to ``capacity`` rows (cir_stage1_index): fill it with
        :meth:`Stage1Index.add` once, search it with :meth:`Stage1Index.topk` for every query batch."""
        return Stage1Index(self, capacity)

    def stage1_rank_members(self, q_emb: torch.Tensor, g_emb: torch.Tensor, members):
        """members int [Q,P] gallery rows -> (dist fp32 [Q,P], order int32 [Q,P]: slot of the r-th closest member)."""
        q_emb = q_emb.to(self.device, torch.float32).contiguous()
        g_emb = g_emb.to(self.device, torch.float32).contiguous()
        self._check_range(members, g_emb.shape[0], "stage1_rank_members")
        mem = self._i32(members)
        Q, P = mem.shape
        md = torch.empty(Q, P, dtype=torch.float32, device=self.device)
        mo = torch.empty(Q, P, dtype=torch.int32, device=self.device)
        self._sync_stream()
        N.check(self._lib.cir_stage1_rank_members(self.ctx, N.ptr(q_emb), N.ptr(g_emb), N.ptr(mem), Q, P, N.ptr(md), N.ptr(mo)),
                "cir_stage1_rank_members")
        return md, mo

    def stage1_logits(self, q_emb: torch.Tensor, t_emb: torch.Tensor, temp: float) -> torch.Tensor:
        """q_emb [Q,256] @ t_emb [G,256]^T / temp in fp32 (src/blip_stage1.py:90-91)."""
        q_emb = q_emb.to(self.device, torch.float32).contiguous()
        t_emb = t_emb.to(self.device, torch.float32).contiguous()
        out = torch.empty(q_emb.shape[0], t_emb.shape[0], dtype=torch.float32, device=self.device)
        self._sync_stream()
        N.check(self._lib.cir_stage1_logits(self.ctx, N.ptr(q_emb), N.ptr(t_emb), q_emb.shape[0], t_emb.shape[0], float(temp),
                                            N.ptr(out)), "cir_stage1_logits")
        return out

    def topk_merge(self, dist_in: torch.Tensor, idx_in: torch.Tensor):
        """dist_in/idx_in [P,Q,K] (per-shard sorted lists) -> merged (dist [Q,K], idx [Q,K])."""
        P, Q, K = dist_in.shape
        dist_in = dist_in.to(self.device, torch.float32).contiguous()
        idx_in = idx_in.to(self.device, torch.int32).contiguous()
        td = torch.empty(Q, K, dtype=torch.float32, device=self.device)
        ti = torch.empty(Q, K, dtype=torch.int32, device=self.device)
        ws = self.workspace(self._lib.cir_topk_workspace_bytes(Q, 0, K))
        self._sync_stream()
        N.check(self._lib.cir_topk_merge(self.ctx, N.ptr(dist_in), N.ptr(idx_in), P, Q, K, N.ptr(td), N.ptr(ti), N.ptr(ws), ws.numel()),
                "cir_topk_merge")
        return td, ti

    def recall_counts(self, labels: torch.Tensor, order: torch.Tensor, ks: Sequence[int], sync: bool = True):
        """-> hit counts per k: a python list (device -> host read, synchronises) or, with sync=False, the int64 device tensor."""
        labels = labels.to(self.device).to(torch.uint8).contiguous()
        order = order.to(self.device, torch.int32).contiguous()
        Q, K = labels.shape
        hits = torch.zeros(len(ks), dtype=torch.int64, device=self.device)
        arr = (N.i32 * len(ks))(*[int(k) for k in ks])
        self._sync_stream()
        N.check(self._lib.cir_recall_counts(self.ctx, N.ptr(labels), N.ptr(order), Q, K, arr, len(ks), N.ptr(hits)), "cir_recall_counts")
        return hits.cpu().tolist() if sync else hits

    # ------------------------------------------------------------------ primitive ops (tests)
    def gemm(self, A, W, bias=None, residual=None, act=N.ACT_NONE, out_f32=False):
        """A [B?,M,K], W [B?,N,K] in act dtype -> C; thin test hook over cir_gemm."""
        batched = A.dim() == 3
        A3 = A if batched else A[None]
        W3 = W if W.dim() == 3 else W[None]
        Bn, M, K = A3.shape
        Nn = W3.shape[1]
        assert A3.dtype == self.act_dtype and W3.dtype == self.act_dtype
        A3, W3 = A3.contiguous(), W3.contiguous()
        c_dtype = torch.float32 if (out_f32 or self.precision == "fp32") else self.act_dtype
        Cm = torch.empty(Bn, M, Nn, dtype=c_dtype, device=self.device)
        g = N.GemmArgs()
        g.A, g.W, g.C = N.ptr(A3), N.ptr(W3), N.ptr(Cm)
        if bias is not None:
            bias = bias.to(self.device, torch.float32).contiguous().view(Bn, Nn)
        g.bias = N.ptr(bias)
        if residual is not None:
            residual = residual.contiguous().view(Bn, M, Nn)
        g.residual = N.ptr(residual)
        g.M, g.N, g.K = M, Nn, K
        g.lda, g.ldw, g.ldc, g.ldres = K, K, Nn, Nn
        g.a_bstride, g.w_bstride, g.c_bstride, g.bias_bstride, g.res_bstride = M * K, Nn * K, M * Nn, Nn, M * Nn
        g.batch, g.act = Bn, act
        g.c_f32 = 1 if c_dtype == torch.float32 else 0
        g.res_f32 = 1 if (residual is not None and residual.dtype == torch.float32) else 0
        self._sync_stream()
        N.check(self._lib.cir_gemm(self.ctx, C.byref(g)), "cir_gemm")
        out = Cm if batched else Cm[0]
        return out

    def attention(self, q, k, v, key_mask=None, kv_index=None, scale=0.125, work=None, tiles=None):
        """q [B,Lq,H*64], k/v [Bk,Lk,H*64] act dtype -> o [B,Lq,H*64]; test hook over cir_attention."""
        B, Lq, HD = q.shape
        Lk = k.shape[1]
        q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
        o = torch.empty_like(q)
        a = N.AttnArgs()
        a.q, a.k, a.v, a.o = N.ptr(q), N.ptr(k), N.ptr(v), N.ptr(o)
        a.q_bs, a.q_rs, a.o_bs, a.o_rs = Lq * HD, HD, Lq * HD, HD
        a.k_bs, a.k_rs, a.v_bs, a.v_rs = Lk * HD, HD, Lk * HD, HD
        km = None if key_mask is None else self._i32(key_mask)
        ki = None if kv_index is None else self._i32(kv_index)
        a.key_mask, a.kv_index, a.mask_index = N.ptr(km), N.ptr(ki), N.vp(0)
        wk = None if work is None else self._i32(work)
        a.work, a.num_work = N.ptr(wk), (0 if wk is None else wk.shape[0])
        tl = None if tiles is None else self._i32(tiles)
        a.tiles, a.num_tiles, a.kv_batches = N.ptr(tl), (0 if tl is None else tl.shape[0]), k.shape[0]
        a.B, a.H, a.Lq, a.Lk, a.scale = B, HD // 64, Lq, Lk, scale
        self._sync_stream()
        N.check(self._lib.cir_attention(self.ctx, C.byref(a)), "cir_attention")
        return o

    def qkv_attention(self, x, w, bias=None, key_mask=None, mask_index=None, scale=0.125):
        """x [batch, captions, L, 768] bf16, w [batch, 2304, 768] bf16 (query | key | value rows), bias [batch, 2304] fp32,
        key_mask int [*, L] -> context [batch, captions, L, 768]; test hook over cir_qkv_attention."""
        nb, caps, L, HD = x.shape
        assert HD == HIDDEN and w.shape == (nb, 3 * HIDDEN, HIDDEN)
        x, w = x.contiguous(), w.contiguous()
        out = torch.empty_like(x)
        b = None if bias is None else bias.float().contiguous()
        km = None if key_mask is None else self._i32(key_mask)
        mi = None if mask_index is None else self._i32(mask_index)
        a = N.QkvAttnArgs()
        a.x, a.x_bs, a.w, a.bias = N.ptr(x), caps * L * HD, N.ptr(w), N.ptr(b)
        a.out, a.out_rs, a.out_bs = N.ptr(out), HD, caps * L * HD
        a.key_mask, a.mask_index = N.ptr(km), N.ptr(mi)
        a.captions, a.L, a.batch, a.scale = caps, L, nb, scale
        self._sync_stream()
        N.check(self._lib.cir_qkv_attention(self.ctx, C.byref(a)), "cir_qkv_attention")
        return out

    def add_layernorm(self, x, gamma, beta, res=None, x_rows=None, rows_per_group=None, eps=1e-12, out_f32=False):
        rows = (res.shape[0] if res is not None else x.shape[0])
        x = x.contiguous()
        y = torch.empty(rows, HIDDEN, dtype=torch.float32 if (out_f32 or self.precision == "fp32") else self.act_dtype, device=self.device)
        self._sync_stream()
        N.check(self._lib.cir_add_layernorm(
            self.ctx, N.ptr(x), 1 if x.dtype == torch.float32 else 0, x_rows or x.shape[0], N.ptr(res.contiguous() if res is not None else None),
            N.ptr(gamma.float().contiguous()), N.ptr(beta.float().contiguous()), rows_per_group or rows, N.ptr(y),
            1 if y.dtype == torch.float32 else 0, rows, eps), "cir_add_layernorm")
        return y


def _kv_weights_key(w) -> tuple:
    """The device pointers of the cross-attention K/V weights in a packed cir_stage2_weights: what a K/V cache depends on."""
    return tuple(int(p or 0) for p in w.cross_kv_w) + tuple(int(p or 0) for p in w.cross_kv_b)


class Stage2KVCache:
    """Resident cross-attention K/V gallery (``cir_stage2_kv_cache`` in include/cir_b200.h): the K0|V0|K1|V1 rows of all 12
    layers of gallery rows [row0, row0 + rows), computed once by :meth:`fill` and read by every scoring call that passes
    ``kv_cache=`` (``Engine.stage2_score_matrix``, ``BLIP_NLVR.score_triplets``, the validation drivers).  Those calls then skip the
    per-chunk token gather and K/V GEMMs (32.7 GF per candidate load) and return the same scores bit for bit.

    The cache remembers the packed weights it is filled with (``weights``; their blob must stay alive, as for any scoring call)
    and refuses to serve other weights.  ``blob``: optional caller-provided uint8 device tensor of at least ``nbytes``."""

    def __init__(self, eng: Engine, w, rows: int, num_tokens: int, row0: int = 0, blob: Optional[torch.Tensor] = None):
        self.eng, self.weights = eng, w
        self._key = _kv_weights_key(w)
        need = eng._lib.cir_stage2_kv_cache_bytes(eng.ctx, rows, num_tokens)
        self._blob = torch.empty(max(need, 256), dtype=torch.uint8, device=eng.device) if blob is None else blob
        if self._blob.device != eng.device or self._blob.dtype != torch.uint8:
            raise N.CirError(f"Stage2KVCache: the blob must be a uint8 tensor on {eng.device}")
        self._s = N.Stage2KVCache()
        N.check(eng._lib.cir_stage2_kv_cache_init(eng.ctx, N.ptr(self._blob), self._blob.numel(), row0, rows, num_tokens,
                                                  C.byref(self._s)), "cir_stage2_kv_cache_init")

    @property
    def row0(self) -> int:
        return int(self._s.row0)

    @property
    def rows(self) -> int:
        return int(self._s.rows)

    @property
    def num_tokens(self) -> int:
        return int(self._s.num_tokens)

    @property
    def nbytes(self) -> int:
        """Bytes of K/V the cache holds (12 layers x rows x N x 3072 activations)."""
        return int(self.eng._lib.cir_stage2_kv_cache_bytes(self.eng.ctx, self.rows, self.num_tokens))

    def layer(self, i: int) -> torch.Tensor:
        """View of layer i's K/V rows: act [rows * N, 3072] (K0 | V0 | K1 | V1 columns)."""
        n = self.rows * self.num_tokens * 4 * HIDDEN
        es = 2 if self.eng.act_dtype == torch.bfloat16 else 4
        return self._blob[i * n * es:(i + 1) * n * es].view(self.eng.act_dtype).view(self.rows * self.num_tokens, 4 * HIDDEN)

    def fill(self, tokens: torch.Tensor, first: Optional[int] = None) -> "Stage2KVCache":
        """Project gallery rows first .. first + n - 1 (``tokens`` act [n, N, 768]; ``first`` defaults to ``row0``) into the cache.
        Slices may come in any order and any size: the bytes of a row do not depend on them."""
        eng = self.eng
        first = self.row0 if first is None else int(first)
        if tokens.dim() != 3 or tokens.shape[1] != self.num_tokens or tokens.shape[2] != HIDDEN:
            raise N.CirError(f"Stage2KVCache.fill: tokens {tuple(tokens.shape)} are not [n, {self.num_tokens}, {HIDDEN}]")
        if tokens.dtype != eng.act_dtype or tokens.device != eng.device:
            raise N.CirError(f"Stage2KVCache.fill: tokens must be {eng.act_dtype} on {eng.device}")
        t = tokens.contiguous()
        eng._sync_stream()
        N.check(eng._lib.cir_stage2_kv_cache_fill(eng.ctx, C.byref(self.weights), C.byref(self._s), N.ptr(t), first, t.shape[0]),
                "cir_stage2_kv_cache_fill")
        return self

    def _check_use(self, eng: Engine, w, num_tokens: int) -> None:
        if eng.device != self.eng.device:
            raise N.CirError(f"Stage2KVCache lives on {self.eng.device}, the engine on {eng.device}")
        if _kv_weights_key(w) != self._key:
            raise N.CirError("Stage2KVCache was filled with other stage-II weights")
        if num_tokens != self.num_tokens:
            raise N.CirError(f"Stage2KVCache holds {self.num_tokens} tokens per image, the gallery has {num_tokens}")

    def _check_rows(self, lo: int, hi: int) -> None:
        if lo < self.row0 or hi >= self.row0 + self.rows:
            raise N.CirError(f"candidates [{lo}, {hi}] outside the K/V cache's rows [{self.row0}, {self.row0 + self.rows})")


ALL_TAGS = 0xFFFFFFFF


def tag_bits(tags) -> np.ndarray:
    """Row tags / query masks (a Python int, a sequence of ints or a numpy integer array, e.g. uint32) -> int32 bit patterns
    (0xFFFFFFFF -> -1), the form the device tensors keep.  Values outside [0, 2^32) raise ValueError."""
    a = np.asarray(tags)
    if a.dtype == object:            # ints beyond 64 bits
        raise ValueError("tags must lie in [0, 2^32)")
    if a.dtype == bool or not np.issubdtype(a.dtype, np.integer):
        raise TypeError(f"tags must be integers, got {a.dtype}")
    if a.size and (a.min() < 0 or a.max() > ALL_TAGS):
        raise ValueError(f"tags must lie in [0, 2^32), got [{a.min()}, {a.max()}]")
    return a.astype(np.uint32).view(np.int32)


class Stage1Index:
    """Resident stage-I gallery index (``cir_stage1_index`` in include/cir_b200.h): gallery embeddings fp32 [n,256] are copied
    and, in bf16 engines, converted to bf16 once, when they are added; every search reuses them.  ``topk`` returns exactly what
    :meth:`Engine.stage1_topk` returns over the same rows, bit for bit.

    Every row carries a 32-bit tag (all bits set unless given).  ``topk(..., tags=masks)`` searches, for query q, only the rows
    whose tag shares a bit with masks[q] (cir_stage1_index_topk_filtered); :meth:`remove` sets tags to 0, so removed rows are
    never returned.  Tags are kept as a device int32 tensor of uint32 bit patterns.

    ``topk`` never synchronises.  Given device tensors (q_emb fp32 contiguous, exclude and masks int32) and ``out=``, it allocates
    and uploads nothing once its workspace exists for that (Q, k) -- run it once before ``torch.cuda.graph`` capture.  A captured
    graph searches the rows the index had at capture time, with the tags and masks those tensors hold at replay.

    Row ids: every row keeps the id it was given when it was added (0, 1, 2, ... in the order of ``add``).  ``topk`` returns ids
    (plus ``col_offset``), ``exclude``, ``set_tags`` and ``remove`` take them.  :meth:`compact` drops the removed rows and
    :meth:`subset` copies the rows of some tags into a new index; both keep the ids, so they change speed and memory but no search
    result.  Until the first compaction the ids are the physical row numbers and the index keeps no id table."""

    def __init__(self, eng: Engine, capacity: int):
        self.eng = eng
        self._ws: Optional[torch.Tensor] = None
        self._retired: List[torch.Tensor] = []    # outgrown workspaces stay alive: a captured graph may still point at one
        self._ids: Optional[torch.Tensor] = None  # device int32 [capacity + 1] id per physical row, from the first compaction on
        self._ids_host: Optional[np.ndarray] = None   # host mirror of _ids[:rows] (checks host ids without a synchronisation)
        self._next_id = 0                         # rows ever added: the id of the next added row
        self._blob = torch.empty(max(1, eng._lib.cir_stage1_index_bytes(eng.ctx, capacity)), dtype=torch.uint8, device=eng.device)
        self._s = N.Stage1Index()
        # one spare slot past the capacity: set_tags with device ids sends the writes of ids that no row holds there
        self._tags = torch.full((capacity + 1,), -1, dtype=torch.int32, device=eng.device)
        eng._sync_stream()
        N.check(eng._lib.cir_stage1_index_init(eng.ctx, N.ptr(self._blob), self._blob.numel(), capacity, C.byref(self._s)),
                "cir_stage1_index_init")

    @property
    def capacity(self) -> int:
        return int(self._s.capacity)

    @property
    def rows(self) -> int:
        return int(self._s.rows)

    @property
    def g_f32(self) -> torch.Tensor:
        """fp32 [rows, 256] view of the indexed rows (the blob starts with them; no copy)."""
        n = self.rows
        return self._blob[: n * EMBED * 4].view(torch.float32).view(n, EMBED)

    @property
    def row_tags(self) -> torch.Tensor:
        """int32 [rows] tag bit patterns of the indexed rows (a view: change tags through :meth:`set_tags` / :meth:`remove`)."""
        return self._tags[: self.rows]

    @property
    def row_ids(self) -> torch.Tensor:
        """int32 [rows] id of each physical row, strictly increasing (a view after a compaction, ``arange(rows)`` before)."""
        if self._ids is None:
            return torch.arange(self.rows, dtype=torch.int32, device=self.eng.device)
        return self._ids[: self.rows]

    @property
    def next_id(self) -> int:
        """The id the next added row gets: the number of rows ever added (compactions do not lower it)."""
        return self._next_id

    def _tag_tensor(self, tags, n: int, what: str) -> torch.Tensor:
        """One int (broadcast), n values (see tag_bits) or an int32 tensor of n bit patterns -> contiguous device int32 [n]."""
        if isinstance(tags, torch.Tensor):
            if tags.dtype != torch.int32:
                raise TypeError(f"{what}: a tag tensor holds int32 bit patterns, got {tags.dtype}")
            if tags.dim() != 1 or tags.numel() != n:
                raise ValueError(f"{what}: expected {n} tags, got shape {tuple(tags.shape)}")
            return tags.to(self.eng.device).contiguous()
        bits = tag_bits(tags)
        if bits.ndim == 0:
            return torch.full((n,), int(bits), dtype=torch.int32, device=self.eng.device)
        if bits.shape != (n,):
            raise ValueError(f"{what}: expected {n} tags, got shape {bits.shape}")
        return torch.from_numpy(np.ascontiguousarray(bits)).to(self.eng.device)

    def add(self, g_emb: torch.Tensor, tags=None) -> "Stage1Index":
        """Append gallery rows fp32 [n,256] (host or device); only the new rows are converted.  ``tags``: the new rows' tags
        (one int or n values; default all bits set, so every non-zero mask sees them)."""
        g = g_emb.to(self.eng.device, torch.float32).contiguous()
        assert g.dim() == 2 and g.shape[1] == EMBED, g.shape
        n, r0 = g.shape[0], self.rows
        if self._next_id + n > 1 << 31:
            raise N.CirError(f"Stage1Index.add: ids {self._next_id}..{self._next_id + n - 1} do not fit int32")
        t = None if tags is None else self._tag_tensor(tags, n, "Stage1Index.add")
        self.eng._sync_stream()
        N.check(self.eng._lib.cir_stage1_index_add(self.eng.ctx, C.byref(self._s), N.ptr(g), n), "cir_stage1_index_add")
        if t is None:
            self._tags[r0:r0 + n].fill_(-1)
        else:
            self._tags[r0:r0 + n].copy_(t)
        if self._ids is not None:
            new = np.arange(self._next_id, self._next_id + n, dtype=np.int32)
            self._ids[r0:r0 + n].copy_(torch.from_numpy(new))
            self._ids_host = np.concatenate([self._ids_host, new])
        self._next_id += n
        return self

    def _rows_of(self, ids, what: str, missing_ok: bool) -> torch.Tensor:
        """Row ids -> device int64 physical rows.  Host ids outside [0, next_id) raise; host ids that no row holds any more (dropped
        by a compaction) raise unless ``missing_ok``, else they are left out.  Device ids are mapped on the device without a
        synchronisation; those no row holds go to the spare tag slot past the capacity, so they change no row."""
        if self._ids is None:                     # ids are physical rows
            if isinstance(ids, torch.Tensor) and ids.is_cuda:
                return ids.reshape(-1).long()
            r_np = np.asarray(ids, dtype=np.int64).reshape(-1)
            self.eng._check_range(r_np, self.rows, what)
            return torch.from_numpy(r_np).to(self.eng.device)
        n = self.rows
        if isinstance(ids, torch.Tensor) and ids.is_cuda:
            want = ids.reshape(-1).to(torch.int32)
            pos = torch.searchsorted(self._ids[:n], want)
            hit = self._ids[:n][pos.clamp(max=max(n - 1, 0))] == want if n else torch.zeros_like(want, dtype=torch.bool)
            return torch.where(hit & (pos < n), pos, torch.full_like(pos, self.capacity))
        i_np = np.asarray(ids, dtype=np.int64).reshape(-1)
        self.eng._check_range(i_np, self._next_id, what)
        pos = np.searchsorted(self._ids_host, i_np)
        hit = (pos < n) & (self._ids_host[np.minimum(pos, max(n - 1, 0))] == i_np) if n else np.zeros(i_np.shape, dtype=bool)
        if not hit.all():
            if not missing_ok:
                raise ValueError(f"{what}: ids {i_np[~hit][:8].tolist()} are no longer in the index (dropped by a compaction)")
            pos = pos[hit]
        return torch.from_numpy(pos.astype(np.int64)).to(self.eng.device)

    def set_tags(self, rows, tags) -> "Stage1Index":
        """Set the tags of indexed rows (row ids: a device int tensor, or host ints checked here) to one int or one value per row.
        An on-stream tensor write: with device tensors it can be captured in a CUDA graph.  After a compaction, host ids that no
        row holds any more raise ValueError, device ones are ignored."""
        r = self._rows_of(rows, "Stage1Index.set_tags rows", missing_ok=False)
        t = self._tag_tensor(tags, r.numel(), "Stage1Index.set_tags")
        self._tags.index_copy_(0, r, t)
        return self

    def remove(self, rows) -> "Stage1Index":
        """Remove indexed rows (row ids): their tags become 0, so no filtered search returns them (search with ``tags=ALL_TAGS``
        for everything not removed; ``tags=None`` ignores tags until :meth:`compact` drops them).  Ids stay; ``set_tags``
        restores a row that has not been compacted away.  Removing an id that a compaction already dropped does nothing."""
        r = self._rows_of(rows, "Stage1Index.remove rows", missing_ok=True)
        self._tags.index_fill_(0, r, 0)
        return self

    def _compact_into(self, dst: "Stage1Index", keep_mask: int, id_offset: int = 0) -> None:
        """cir_stage1_index_compact of this index into the empty index ``dst`` (rows with tag & keep_mask != 0, ids kept)."""
        eng = self.eng
        ids = self._ids
        if ids is None and id_offset:
            ids = torch.arange(id_offset, id_offset + self.rows, dtype=torch.int32, device=eng.device)
        dst._ids = torch.zeros(dst.capacity + 1, dtype=torch.int32, device=eng.device)
        ws = eng.workspace(eng._lib.cir_stage1_index_compact_workspace_bytes(eng.ctx, C.byref(self._s)))
        eng._sync_stream()
        N.check(eng._lib.cir_stage1_index_compact(eng.ctx, C.byref(self._s), N.ptr(self._tags), N.ptr(ids), int(keep_mask) & ALL_TAGS,
                                                  C.byref(dst._s), N.ptr(dst._tags), N.ptr(dst._ids), N.ptr(ws), ws.numel()),
                "cir_stage1_index_compact")
        dst._ids_host = dst._ids[: dst.rows].cpu().numpy()
        dst._next_id = self._next_id + id_offset

    def compact(self, capacity: Optional[int] = None) -> "Stage1Index":
        """Drop the removed rows (tag 0): the kept rows move, in their order, into a new blob of the same capacity (or of
        ``capacity``, e.g. to shrink the index), which replaces the old one; their bf16 copy and the gallery maxima are rebuilt
        from the kept rows.  Ids, tags and every filtered search result stay as they were; a search without tags no longer
        sees the removed rows.  Synchronises once.  While it runs the index takes two blobs of memory.  CUDA graphs captured
        before ``compact()`` point at the old blob and must be captured again."""
        return self._compact(capacity, 0)

    def _compact(self, capacity: Optional[int], id_offset: int) -> "Stage1Index":
        """:meth:`compact`; ``id_offset`` (first compaction only) is added to the row numbers that serve as ids until then."""
        assert id_offset == 0 or self._ids is None
        new = Stage1Index(self.eng, self.capacity if capacity is None else capacity)
        self._compact_into(new, ALL_TAGS, id_offset)
        self._blob, self._s, self._tags, self._ids = new._blob, new._s, new._tags, new._ids
        self._ids_host, self._next_id = new._ids_host, new._next_id
        return self

    def subset(self, mask, capacity: Optional[int] = None) -> "Stage1Index":
        """A new index of the rows whose tag shares a bit with ``mask``, in their order, with their ids and tags; this index is
        unchanged.  ``sub.topk(q, k, exclude=ex)`` equals ``self.topk(q, k, exclude=ex, tags=mask)`` bit for bit.  Capacity: this
        index's unless given (the subset can grow by ``add``; its new rows get ids from ``next_id`` on).  Synchronises once."""
        sub = Stage1Index(self.eng, self.capacity if capacity is None else capacity)
        self._compact_into(sub, int(tag_bits(mask)) & ALL_TAGS)
        return sub

    def topk(self, q_emb: torch.Tensor, k: int, exclude=None, col_offset: int = 0, out=None, exact_rows: Optional[torch.Tensor] = None,
             tags=None):
        """-> (dist fp32 [Q,k], idx int32 [Q,k]) of the k nearest indexed rows (global index = col_offset + row id), skipping
        exclude[q] (-1 = none).  ``out``: optional (dist, idx) to fill.  ``exact_rows``: optional int32 [Q] device tensor, set to 1
        for the queries whose list came from the exact fallback scan.  ``tags``: per-query masks [Q] (or one int for all queries):
        query q then ranks only the rows with (row tag & tags[q]) != 0 and pads a short list with (+inf, -1).  After a
        compaction the search maps ids on the device (cir_stage1_index_topk_ids); it still never synchronises."""
        eng = self.eng
        q = q_emb.to(eng.device, torch.float32).contiguous()
        Q = q.shape[0]
        if out is None:
            out = (torch.empty(Q, k, dtype=torch.float32, device=eng.device), torch.empty(Q, k, dtype=torch.int32, device=eng.device))
        td, ti = out
        assert td.shape == ti.shape == (Q, k) and td.dtype == torch.float32 and ti.dtype == torch.int32
        assert td.is_contiguous() and ti.is_contiguous()
        assert exact_rows is None or (exact_rows.dtype == torch.int32 and exact_rows.numel() == Q and exact_rows.is_contiguous())
        ex = None if exclude is None else eng._i32(exclude)
        masks = None if tags is None else self._tag_tensor(tags, Q, "Stage1Index.topk")
        ws_bytes = eng._lib.cir_stage1_index_topk_workspace_bytes if self._ids is None else eng._lib.cir_stage1_index_topk_ids_workspace_bytes
        need = ws_bytes(eng.ctx, C.byref(self._s), Q, k)
        if self._ws is None or self._ws.numel() < need:
            if self._ws is not None:
                self._retired.append(self._ws)
            self._ws = torch.empty(max(need, 256), dtype=torch.uint8, device=eng.device)
        eng._sync_stream()
        if self._ids is not None:
            N.check(eng._lib.cir_stage1_index_topk_ids(eng.ctx, C.byref(self._s), N.ptr(q), Q, N.ptr(self._ids), self._next_id,
                                                       N.ptr(None if masks is None else self._tags), N.ptr(masks), N.ptr(ex), col_offset,
                                                       k, N.ptr(td), N.ptr(ti), N.ptr(exact_rows), N.ptr(self._ws), self._ws.numel()),
                    "cir_stage1_index_topk_ids")
        elif masks is None:
            N.check(eng._lib.cir_stage1_index_topk(eng.ctx, C.byref(self._s), N.ptr(q), Q, N.ptr(ex), col_offset, k, N.ptr(td), N.ptr(ti),
                                                   N.ptr(exact_rows), N.ptr(self._ws), self._ws.numel()), "cir_stage1_index_topk")
        else:
            N.check(eng._lib.cir_stage1_index_topk_filtered(eng.ctx, C.byref(self._s), N.ptr(q), Q, N.ptr(self._tags), N.ptr(masks),
                                                            N.ptr(ex), col_offset, k, N.ptr(td), N.ptr(ti), N.ptr(exact_rows),
                                                            N.ptr(self._ws), self._ws.numel()), "cir_stage1_index_topk_filtered")
        return td, ti


_engines: Dict[Tuple[int, str], Engine] = {}


def get_engine(device=None, precision: str = "bf16") -> Engine:
    """Process-wide engine cache (one per device and precision)."""
    if not torch.cuda.is_available():
        raise N.CirError("no CUDA device: the B200 path has no CPU fallback")
    idx = None if device is None else torch.device(device).index       # index 0 is a valid explicit choice
    if idx is None:
        idx = torch.cuda.current_device()
    key = (idx, precision)
    if key not in _engines:
        _engines[key] = Engine(torch.device("cuda", idx), precision)
    return _engines[key]
