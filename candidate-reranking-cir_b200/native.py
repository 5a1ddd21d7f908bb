"""ctypes binding of ``csrc/libcir_b200.so`` (the C-ABI in ``include/cir_b200.h``).

There is NO fallback: if the library is missing or a call fails, a ``CirError`` is raised.
Only raw device pointers / sizes cross the boundary; torch is used by the callers for device
memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CIR_B200_LIB") or os.path.join(HERE, "csrc", "libcir_b200.so")   # override: A/B of kernel builds

DTYPE_F32, DTYPE_BF16 = 0, 1
KV_MXFP8 = 2                  # cir_stage2_kv_cache.dtype of an MXFP8 K/V cache
GEMM_AUTO, GEMM_SIMT, GEMM_TCGEN05, GEMM_TCGEN05_1CTA = 0, 1, 2, 3
ACT_NONE, ACT_GELU, ACT_RELU = 0, 1, 2
PROF_GEMM, PROF_ATTN_TC, PROF_ATTN_SELF, PROF_LAYERNORM, PROF_QKV_ATTN = 0, 1, 2, 3, 4
LAYERS = 12

vp = C.c_void_p
i64 = C.c_int64
i32 = C.c_int32


class CirError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [("A", vp), ("W", vp), ("C", vp), ("bias", vp), ("residual", vp),
                ("M", i64), ("N", i64), ("K", i64),
                ("lda", i64), ("ldw", i64), ("ldc", i64), ("ldres", i64),
                ("a_bstride", i64), ("w_bstride", i64), ("c_bstride", i64), ("bias_bstride", i64), ("res_bstride", i64),
                ("batch", i32), ("act", i32), ("c_f32", i32), ("res_f32", i32)]


class AttnArgs(C.Structure):
    _fields_ = [("q", vp), ("k", vp), ("v", vp), ("o", vp),
                ("q_bs", i64), ("q_rs", i64), ("k_bs", i64), ("k_rs", i64),
                ("v_bs", i64), ("v_rs", i64), ("o_bs", i64), ("o_rs", i64),
                ("kv_index", vp), ("key_mask", vp), ("mask_index", vp), ("work", vp), ("num_work", i32),
                ("tiles", vp), ("num_tiles", i32), ("kv_batches", i32),
                ("B", i32), ("H", i32), ("Lq", i32), ("Lk", i32), ("scale", C.c_float)]


class QkvAttnArgs(C.Structure):
    _fields_ = [("x", vp), ("x_bs", i64), ("w", vp), ("bias", vp), ("out", vp), ("out_rs", i64), ("out_bs", i64),
                ("key_mask", vp), ("mask_index", vp), ("captions", i64), ("L", i32), ("batch", i32), ("scale", C.c_float)]


class Stage1Index(C.Structure):
    _fields_ = [("capacity", i64), ("rows", i64), ("g_f32", vp), ("g_bf16", vp), ("gmax", vp)]


class Stage2KVCache(C.Structure):
    _fields_ = [("row0", i64), ("rows", i64), ("num_tokens", i64), ("dtype", i32), ("kv", vp)]


_A = vp * LAYERS


class VitWeights(C.Structure):
    _fields_ = [("patch_w", vp), ("patch_b", vp), ("cls_token", vp), ("pos_embed", vp),
                ("norm1_g", _A), ("norm1_b", _A), ("qkv_w", _A), ("qkv_b", _A), ("proj_w", _A), ("proj_b", _A),
                ("norm2_g", _A), ("norm2_b", _A), ("fc1_w", _A), ("fc1_b", _A), ("fc2_w", _A), ("fc2_b", _A),
                ("norm_g", vp), ("norm_b", vp)]


class Stage1Weights(C.Structure):
    _fields_ = [("word_emb", vp), ("pos_emb", vp), ("emb_ln_g", vp), ("emb_ln_b", vp),
                ("self_qkv_w", _A), ("self_qkv_b", _A), ("self_out_w", _A), ("self_out_b", _A),
                ("self_ln_g", _A), ("self_ln_b", _A), ("cross_q_w", _A), ("cross_q_b", _A),
                ("cross_kv_w", _A), ("cross_kv_b", _A), ("cross_out_w", _A), ("cross_out_b", _A),
                ("cross_ln_g", _A), ("cross_ln_b", _A), ("ffn1_w", _A), ("ffn1_b", _A),
                ("ffn2_w", _A), ("ffn2_b", _A), ("ffn_ln_g", _A), ("ffn_ln_b", _A),
                ("text_proj_w", vp), ("text_proj_b", vp), ("vision_proj_w", vp), ("vision_proj_b", vp)]


_A2 = _A * 2


class VitState(C.Structure):
    _fields_ = [("patch_w", vp), ("patch_b", vp), ("cls_token", vp), ("pos_embed", vp), ("num_tokens", i64),
                ("norm1_g", _A), ("norm1_b", _A), ("qkv_w", _A), ("qkv_b", _A), ("proj_w", _A), ("proj_b", _A),
                ("norm2_g", _A), ("norm2_b", _A), ("fc1_w", _A), ("fc1_b", _A), ("fc2_w", _A), ("fc2_b", _A),
                ("norm_g", vp), ("norm_b", vp)]


class TextEmbedState(C.Structure):
    _fields_ = [("word_emb", vp), ("vocab_rows", i64), ("pos_emb", vp), ("pos_rows", i64), ("ln_g", vp), ("ln_b", vp)]


class Stage1State(C.Structure):
    _fields_ = [("emb", TextEmbedState)] + [(n, _A) for n in (
        "self_q_w", "self_q_b", "self_k_w", "self_k_b", "self_v_w", "self_v_b", "self_out_w", "self_out_b", "self_ln_g", "self_ln_b",
        "cross_q_w", "cross_q_b", "cross_k_w", "cross_k_b", "cross_v_w", "cross_v_b", "cross_out_w", "cross_out_b", "cross_ln_g", "cross_ln_b",
        "ffn1_w", "ffn1_b", "ffn2_w", "ffn2_b", "ffn_ln_g", "ffn_ln_b")] + [
        ("text_proj_w", vp), ("text_proj_b", vp), ("vision_proj_w", vp), ("vision_proj_b", vp)]


class Stage2State(C.Structure):
    _fields_ = [("emb", TextEmbedState)] + [(n, _A2) for n in (
        "self_q_w", "self_q_b", "self_k_w", "self_k_b", "self_v_w", "self_v_b", "self_out_w", "self_out_b", "self_ln_g", "self_ln_b",
        "cross_q_w", "cross_q_b", "cross_k_w", "cross_k_b", "cross_v_w", "cross_v_b", "cross_out_w", "cross_out_b")] + [
        ("merge_w", _A), ("merge_b", _A), ("cross_ln_g", _A2), ("cross_ln_b", _A2),
        ("ffn1_w", _A), ("ffn1_b", _A), ("ffn2_w", _A), ("ffn2_b", _A), ("ffn_ln_g", _A), ("ffn_ln_b", _A),
        ("cls0_w", vp), ("cls0_b", vp), ("cls2_w", vp), ("cls2_b", vp)]


class Stage2Weights(C.Structure):
    _fields_ = [("word_emb", vp), ("pos_emb", vp), ("emb_ln_g", vp), ("emb_ln_b", vp),
                ("self_qkv_w", _A), ("self_qkv_b", _A), ("self_out_w", _A), ("self_out_b", _A),
                ("self_ln_g", _A), ("self_ln_b", _A), ("cross_q_w", _A), ("cross_q_b", _A),
                ("cross_kv_w", _A), ("cross_kv_b", _A), ("cross_out_w", _A), ("cross_out_b", _A),
                ("cross_ln_g", _A), ("cross_ln_b", _A), ("ffn1_w", _A), ("ffn1_b", _A),
                ("ffn2_w", _A), ("ffn2_b", _A), ("ffn_ln_g", _A), ("ffn_ln_b", _A),
                ("cls0_w", vp), ("cls0_b", vp), ("cls2_w", vp), ("cls2_b", vp)]


_SIGS = {
    "cir_last_error": (C.c_char_p, []),
    "cir_version": (C.c_int, []),
    "cir_create": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int]),
    "cir_destroy": (C.c_int, [vp]),
    "cir_set_stream": (C.c_int, [vp, vp]),
    "cir_set_gemm_impl": (C.c_int, [vp, C.c_int]),
    "cir_set_attention_impl": (C.c_int, [vp, C.c_int]),
    "cir_set_prune_last_layer": (C.c_int, [vp, C.c_int]),
    "cir_set_dedup_first_layer": (C.c_int, [vp, C.c_int]),
    "cir_set_fuse_qkv_attention": (C.c_int, [vp, C.c_int]),
    "cir_set_stage1_tensor_cores": (C.c_int, [vp, C.c_int]),
    "cir_set_gemm_tma_store": (C.c_int, [vp, C.c_int]),
    "cir_get_dtype": (C.c_int, [vp]),
    "cir_launch_count": (i64, [vp, C.c_int]),
    "cir_profile_gemm": (C.c_int, [vp, C.c_int]),
    "cir_profile_read": (C.c_int, [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(i64)]),
    "cir_profile_gemm_read": (C.c_int, [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(i64)]),
    "cir_gemm": (C.c_int, [vp, C.POINTER(GemmArgs)]),
    "cir_add_layernorm": (C.c_int, [vp, vp, C.c_int, i64, vp, vp, vp, i64, vp, C.c_int, i64, C.c_float]),
    "cir_attention": (C.c_int, [vp, C.POINTER(AttnArgs)]),
    "cir_pack_vit_bytes": (C.c_size_t, [vp, i64]),
    "cir_pack_vit_weights": (C.c_int, [vp, C.POINTER(VitState), vp, C.c_size_t, C.POINTER(VitWeights)]),
    "cir_pack_stage1_bytes": (C.c_size_t, [vp, i64, i64]),
    "cir_pack_stage1_weights": (C.c_int, [vp, C.POINTER(Stage1State), vp, C.c_size_t, C.POINTER(Stage1Weights)]),
    "cir_pack_stage2_bytes": (C.c_size_t, [vp, i64, i64]),
    "cir_pack_stage2_weights": (C.c_int, [vp, C.POINTER(Stage2State), vp, C.c_size_t, C.POINTER(Stage2Weights)]),
    "cir_qkv_attention": (C.c_int, [vp, C.POINTER(QkvAttnArgs)]),
    "cir_bert_embeddings": (C.c_int, [vp, vp, i64, i64, vp, vp, vp, vp, vp]),
    "cir_gather_rows": (C.c_int, [vp, vp, vp, vp, i64, i64]),
    "cir_cast_f32_to_act": (C.c_int, [vp, vp, vp, i64]),
    "cir_cast_act_to_f32": (C.c_int, [vp, vp, vp, i64]),
    "cir_l2_normalize": (C.c_int, [vp, vp, vp, i64, i64]),
    "cir_rerank_sort": (C.c_int, [vp, vp, i64, i64, vp]),
    "cir_topk_from_dist": (C.c_int, [vp, vp, i64, i64, i64, vp, i64, i64, vp, vp, vp, C.c_size_t]),
    "cir_topk_workspace_bytes": (C.c_size_t, [i64, i64, i64]),
    "cir_stage1_topk": (C.c_int, [vp, vp, vp, i64, i64, vp, i64, i64, vp, vp, vp, C.c_size_t]),
    "cir_stage1_topk_workspace_bytes": (C.c_size_t, [i64, i64, i64]),
    "cir_stage1_index_bytes": (C.c_size_t, [vp, i64]),
    "cir_stage1_index_init": (C.c_int, [vp, vp, C.c_size_t, i64, C.POINTER(Stage1Index)]),
    "cir_stage1_index_add": (C.c_int, [vp, C.POINTER(Stage1Index), vp, i64]),
    "cir_stage1_index_topk_workspace_bytes": (C.c_size_t, [vp, C.POINTER(Stage1Index), i64, i64]),
    "cir_stage1_index_topk": (C.c_int, [vp, C.POINTER(Stage1Index), vp, i64, vp, i64, i64, vp, vp, vp, vp, C.c_size_t]),
    "cir_stage1_index_topk_filtered": (C.c_int, [vp, C.POINTER(Stage1Index), vp, i64, vp, vp, vp, i64, i64, vp, vp, vp, vp, C.c_size_t]),
    "cir_stage1_index_compact_workspace_bytes": (C.c_size_t, [vp, C.POINTER(Stage1Index)]),
    "cir_stage1_index_compact": (C.c_int, [vp, C.POINTER(Stage1Index), vp, vp, C.c_uint32, C.POINTER(Stage1Index), vp, vp, vp, C.c_size_t]),
    "cir_stage1_index_topk_ids_workspace_bytes": (C.c_size_t, [vp, C.POINTER(Stage1Index), i64, i64]),
    "cir_stage1_index_topk_ids": (C.c_int, [vp, C.POINTER(Stage1Index), vp, i64, vp, i64, vp, vp, vp, i64, i64, vp, vp, vp, vp, C.c_size_t]),
    "cir_stage1_logits": (C.c_int, [vp, vp, vp, i64, i64, C.c_float, vp]),
    "cir_stage1_rank_members": (C.c_int, [vp, vp, vp, vp, i64, i64, vp, vp]),
    "cir_topk_merge": (C.c_int, [vp, vp, vp, i64, i64, i64, vp, vp, vp, C.c_size_t]),
    "cir_recall_counts": (C.c_int, [vp, vp, vp, i64, i64, C.POINTER(i32), i32, vp]),
    "cir_vit_workspace_bytes": (C.c_size_t, [vp, i64, i64]),
    "cir_vit_forward": (C.c_int, [vp, C.POINTER(VitWeights), vp, i64, i64, vp, vp, C.c_size_t]),
    "cir_stage1_workspace_bytes": (C.c_size_t, [vp, i64, i64, i64]),
    "cir_stage1_encode": (C.c_int, [vp, C.POINTER(Stage1Weights), vp, vp, vp, vp, i64, i64, i64, vp, vp, C.c_int, vp, C.c_size_t]),
    "cir_stage1_gallery_embed": (C.c_int, [vp, C.POINTER(Stage1Weights), vp, i64, i64, vp, vp, C.c_size_t]),
    "cir_stage2_workspace_bytes": (C.c_size_t, [vp, i64, i64, i64, i64, i64]),
    "cir_stage2_score": (C.c_int, [vp, C.POINTER(Stage2Weights), vp, vp, i64, vp, vp, vp, i64, i64, i64, vp, vp, i64, vp, i64, vp, i64, vp, i64, vp, vp, vp, C.c_size_t]),
    "cir_stage2_prefix_workspace_bytes": (C.c_size_t, [vp, i64, i64]),
    "cir_stage2_prefix": (C.c_int, [vp, C.POINTER(Stage2Weights), vp, vp, vp, i64, i64, vp, vp, vp, C.c_size_t]),
    "cir_stage2_score_prefixed": (C.c_int, [vp, C.POINTER(Stage2Weights), vp, vp, i64, vp, vp, vp, i64, i64, i64, vp, vp, i64, vp, i64, vp, i64, vp, i64, vp, vp, vp, C.c_size_t]),
    "cir_stage2_kv_cache_bytes": (C.c_size_t, [vp, i64, i64]),
    "cir_stage2_kv_cache_init": (C.c_int, [vp, vp, C.c_size_t, i64, i64, i64, C.POINTER(Stage2KVCache)]),
    "cir_stage2_kv_cache_fill": (C.c_int, [vp, C.POINTER(Stage2Weights), C.POINTER(Stage2KVCache), vp, i64, i64]),
    "cir_stage2_score_cached_workspace_bytes": (C.c_size_t, [vp, i64, i64, i64, i64]),
    "cir_stage2_score_cached": (C.c_int, [vp, C.POINTER(Stage2Weights), C.POINTER(Stage2KVCache), vp, i64, vp, vp, vp, vp, vp, i64, i64,
                                          vp, vp, i64, vp, i64, vp, i64, vp, i64, vp, vp, vp, C.c_size_t]),
    "cir_stage2_kv_cache_bytes_mxfp8": (C.c_size_t, [vp, i64, i64]),
    "cir_stage2_kv_cache_init_mxfp8": (C.c_int, [vp, vp, C.c_size_t, i64, i64, i64, C.POINTER(Stage2KVCache)]),
    "cir_stage2_kv_cache_fill_mxfp8_workspace_bytes": (C.c_size_t, [vp, C.POINTER(Stage2KVCache), i64]),
    "cir_stage2_kv_cache_fill_mxfp8": (C.c_int, [vp, C.POINTER(Stage2Weights), C.POINTER(Stage2KVCache), vp, i64, i64, vp, C.c_size_t]),
    "cir_stage2_kv_score_workspace_bytes": (C.c_size_t, [vp, C.POINTER(Stage2KVCache), i64, i64, i64, i64]),
    "cir_stage2_kv_rerank_workspace_bytes": (C.c_size_t, [vp, C.POINTER(Stage2KVCache), i64, i64, i64]),
    "cir_stage2_plan_topk": (C.c_int, [vp, vp, i64, i64, i64, i64, i64, vp, vp, vp, vp, vp, vp]),
    "cir_stage2_rerank_cached_workspace_bytes": (C.c_size_t, [vp, i64, i64, i64, i64]),
    "cir_stage2_rerank_cached": (C.c_int, [vp, C.POINTER(Stage2Weights), C.POINTER(Stage2KVCache), vp, i64, i64, vp, vp, vp, i64,
                                           vp, vp, vp, vp, vp, C.c_size_t]),
}

_lib = None


def lib():
    """dlopen the CUDA library (once).  Raises CirError when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CirError(f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` "
                           "(nvcc, sm_100a). There is no CPU/PyTorch fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def exported_symbols():
    return sorted(_SIGS)


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().cir_last_error()
        raise CirError(f"{what or 'cir call'} failed (rc={rc}): {msg.decode() if msg else ''}")


def ptr(t):
    """torch tensor (or None) -> c_void_p of its device pointer."""
    if t is None:
        return vp(0)
    return vp(t.data_ptr())
