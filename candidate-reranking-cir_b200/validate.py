"""Stage-I evaluation / candidate-filtering drivers (reference: src/validate.py:33-99,176-268 and
src/utils.py:25-72).  The reference materialises ``1 - q @ G.T`` and fully argsorts it on the
device, then maps names and removes the reference image on the host (src/validate.py:202-210);
here the similarity tiles and the per-query top-K (with the reference index excluded in-kernel)
are fused, so nothing of size [Q, G] is ever stored.  The CIRR ``group_labels`` the reference obtains
by masking the full ranking (src/validate.py:213-218) come from ranking the five group members directly
(``cir_stage1_rank_members``)."""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from .topk_file import save_topk
from .validate_stage2 import LENGTH_BUCKET, _fiq_captions, _length_buckets, _name_index, _percent, _tokens

INDEX_BATCH = 16          # src/utils.py:33 (DataLoader batch_size=16)


def extract_index_features(dataset, blip_model, blip_stage2=False, blip_stage1=False):
    """src/utils.py:25-72.  ``dataset`` is a 'classic'-mode dataset: ``len(dataset)`` items, ``dataset[i]`` ->
    ``(image_name, image [3,S,S] float tensor)`` (src/data_utils.py 'classic' mode).  Images go through the ViT in
    batches of 16 like the reference's DataLoader.
    blip_stage2 -> (index_features [G,577,768], index_names);
    blip_stage1 -> (index_features, pooled+normalised [G,256], index_names).
    Features come back in the engine's activation dtype (bf16 in production mode, fp32 in the check mode)."""
    if blip_stage2:
        assert not blip_stage1, ValueError("only one condition shall be selected")      # src/utils.py:44
    elif blip_stage1:
        assert not blip_stage2, ValueError("only one condition shall be selected")      # src/utils.py:57
    else:
        raise RuntimeError                                                               # src/utils.py:71-72
    eng = blip_model.engine
    G = len(dataset)
    index_names: List[str] = []
    feats = None
    pooled = torch.empty(G, 256, dtype=torch.float32, device=eng.device) if blip_stage1 else None
    for g0 in range(0, G, INDEX_BATCH):
        items = [dataset[i] for i in range(g0, min(g0 + INDEX_BATCH, G))]
        names, images = zip(*items)
        images = torch.stack([torch.as_tensor(im) for im in images])
        if blip_stage2:
            batch_features = blip_model.img_embed(images)                               # src/utils.py:51
        else:
            batch_features, batch_pooled = blip_model.img_embed(images, return_pool_and_normalized=True)   # :65
            pooled[g0:g0 + len(names)] = batch_pooled
        if feats is None:
            feats = torch.empty((G,) + tuple(batch_features.shape[1:]), dtype=batch_features.dtype, device=eng.device)
        feats[g0:g0 + len(names)] = batch_features
        index_names.extend(names)
    if feats is None:
        feats = torch.empty(0, 577, 768, dtype=eng.act_dtype, device=eng.device)
    return (feats, index_names) if blip_stage2 else (feats, pooled, index_names)


def query_embeddings(blip_model, dataset, index_features, index_names, cirr: bool):
    """src/validate.py:305-311 (CIRR: the query embedding is L2-normalised twice) / :140-146 (Fashion-IQ: once).
    -> (q_emb fp32 [Q,256] on device, ref_idx int32 numpy [Q])."""
    eng = blip_model.engine
    n2i = _name_index(index_names)
    ref_idx = np.array([n2i[n] for n in dataset.reference_names], dtype=np.int32)
    caps = list(dataset.captions) if cirr else _fiq_captions(dataset.captions)
    ids, mask = _tokens(blip_model, dataset, caps)
    gallery = eng.to_act(index_features)
    q_emb = torch.empty(len(ref_idx), 256, dtype=torch.float32, device=eng.device)
    for rows, L in _length_buckets(mask, LENGTH_BUCKET):                            # each query at (about) its own length
        r_t = torch.from_numpy(rows).to(eng.device)
        _, qe = blip_model.encode_queries(gallery, ref_idx[rows], ids[r_t, :L].contiguous(), mask[r_t, :L].contiguous(),
                                          want_z=False, want_emb=True, normalize_twice=cirr)
        q_emb[r_t] = qe
    return q_emb, ref_idx


def _stage1_search(eng, q_emb, g_emb, k, exclude, index):
    """top-k of the gallery rows: through the resident ``index`` (engine.Stage1Index) when given, else over ``g_emb``."""
    if index is not None:
        return index.topk(q_emb, k, exclude=exclude)
    return eng.stage1_topk(q_emb, g_emb, k, exclude=exclude)


def _gallery(index_features_normed_pooled, index_names, index):
    """fp32 gallery embeddings ("already normed", :55,:199): the index's own rows when an index is given."""
    if index is None:
        return index_features_normed_pooled.float()
    assert index.rows == len(index_names), f"stage-I index holds {index.rows} rows, the gallery has {len(index_names)} names"
    return index.g_f32


def retrieve_topk(blip_model, dataset, index_features, index_features_normed_pooled, index_names, k: int, cirr: bool,
                  return_embeddings: bool = False, index=None):
    """Query embeddings + fused distance/top-K (src/validate.py:57-58,202-210,257).  Returns (top_dist fp32 [Q,k],
    top_idx int32 [Q,k]) on device; CIRR excludes each query's own reference image.  ``index``: an engine.Stage1Index built
    from ``index_features_normed_pooled`` (which may then be None) -- same results, without per-call gallery conversion."""
    eng = blip_model.engine
    q_emb, ref_idx = query_embeddings(blip_model, dataset, index_features, index_names, cirr)
    g_emb = _gallery(index_features_normed_pooled, index_names, index)
    td, ti = _stage1_search(eng, q_emb, g_emb, k, ref_idx if cirr else None, index)
    return (td, ti, q_emb, g_emb, ref_idx) if return_embeddings else (td, ti)


def _labels_and_recalls(eng, top_idx, target_idx, ks):
    labels = top_idx.to(torch.int64) == torch.as_tensor(target_idx, device=top_idx.device)[:, None]
    ident = torch.arange(top_idx.shape[1], dtype=torch.int32, device=top_idx.device).expand_as(top_idx).contiguous()
    hits = eng.recall_counts(labels, ident, ks)
    return labels, [_percent(h, len(labels)) for h in hits]


def _names_of(index_names, top_idx: torch.Tensor) -> np.ndarray:
    idx = top_idx.cpu().numpy()
    assert (idx >= 0).all(), "top-K list has empty slots (K larger than the gallery?)"   # -1 would wrap to the last name
    return np.array(index_names)[idx]


def fiq_val_topk(relative_val_dataset, blip_model, index_features, index_features_normed_pooled, index_names, k: int = 100, index=None):
    """-> ((recall@10, recall@50), top-K dict shaped like the file written at src/validate.py:87-94).  ``index``: see retrieve_topk."""
    eng = blip_model.engine
    k = min(max(k, 50), len(index_names))
    _, top_idx = retrieve_topk(blip_model, relative_val_dataset, index_features, index_features_normed_pooled, index_names, k, cirr=False,
                               index=index)
    n2i = _name_index(index_names)
    tgt = np.array([n2i[n] for n in relative_val_dataset.target_names])
    labels, (r10, r50) = _labels_and_recalls(eng, top_idx, tgt, (10, 50))
    topk = {"sorted_index_names": _names_of(index_names, top_idx), "target_names": list(relative_val_dataset.target_names),
            "index_names": list(index_names), "labels": labels.cpu(), "split": relative_val_dataset.split,
            "dress_types": ",".join(relative_val_dataset.dress_types)}
    return (r10, r50), topk


def cirr_topk_from_embeddings(eng, q_emb, g_emb, ref_idx, target_idx, group_idx_noref, k: int, index=None):
    """The index arithmetic of src/validate.py:202-226 on the GPU, from query / gallery embeddings:
    top-k gallery rows per query without the reference (ascending distance), labels, and ``group_labels`` [Q,5] = the labels
    of the group members in stage-I ranking order (``labels[group_mask]``, :213-218).  ``index``: an engine.Stage1Index of
    the gallery, searched instead of ``g_emb`` (which may then be None).
    -> (top_idx int32 [Q,k], labels bool [Q,k], group_labels bool [Q,P], group_order int32 [Q,P]) on device."""
    ref_idx = np.asarray(ref_idx, dtype=np.int32)
    if index is not None:
        g_emb = index.g_f32
    _, top_idx = _stage1_search(eng, q_emb, g_emb, k, ref_idx, index)
    tgt = torch.as_tensor(np.asarray(target_idx), device=eng.device)
    labels = top_idx.to(torch.int64) == tgt[:, None]
    members = torch.as_tensor(np.asarray(group_idx_noref), dtype=torch.int64)
    _, gorder = eng.stage1_rank_members(q_emb, g_emb, members.numpy())
    ranked_members = torch.gather(members.to(eng.device), 1, gorder.to(torch.int64))
    group_labels = ranked_members == tgt[:, None]
    return top_idx, labels, group_labels, gorder


def cirr_val_topk(relative_val_dataset, blip_model, index_features, index_features_normed_pooled, index_names, k: int = 50, index=None):
    """-> ((group_recall@1,2,3, recall@1,5,10,50), top-K dict shaped like the file written at src/validate.py:256-263,
    including ``group_labels``, which the reference's CIRR reader requires: src/data_utils.py:301).  ``index``: see retrieve_topk."""
    ds = relative_val_dataset
    eng = blip_model.engine
    k = min(max(k, 50), len(index_names) - 1)          # the reference image is removed from every row (:207-210)
    q_emb, ref_idx = query_embeddings(blip_model, ds, index_features, index_names, cirr=True)
    g_emb = _gallery(index_features_normed_pooled, index_names, index)
    n2i = _name_index(index_names)
    tgt = np.array([n2i[n] for n in ds.target_names])
    gm = np.asarray(ds.group_members)
    refs = np.asarray(ds.reference_names)
    group_noref = [[n2i[m] for m in row if m != r] for row, r in zip(gm.tolist(), refs.tolist())]   # the reference never matches (:214)
    assert all(len(g) == len(group_noref[0]) for g in group_noref), "every img_set must have the same number of members"
    top_idx, labels, group_labels, _ = cirr_topk_from_embeddings(eng, q_emb, g_emb, ref_idx, tgt, group_noref, k, index=index)
    Q = len(tgt)
    if k == len(index_names) - 1:                       # the reference asserts on the FULL ranking (:221-222)
        assert torch.equal(labels.sum(-1).int().cpu(), torch.ones(Q).int())
    assert torch.equal(group_labels.sum(-1).int().cpu(), torch.ones(Q).int())
    ident = torch.arange(k, dtype=torch.int32, device=eng.device).expand(Q, k).contiguous()
    r1, r5, r10, r50 = [_percent(h, Q) for h in eng.recall_counts(labels, ident, (1, 5, 10, 50))]
    P = group_labels.shape[1]
    gident = torch.arange(P, dtype=torch.int32, device=eng.device).expand(Q, P).contiguous()
    g1, g2, g3 = [_percent(h, Q) for h in eng.recall_counts(group_labels, gident, (1, 2, 3))]
    topk = {"sorted_index_names": _names_of(index_names, top_idx), "target_names": list(ds.target_names),
            "index_names": list(index_names), "labels": labels.cpu(), "group_labels": group_labels.cpu(), "split": ds.split}
    return (g1, g2, g3, r1, r5, r10, r50), topk


def compute_fiq_val_metrics(relative_val_dataset, blip_model, index_features, index_features_normed_pooled, index_names,
                            k: int = 100, save_topk_path: Optional[str] = None, index=None) -> Tuple[float, float]:
    """src/validate.py:33-99 -> (recall@10, recall@50).  ``save_topk_path`` plays the role of the reference's SAVE_TOPK /
    K_VALUE globals (:82-97): the top-``k`` file is written there.  ``index``: see retrieve_topk."""
    metrics, topk = fiq_val_topk(relative_val_dataset, blip_model, index_features, index_features_normed_pooled, index_names, k, index=index)
    if save_topk_path:
        save_topk(save_topk_path, topk)
    return metrics


def compute_cirr_val_metrics(relative_val_dataset, blip_model, index_features, index_features_normed_pooled, index_names,
                             k: int = 50, save_topk_path: Optional[str] = None,
                             index=None) -> Tuple[float, float, float, float, float, float, float]:
    """src/validate.py:176-268 -> (group_recall@1, @2, @3, recall@1, @5, @10, @50), the reference's order (:268).
    ``index``: see retrieve_topk."""
    metrics, topk = cirr_val_topk(relative_val_dataset, blip_model, index_features, index_features_normed_pooled, index_names, k,
                                  index=index)
    if save_topk_path:
        save_topk(save_topk_path, topk)
    return metrics
