"""Stage-II evaluation drivers with the reference's function surface (src/validate_stage2.py:33-298),
restructured for the GPU: instead of a Python loop issuing one query at a time
(src/validate_stage2.py:94-125,235-275) all queries' z_t are computed in batches, all Q*K triplets
are scored candidate-major, and the re-sort + recall counting run as kernels."""
from __future__ import annotations

from typing import List, Tuple

import numpy as np
import torch

from .blip import tokenize
from .engine import NEG_FILL


def _name_index(index_names):
    return {n: i for i, n in enumerate(index_names)}


def _names_to_rows(index_names, n2i, names) -> np.ndarray:
    """[Q,K] array of image names -> gallery rows (the reference does this with per-query itemgetter lookups,
    src/validate_stage2.py:111-116,251); one hash join for the whole matrix."""
    names = np.asarray(names)
    try:
        import pandas as pd
        rows = pd.Index(index_names).get_indexer(names.reshape(-1))
        if (rows < 0).any():
            raise KeyError(str(names.reshape(-1)[np.flatnonzero(rows < 0)[0]]))
        return rows.astype(np.int32).reshape(names.shape)
    except ImportError:                                           # pragma: no cover
        return np.vectorize(n2i.__getitem__, otypes=[np.int32])(names)


def _names_to_rows_sharded(eng, index_names, n2i, names) -> np.ndarray:
    """The name -> gallery-row join of a [Q,K] name matrix.  Under torch.distributed every rank joins its block of query rows and the
    int32 blocks are all-gathered (the join is the largest host-side item of a step: ~25 ms for 200 k names)."""
    from .distributed import all_gather_rows, world
    from .schedule import shard_rows
    names = np.asarray(names)
    rank, ws = world()
    if ws == 1 or names.shape[0] < 4 * ws:
        return _names_to_rows(index_names, n2i, names)
    rows = shard_rows(names.shape[0], rank, ws)
    local = torch.from_numpy(_names_to_rows(index_names, n2i, names[rows])).to(eng.device)
    return all_gather_rows(local, names.shape[0]).cpu().numpy()


def _percent(count: int, total: int) -> float:
    # (torch.sum(labels[:, :k]) / len(labels)).item() * 100   (src/validate_stage2.py:60-62,196-203)
    return (torch.tensor(int(count)) / total).item() * 100


def _fiq_captions(captions) -> List[str]:
    # src/validate_stage2.py:97-100
    out = []
    for c in captions:
        if isinstance(c, (list, tuple)) and len(c) == 2:
            out.append(f"{c[0].strip('.?, ').capitalize()} and {c[1].strip('.?, ')}")
        else:
            out.append(c)
    return out


def _tokens(blip_model, dataset, captions):
    tb = getattr(dataset, "token_batch", None)
    return tokenize(blip_model.tokenizer, tb if tb is not None else captions, blip_model.engine.device)


LENGTH_BUCKET = 8      # queries are grouped by token length rounded up to a multiple of this


def _length_buckets(mask: torch.Tensor, bucket: int):
    """The reference tokenises one query at a time, so every query runs at its own length
    (src/validate_stage2.py:104-106, padding='longest' over a batch of one).  Batching all queries at the
    longest caption's length would waste FLOPs on padding, so queries are grouped by their own length
    (rounded up to ``bucket``) and each group runs at that length; padded positions inside a group are
    masked keys (-10000) exactly as in a padded reference batch.  Yields (row indices, L)."""
    lens = mask.sum(dim=1).cpu().numpy()
    Lmax = mask.shape[1]
    padded = np.minimum(((np.maximum(lens, 1) + bucket - 1) // bucket) * bucket, Lmax)
    for L in np.unique(padded):
        yield np.flatnonzero(padded == L), int(L)


def _predict(blip_model, model_stage1, dataset, index_names, index_features, captions, cand_names, row_active,
             extra_cand_names=None, kv_cache=None):
    """-> (scores [Q,K], extra scores [Q,K'] | None).  z_t is computed once per query and shared by both lists.
    ``kv_cache``: optional ``blip_model.kv_cache(...)`` of the gallery rows the lists name (same scores, bit for bit)."""
    eng = blip_model.engine
    n2i = _name_index(index_names)
    ref_idx = np.array([n2i[n] for n in dataset.reference_names], dtype=np.int32)
    cand_idx = _names_to_rows_sharded(eng, index_names, n2i, cand_names)
    extra_idx = None if extra_cand_names is None else _names_to_rows_sharded(eng, index_names, n2i, extra_cand_names)
    ids, mask = _tokens(blip_model, dataset, captions)
    gallery = eng.to_act(index_features)
    Q = cand_idx.shape[0]
    scores = torch.empty(Q, cand_idx.shape[1], dtype=torch.float32, device=eng.device)
    extra = None if extra_idx is None else torch.empty(Q, extra_idx.shape[1], dtype=torch.float32, device=eng.device)
    active = np.ones(Q, bool) if row_active is None else np.asarray(row_active, bool)
    from .distributed import encode_queries_sharded, score_matrix_sharded
    for rows, L in _length_buckets(mask, LENGTH_BUCKET):
        r_t = torch.from_numpy(rows).to(eng.device)
        ids_b, mask_b = ids[r_t, :L].contiguous(), mask[r_t, :L].contiguous()
        # z_t from the frozen stage-I encoder on the reference image's tokens (src/validate_stage2.py:105-106,243-244).
        # Under torch.distributed (one process per GPU) the queries' z_t and the candidate ranges are split over the ranks
        # and every rank ends up with the full score rows; single-process: plain calls.
        z_t = encode_queries_sharded(model_stage1, gallery, ref_idx[rows], ids_b, mask_b)
        scores[r_t] = score_matrix_sharded(blip_model, gallery, z_t, ids_b, mask_b, cand_idx[rows], active[rows], kv_cache=kv_cache)
        if extra is not None:
            extra[r_t] = score_matrix_sharded(blip_model, gallery, z_t, ids_b, mask_b, extra_idx[rows], None, kv_cache=kv_cache)
    return scores, extra


def generate_fiq_val_predictions(blip_model, model_stage1, relative_val_dataset, index_names, index_features, kv_cache=None):
    """src/validate_stage2.py:69-129 -> (predicted_logits [Q,K] fp32 on device, target_names)."""
    caps = _fiq_captions(relative_val_dataset.captions)
    active = np.asarray(relative_val_dataset.K_labels).any(axis=1)                  # `if True in K_labels` (:95)
    logits, _ = _predict(blip_model, model_stage1, relative_val_dataset, index_names, index_features, caps,
                         relative_val_dataset.K_sorted_index_names, active, kv_cache=kv_cache)
    return logits, list(relative_val_dataset.target_names)


def compute_fiq_val_metrics(relative_val_dataset, blip_model, model_stage1, index_features, index_names, return_order: bool = False,
                            kv_cache=None):
    """src/validate_stage2.py:33-66 -> (recall@10, recall@50).  ``return_order=True`` appends the re-ranked order [Q,K] as a
    HOST int32 array -- the ``sorted_indices`` the reference brings to the CPU at :53.  ``kv_cache``: optional
    ``blip_model.kv_cache(...)`` of the gallery (same metrics and order)."""
    predicted_logits, _ = generate_fiq_val_predictions(blip_model, model_stage1, relative_val_dataset, index_names, index_features,
                                                       kv_cache=kv_cache)
    eng = blip_model.engine
    order = eng.rerank_sort(predicted_logits)                                       # argsort descending (:53)
    labels = torch.from_numpy(np.asarray(relative_val_dataset.K_labels))
    h10, h50 = eng.recall_counts(labels, order, (10, 50))                           # take_along_axis + sums (:56-61)
    Q = len(labels)
    if return_order:
        return _percent(h10, Q), _percent(h50, Q), order.cpu().numpy()
    return _percent(h10, Q), _percent(h50, Q)


def generate_cirr_val_predictions(blip_model, model_stage1, relative_val_dataset, index_names, index_features, kv_cache=None):
    """src/validate_stage2.py:209-278 -> (predicted_logits [Q,K], group_predicted_logits [Q,5],
    reference_names, target_names, group_members_noRef)."""
    ds = relative_val_dataset
    active = np.asarray(ds.K_labels).any(axis=1)                                    # `if True in K_labels` (:239)
    # group members without the reference image, scored for EVERY query (:260-269)
    gm = np.asarray(ds.group_members)
    refs = np.asarray(ds.reference_names)
    group_noref = [[m for m in row if m != r] for row, r in zip(gm.tolist(), refs.tolist())]
    assert all(len(g) == 5 for g in group_noref)
    logits, group_logits = _predict(blip_model, model_stage1, ds, index_names, index_features, list(ds.captions),
                                    ds.K_sorted_index_names, active, extra_cand_names=group_noref, kv_cache=kv_cache)
    return logits, group_logits, list(ds.reference_names), list(ds.target_names), group_noref


def compute_cirr_val_metrics(relative_val_dataset, blip_model, model_stage1, index_features, index_names, kv_cache=None):
    """src/validate_stage2.py:153-206 -> (group_recall@1,2,3, recall@1,5,10,50).  ``kv_cache``: as compute_fiq_val_metrics."""
    predicted_logits, group_logits, _, target_names, group_members = generate_cirr_val_predictions(
        blip_model, model_stage1, relative_val_dataset, index_names, index_features, kv_cache=kv_cache)
    eng = blip_model.engine
    order = eng.rerank_sort(predicted_logits)                                       # :174
    labels = torch.from_numpy(np.asarray(relative_val_dataset.K_labels))            # :178
    r1, r5, r10, r50 = eng.recall_counts(labels, order, (1, 5, 10, 50))
    group_members = np.array(group_members)
    assert group_members.shape[1] == 5                                              # :187
    gorder = eng.rerank_sort(group_logits)                                          # :190
    glabels = torch.from_numpy(group_members == np.array(target_names)[:, None])    # :192-193 (before sorting; gathered by recall_counts)
    g1, g2, g3 = eng.recall_counts(glabels, gorder, (1, 2, 3))
    Q = len(labels)
    return (_percent(g1, Q), _percent(g2, Q), _percent(g3, Q), _percent(r1, Q), _percent(r5, Q), _percent(r10, Q), _percent(r50, Q))
