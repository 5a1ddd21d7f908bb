"""Generate the golden fixtures in this directory from the UNMODIFIED reference.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

It loads the seeded synthetic ``state_dict``s (cir_b200.synthetic) into the reference's own
``BLIP_Retrieval`` / ``BLIP_NLVR`` modules (strict key match), runs the reference methods the
hot path is made of, and stores inputs + outputs as small ``.npz`` files:

  * ``pipeline_small.npz``  -- G=6 images @384, Q=3 ragged 12-token captions, K=4:
      ViT tokens (strided sample + per-image moments), stage-I gallery/query embeddings,
      stage-I top-K, z_t, stage-II 1536-d features and scores, sorted labels, recalls.
  * ``stage2_L32.npz``      -- reference-style init, Q=1, L=32 full mask, K=3 (BASELINE shape).
  * ``training_forward.npz`` -- the in-batch B x B forward of both stages (train=True paths), B=3.
  * ``config1_8x50.npz``     -- BASELINE.json configs[0]: 8 queries x top-50 (stage-I lists of the same run), L=32,
      reference-style init, 384 px, G=56; targets planted at ranks with a score margin so that Recall@{1,5,10,50}
      is well defined under the bf16 tolerance.
  * ``interop.npz``          -- reference-function outputs for format work: ``interpolate_pos_embed`` (src/vit.py:281-305)
      on a 224 px -> 384 px resize, and the CIRR stage-I writer lines (src/validate.py:202-226) on a small distance matrix.

The few lines of ``validate.py`` / ``validate_stage2.py`` that need datasets are restated
inline with their file:line (they are index bookkeeping around the model calls).
"""
import os
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import cir_b200 as cir  # noqa: E402
from ref_shim import build_models  # noqa: E402

syn = cir.synthetic
torch.manual_seed(0)
torch.set_num_threads(os.cpu_count())


def run(name, *, seed, style, G, Q, K, L, min_len, head_gain):
    t0 = time.time()
    sd1 = syn.make_stage1_state_dict(seed, 384, style)
    sd2 = syn.make_stage2_state_dict(seed, 384, style, head_gain=head_gain)
    m1, m2, tok, _ = build_models(sd1, sd2)
    images = syn.make_images(G, 384, seed=1)
    ref_idx, target_idx, ids, mask = syn.make_queries(Q, G, L, seed=3, min_len=min_len)
    feats_in = []
    m2.cls_head.register_forward_hook(lambda mod, inp, out: feats_in.append(inp[0].detach().clone()))
    with torch.no_grad():
        # utils.extract_index_features: src/utils.py:43-55 (stage II) and :56-70 (stage I)
        tokens2 = m2.img_embed(images)
        tokens1, g_emb = m1.img_embed(images, return_pool_and_normalized=True)
        # validate.generate_cirr_val_predictions: src/validate.py:305-311 (normalised twice)
        tok.push(ids, mask)
        q_emb = m1.img_txt_fusion(tokens1[ref_idx], None, ["x"] * Q, train=False)
        q_emb = F.normalize(q_emb)
        # validate.compute_cirr_val_metrics: src/validate.py:202-210
        distances = 1 - q_emb @ g_emb.float().T
        sorted_indices = torch.sort(distances, dim=-1, stable=True).indices
        keep = sorted_indices != ref_idx[:, None]
        sorted_noref = sorted_indices[keep].reshape(Q, G - 1)
        cand_idx = sorted_noref[:, :K]
        k_labels = (cand_idx == target_idx[:, None]).numpy()
        # validate_stage2.generate_cirr_val_predictions: src/validate_stage2.py:235-258
        z_all, scores = [], []
        for q in range(Q):
            tok.push(ids[q:q + 1], mask[q:q + 1])
            z = m1.img_txt_fusion(tokens2[ref_idx[q]][None], None, ["x"], train=False, return_raw=True)
            z_all.append(z.last_hidden_state[0])
            tok.push(ids[q:q + 1], mask[q:q + 1])
            scores.append(m2.img_txt_fusion_val(z, tokens2[cand_idx[q]], ["x"]))
        scores = torch.stack(scores)
        feats = torch.stack(feats_in)
        # validate_stage2.compute_cirr_val_metrics: src/validate_stage2.py:174-179,196-199
        order = torch.sort(scores, dim=-1, descending=True, stable=True).indices
        labels = np.take_along_axis(k_labels, order.numpy(), axis=1)
        lab_t = torch.tensor(labels)
        recalls = [(torch.sum(lab_t[:, :k]) / len(lab_t)).item() * 100 for k in (1, 2, 3, 4)]
    out = dict(
        seed=seed, style=style, G=G, Q=Q, K=K, L=L, min_len=-1 if min_len is None else min_len,
        head_gain=head_gain,
        ref_idx=ref_idx.numpy(), target_idx=target_idx.numpy(), ids=ids.numpy(), mask=mask.numpy(),
        tokens2_sample=tokens2[:, ::48, ::16].numpy(), tokens2_mean=tokens2.mean((1, 2)).numpy(),
        tokens2_std=tokens2.std((1, 2)).numpy(), tokens2_cls=tokens2[:, 0, :].numpy(),
        tokens1_cls=tokens1[:, 0, :].numpy(),
        g_emb=g_emb.numpy(), q_emb=q_emb.numpy(), distances_topk=torch.gather(distances, 1, cand_idx).numpy(),
        cand_idx=cand_idx.numpy().astype(np.int32), k_labels=k_labels,
        z_t=torch.stack(z_all).numpy(), feats=feats.numpy(), scores=scores.numpy(),
        order=order.numpy().astype(np.int32), sorted_labels=labels, recalls=np.array(recalls),
    )
    np.savez_compressed(os.path.join(HERE, name), **out)
    print(f"{name}: {time.time() - t0:.1f}s  scores={scores.numpy().round(4).tolist()}")


def run_training_forward(name, *, seed, style, G, B, L, min_len):
    """In-batch (B x B) forward of both stages: BLIP_Retrieval.img_txt_fusion(train=True) (src/blip_stage1.py:67-92,
    as called by src/stage1_train.py) and BLIP_NLVR.img_txt_fusion (src/blip_stage2.py:65-99, as called by
    src/stage2_train.py:207,468).  Same seeded weights / images / queries as ``pipeline_small.npz``."""
    t0 = time.time()
    sd1 = syn.make_stage1_state_dict(seed, 384, style)
    sd2 = syn.make_stage2_state_dict(seed, 384, style, head_gain=1.0)
    m1, m2, tok, _ = build_models(sd1, sd2)
    images = syn.make_images(G, 384, seed=1)
    ref_idx, target_idx, ids, mask = syn.make_queries(B, G, L, seed=3, min_len=min_len)
    with torch.no_grad():
        tokens2 = m2.img_embed(images)
        tokens1, g_emb = m1.img_embed(images, return_pool_and_normalized=True)
        tok.push(ids, mask)
        s1_logits = m1.img_txt_fusion(tokens1[ref_idx], g_emb[target_idx], ["x"] * B, train=True)          # [B,B] / temp
        tok.push(ids, mask)
        z = m1.img_txt_fusion(tokens2[ref_idx], None, ["x"] * B, train=False, return_raw=True)           # batched z_t
        tok.push(ids, mask)
        s2_logits = m2.img_txt_fusion(z, tokens2[target_idx], ["x"] * B, train=True)                     # [B,B]
    np.savez_compressed(os.path.join(HERE, name), seed=seed, style=style, G=G, B=B, L=L, min_len=min_len,
                        ref_idx=ref_idx.numpy(), target_idx=target_idx.numpy(), ids=ids.numpy(), mask=mask.numpy(),
                        temp=float(m1.temp), s1_logits=s1_logits.numpy(), s2_logits=s2_logits.numpy(),
                        z_t=z.last_hidden_state.numpy())
    print(f"{name}: {time.time() - t0:.1f}s  s2_logits={s2_logits.numpy().round(4).tolist()}")


def run_config1(name, *, seed=2, G=56, Q=8, K=50, L=32, cross_gain=6.0):
    """BASELINE.json configs[0]: 8 synthetic queries x top-50 candidates, 384 px, reference-style random init.
    Candidate lists come from the reference's own stage I on the same inputs (CIRR mode: reference removed,
    src/validate.py:202-210); scoring follows src/validate_stage2.py:235-258.  Labels are synthetic: for query q the
    target is planted at a chosen rank of the REFERENCE's fp32 ranking, picking inside each recall bucket the candidate
    with the largest score margin to the bucket edges (SURVEY 7.3(ii)), so Recall@{1,5,10,50} is a meaningful
    parity check for a bf16 implementation; one query has no positive (filled row, src/validate_stage2.py:123,258)."""
    t0 = time.time()
    sd1 = syn.make_stage1_state_dict(seed, 384, "reference")
    # Reference-style init with two changes that give the candidates of a query distinguishable scores (with the plain
    # N(0, 0.02) init and i.i.d. noise images the score spread of a list is ~0.06 with top gaps of ~0.005, below the 1e-2
    # in-row rounding noise of ANY bf16 implementation -- measured on the B200 with tools/recall_margin_probe.py):
    # images with per-image contrast / brightness, and the cross-attention output projections scaled by `cross_gain`.
    sd2 = syn.make_stage2_state_dict(seed, 384, "reference", head_gain=1.0, cross_gain=cross_gain)
    m1, m2, tok, _ = build_models(sd1, sd2)
    images = syn.make_diverse_images(G, 384, seed=1)
    ref_idx, _, ids, mask = syn.make_queries(Q, G, L, seed=3, min_len=None)
    feats_in = []
    m2.cls_head.register_forward_hook(lambda mod, inp, out: feats_in.append(inp[0].detach().clone()))
    with torch.no_grad():
        tokens2 = m2.img_embed(images)
        tokens1, g_emb = m1.img_embed(images, return_pool_and_normalized=True)
        tok.push(ids, mask)
        q_emb = F.normalize(m1.img_txt_fusion(tokens1[ref_idx], None, ["x"] * Q, train=False))
        distances = 1 - q_emb @ g_emb.float().T
        sorted_indices = torch.sort(distances, dim=-1, stable=True).indices
        keep = sorted_indices != ref_idx[:, None]
        cand_idx = sorted_indices[keep].reshape(Q, G - 1)[:, :K]
        z_all, scores = [], []
        for q in range(Q):
            tok.push(ids[q:q + 1], mask[q:q + 1])
            z = m1.img_txt_fusion(tokens2[ref_idx[q]][None], None, ["x"], train=False, return_raw=True)
            z_all.append(z.last_hidden_state[0])
            tok.push(ids[q:q + 1], mask[q:q + 1])
            scores.append(m2.img_txt_fusion_val(z, tokens2[cand_idx[q]], ["x"]))
        scores = torch.stack(scores)
        feats = torch.stack(feats_in)
        order = torch.sort(scores, dim=-1, descending=True, stable=True).indices
    # ---- plant the targets.  Needed: one query with the target at rank 0, two in ranks [1,5), two in [5,10), two in
    #      [10,50) and one whose target is outside the list.  For every (query, bucket) the best rank is the one with the
    #      largest score margin to the bucket edges; buckets are then handed to queries greedily by that margin.
    s_sorted = np.take_along_axis(scores.numpy(), order.numpy(), axis=1)

    def best_rank(q, lo, hi):
        best, best_m = lo, -1.0
        for r in range(lo, hi):
            up = s_sorted[q, lo - 1] - s_sorted[q, r] if lo > 0 else np.inf          # gap to the last rank of the bucket above
            dn = s_sorted[q, r] - s_sorted[q, hi] if hi < K else np.inf             # gap to the first rank of the bucket below
            if min(up, dn) > best_m:
                best, best_m = r, min(up, dn)
        return best, best_m
    need = [(0, 1), (1, 5), (1, 5), (5, 10), (5, 10), (10, 50), (10, 50)]
    target_idx = np.zeros(Q, np.int64)
    margins = np.zeros(Q, np.float32)
    bucket_lo = np.full(Q, -1, np.int32)
    # assignment of buckets to queries that maximises the smallest margin (8 queries: exhaustive)
    import itertools
    table = {(q, b): best_rank(q, *b) for q in range(Q) for b in set(need)}
    best_perm, best_min = None, -1.0
    for perm in itertools.permutations(range(Q), len(need)):
        m = min(table[(q, b)][1] for q, b in zip(perm, need))
        if m > best_min:
            best_perm, best_min = perm, m
    free = set(range(Q))
    for q, (lo, hi) in zip(best_perm, need):
        r, m = table[(q, (lo, hi))]
        target_idx[q] = int(cand_idx[q, order[q, r]])
        margins[q], bucket_lo[q] = m, lo
        free.discard(q)
    for q in free:                                                                    # target outside the list
        outside = [g for g in range(G) if g != int(ref_idx[q]) and g not in cand_idx[q].tolist()]
        target_idx[q] = outside[0]
        margins[q] = np.inf
    k_labels = (cand_idx.numpy() == target_idx[:, None])
    sc = scores.clone()
    sc[~torch.tensor(k_labels).any(1)] = -99999.99                                   # src/validate_stage2.py:123,258
    order_f = torch.sort(sc, dim=-1, descending=True, stable=True).indices
    labels = np.take_along_axis(k_labels, order_f.numpy(), axis=1)
    lab_t = torch.tensor(labels)
    recalls = [(torch.sum(lab_t[:, :k]) / len(lab_t)).item() * 100 for k in (1, 5, 10, 50)]   # :196-199
    # kept under 1 MB: z_t of the two queries the tests score in fp32, features on a seeded sample of 512 of 1536 columns
    z_rows = np.array([0, 5], np.int64)
    f_cols = np.sort(np.random.default_rng(0).choice(1536, size=512, replace=False)).astype(np.int64)
    np.savez_compressed(os.path.join(HERE, name), seed=seed, style="reference", head_gain=1.0, cross_gain=cross_gain, images="diverse", G=G, Q=Q, K=K, L=L,
                        ref_idx=ref_idx.numpy(), target_idx=target_idx, ids=ids.numpy(), mask=mask.numpy(),
                        cand_idx=cand_idx.numpy().astype(np.int32), k_labels=k_labels,
                        z_t=torch.stack(z_all).numpy()[z_rows], z_t_rows=z_rows, scores=scores.numpy(),
                        feats=feats.numpy()[:, :, f_cols].astype(np.float16), feats_cols=f_cols, order=order.numpy().astype(np.int32),
                        margins=margins, bucket_lo=bucket_lo, recalls=np.array(recalls), tokens2_cls=tokens2[:, 0, :].numpy())
    print(f"{name}: {time.time() - t0:.1f}s recalls={recalls} margins={margins.round(5).tolist()} "
          f"score range=({float(scores.min()):.4f},{float(scores.max()):.4f}) std={float(scores.std()):.4f}")


def run_interop(name):
    """Outputs of two reference code fragments used by the format layer:
    (1) ``vit.interpolate_pos_embed`` (src/vit.py:281-305) resizing a 224 px position table (197 tokens) to 384 px (577);
    (2) the CIRR stage-I writer lines, src/validate.py:202-226, restated verbatim on a seeded [Q,G] distance matrix
        (they need only numpy/torch): sorted names without the reference, labels, group_labels."""
    sys.path.insert(0, os.path.join(os.environ.get("CIR_REFERENCE", "/root/reference"), "src"))
    from ref_shim import load_reference
    load_reference()
    import vit as ref_vit

    class _V:                                            # the two attributes interpolate_pos_embed reads
        class patch_embed:
            num_patches = (384 // 16) ** 2
        pos_embed = torch.zeros(1, 577, 768)
    g = torch.Generator().manual_seed(7)
    pos224 = torch.randn(1, 197, 768, generator=g) * 0.02
    pos384 = ref_vit.interpolate_pos_embed(pos224, _V)
    # ---- (2) src/validate.py:202-226
    Q, G = 7, 23
    index_names = syn.index_names_for(G)
    gq = torch.Generator().manual_seed(8)
    predicted_features = F.normalize(torch.randn(Q, 256, generator=gq), dim=-1)
    index_features = F.normalize(torch.randn(G, 256, generator=gq), dim=-1)
    ref_i, tgt_i, _, _ = syn.make_queries(Q, G, 8, seed=9)
    groups = syn.make_group_members(ref_i, tgt_i, G, seed=10)
    reference_names = [index_names[i] for i in ref_i.tolist()]
    target_names = [index_names[i] for i in tgt_i.tolist()]
    group_members = [[index_names[i] for i in row[1:]] for row in groups.tolist()]       # reference removed (validate.py:300-303)
    distances = 1 - predicted_features @ index_features.T
    sorted_indices = torch.argsort(distances, dim=-1).cpu()
    sorted_index_names = np.array(index_names)[sorted_indices]
    reference_mask = torch.tensor(
        sorted_index_names != np.repeat(np.array(reference_names), len(index_names)).reshape(len(target_names), -1))
    sorted_index_names = sorted_index_names[reference_mask].reshape(sorted_index_names.shape[0], sorted_index_names.shape[1] - 1)
    labels = torch.tensor(
        sorted_index_names == np.repeat(np.array(target_names), len(index_names) - 1).reshape(len(target_names), -1))
    group_members_a = np.array(group_members)
    group_mask = (sorted_index_names[..., None] == group_members_a[:, None, :]).sum(-1).astype(bool)
    group_labels = labels[group_mask].reshape(labels.shape[0], -1)
    rec = [(torch.sum(labels[:, :k]) / len(labels)).item() * 100 for k in (1, 5, 10, 50)]
    grec = [(torch.sum(group_labels[:, :k]) / len(group_labels)).item() * 100 for k in (1, 2, 3)]
    # kept under 1 MB: the input regenerates from its seed (its class-token row checks that), the output is stored for all
    # 577 rows on a seeded sample of 384 of 768 channels
    ch = np.sort(np.random.default_rng(0).choice(768, size=384, replace=False)).astype(np.int64)
    np.savez_compressed(os.path.join(HERE, name), pos224_cls=pos224[:, 0].numpy(), pos384=pos384.numpy()[..., ch], pos384_channels=ch,
                        q_emb=predicted_features.numpy(), g_emb=index_features.numpy(), ref_idx=ref_i.numpy(), target_idx=tgt_i.numpy(),
                        groups=groups.numpy(), sorted_index_names=sorted_index_names, labels=labels.numpy(),
                        group_labels=group_labels.numpy(), recalls=np.array(rec), group_recalls=np.array(grec))
    print(f"{name}: recalls={rec} group={grec}")


if __name__ == "__main__":
    if len(sys.argv) > 1:                                 # e.g. `make_golden.py config1 interop`
        if "config1" in sys.argv:
            run_config1("config1_8x50.npz")
        if "interop" in sys.argv:
            run_interop("interop.npz")
        sys.exit(0)
    run("pipeline_small.npz", seed=0, style="dense", G=6, Q=3, K=4, L=12, min_len=8, head_gain=1.0)
    run("stage2_L32.npz", seed=1, style="reference", G=4, Q=1, K=3, L=32, min_len=None, head_gain=1.0)
    run_training_forward("training_forward.npz", seed=0, style="dense", G=6, B=3, L=12, min_len=8)
    run_config1("config1_8x50.npz")
    run_interop("interop.npz")
