"""Round-2 parity cases (all through the C-ABI on the GPU):
  * BASELINE.json configs[0] (8 queries x top-50, L=32, ViT-produced tokens) against the UNMODIFIED reference's fp32 scores:
    |dscore| <= 2e-2 on all 400 triplets, feature relative error, Recall@{1,5,10,50} identical (targets planted with a margin);
  * the CIRR stage-I writer lines (group_labels, 7-tuple) against the fixture produced by the reference's own lines;
  * utils.extract_index_features with the reference's signature (both modes, batches of 16);
  * checkpoint ingestion: reference-layout files loaded through blip_stage{1,2}(pretrained=...)."""
import os

import numpy as np
import pytest
import torch

import cir_b200 as cir
from helpers import golden_images, golden_weights, load_golden
from oracle import cir_oracle as O

pytestmark = pytest.mark.gpu
syn = cir.synthetic
SCORE_TOL = 2e-2          # BASELINE.json north_star: per-triplet scores within 2e-2 absolute in bf16


@pytest.fixture(scope="module")
def config1():
    g = load_golden("config1_8x50.npz")
    sd1, sd2 = golden_weights(g)
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd1, precision="bf16")
    m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision="bf16")
    tokens2 = m2.img_embed(golden_images(g))                                 # the stage-II model's ViT (validate_stage2.py:145,293)
    return g, m1, m2, tokens2


def test_config1_scores_and_features_bf16(config1):
    g, m1, m2, tokens2 = config1
    Q, K = int(g["Q"]), int(g["K"])
    ids, mask = torch.tensor(g["ids"]), torch.tensor(g["mask"])
    z_t, _ = m1.encode_queries(tokens2, torch.tensor(g["ref_idx"]).int(), ids, mask, want_z=True, want_emb=False)
    s = m2.score_triplets(z_t, ids, mask, tokens2, g["cand_idx"])
    err = np.abs(s.cpu().numpy() - g["scores"])
    assert err.shape == (Q, K) and err.max() <= SCORE_TOL, err.max()
    # within a query the error is mostly common-mode: the RANKING error (score minus the row mean) is what recall sees
    d = s.cpu().numpy() - g["scores"]
    rank_err = np.abs(d - d.mean(1, keepdims=True)).max()
    print(f"config1: max|dscore|={err.max():.2e} mean={err.mean():.2e} max in-row ranking error={rank_err:.2e} "
          f"(planted margin/2 = {float(g['margins'].min()) / 2:.2e})")
    # 1536-d pre-head features of all 400 triplets, relative Frobenius error over the fixture's seeded column sample
    ch = cir.schedule.plan_chunks(g["cand_idx"], None, 4096, 64)[0]
    assert ch.flat_pos.size == Q * K
    _, f = m2.engine.stage2_score_chunk(m2._w, tokens2, ch.cand_list, z_t, ids.cuda(), mask.cuda(), ch.trip_query, ch.trip_slot, want_feats=True)
    assert f.shape[1] == 1536
    cols = torch.from_numpy(g["feats_cols"])
    want = torch.tensor(g["feats"].astype(np.float32)).reshape(-1, cols.numel())[torch.from_numpy(ch.flat_pos)]
    rel = ((f.cpu()[:, cols] - want).norm() / want.norm()).item()
    assert rel < 3e-2, rel


def test_config1_recall_identical_to_reference(config1):
    """validate_stage2-shaped run on the synthetic dataset object: Recall@{1,5,10,50} of the bf16 CUDA path equals the recall
    the reference's own fp32 scores give (fixture), including the row whose target is not in the list (-99999.99 fill)."""
    g, m1, m2, tokens2 = config1
    G, Q = int(g["G"]), int(g["Q"])
    names = syn.index_names_for(G)
    tb = syn.TokenBatch(input_ids=torch.tensor(g["ids"]), attention_mask=torch.tensor(g["mask"]))
    groups = syn.make_group_members(torch.tensor(g["ref_idx"]), torch.tensor(g["target_idx"]), G, seed=11)
    ds = syn.SyntheticRelativeDataset(names, g["ref_idx"], g["target_idx"], ["x"] * Q, g["cand_idx"], kind="cirr",
                                      group_idx=groups.numpy(), token_batch=tb)
    assert np.array_equal(ds.K_labels, g["k_labels"])
    got = cir.validate_stage2.compute_cirr_val_metrics(ds, m2, m1, tokens2, names)
    assert list(got[3:]) == g["recalls"].tolist(), (got, g["recalls"])
    # the full re-ranked label matrix, not only its prefix sums
    logits, _, _, _, _ = cir.validate_stage2.generate_cirr_val_predictions(m2, m1, ds, names, tokens2)
    order = m2.engine.rerank_sort(logits).cpu().numpy()
    ref_scores = torch.tensor(g["scores"]).clone()
    ref_scores[~torch.tensor(g["k_labels"]).any(1)] = O.NEG_FILL
    want_pos = np.argmax(O.sorted_labels(ref_scores, g["k_labels"]).numpy(), axis=1)
    got_pos = np.argmax(np.take_along_axis(g["k_labels"], order, axis=1), axis=1)
    active = g["k_labels"].any(1)
    assert np.array_equal(want_pos[active] < 1, got_pos[active] < 1)
    for k in (5, 10, 50):
        assert np.array_equal(want_pos[active] < k, got_pos[active] < k), (k, want_pos, got_pos)
    r10, r50 = cir.validate_stage2.compute_fiq_val_metrics(ds, m2, m1, tokens2, names)
    assert [r10, r50] == g["recalls"].tolist()[2:]


def test_config1_fp32_check_mode(config1):
    """fp32 check mode on two of the eight queries: <= 1e-4 on scores against the reference (ViT tokens included)."""
    g = config1[0]
    sd1, sd2 = golden_weights(g)
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd1, precision="fp32")
    m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision="fp32")
    tokens = m2.img_embed(golden_images(g))
    assert np.abs(tokens[:, 0, :].cpu().numpy() - g["tokens2_cls"]).max() < 2e-4
    rows = g["z_t_rows"].tolist()                                            # queries 0 and 5
    ids, mask = torch.tensor(g["ids"][rows]), torch.tensor(g["mask"][rows])
    z_t, _ = m1.encode_queries(tokens, torch.tensor(g["ref_idx"][rows]).int(), ids, mask, want_z=True, want_emb=False)
    assert np.abs(z_t.cpu().numpy() - g["z_t"]).max() < 3e-4
    s = m2.score_triplets(z_t, ids, mask, tokens, g["cand_idx"][rows])
    assert np.abs(s.cpu().numpy() - g["scores"][rows]).max() <= 1e-4


def test_cirr_stage1_lists_match_reference_writer():
    """group_labels / labels / sorted names from cir_stage1_topk + cir_stage1_rank_members == the arrays the reference's own
    writer lines (src/validate.py:202-226) produced for the same embeddings (tests/golden/interop.npz)."""
    g = load_golden("interop.npz")
    eng = cir.engine.get_engine(None, "bf16")
    G = g["g_emb"].shape[0]
    names = np.array(syn.index_names_for(G))
    q_emb, g_emb = torch.tensor(g["q_emb"]).cuda(), torch.tensor(g["g_emb"]).cuda()
    top_idx, labels, group_labels, gorder = cir.validate.cirr_topk_from_embeddings(
        eng, q_emb, g_emb, g["ref_idx"], g["target_idx"], g["groups"][:, 1:], G - 1)
    assert np.array_equal(names[top_idx.cpu().numpy()], g["sorted_index_names"])
    assert np.array_equal(labels.cpu().numpy(), g["labels"])
    assert np.array_equal(group_labels.cpu().numpy(), g["group_labels"])
    # member distances are the same numbers the fused top-K reports for those gallery rows
    md, mo = eng.stage1_rank_members(q_emb, g_emb, g["groups"][:, 1:])
    td, ti = eng.stage1_topk(q_emb, g_emb, G - 1, exclude=g["ref_idx"].astype(np.int32))
    for q in range(len(ti)):
        pos = {int(i): p for p, i in enumerate(ti[q].tolist())}
        for j, m in enumerate(g["groups"][q, 1:].tolist()):
            assert md[q, j].item() == td[q, pos[m]].item()


def test_stage1_cirr_driver_returns_reference_tuple(tmp_path):
    """validate.compute_cirr_val_metrics: 7-tuple in the reference's order (src/validate.py:268) and a saved top-K file
    that the CIRR reader logic accepts (group_labels present, one positive per row)."""
    g = load_golden("pipeline_small.npz")
    sd1, _ = golden_weights(g)
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd1, precision="bf16")
    G = int(g["G"])
    names = syn.index_names_for(G)
    images = syn.make_images(G, 384, seed=1)
    tokens1, g_emb = m1.img_embed(images, return_pool_and_normalized=True)
    Q = 5
    ref, tgt, ids, mask = syn.make_queries(Q, G, 10, seed=9, min_len=6)
    groups = syn.make_group_members(ref, tgt, G, seed=11)             # 6 members incl. the reference: needs G >= 6
    tb = syn.TokenBatch(input_ids=ids, attention_mask=mask)
    ds = syn.SyntheticRelativeDataset(names, ref, tgt, ["x"] * Q, np.zeros((Q, 4), int), kind="cirr", group_idx=groups.numpy(), token_batch=tb)
    p = os.path.join(tmp_path, "cirr_top_5_val.pt")
    out = cir.validate.compute_cirr_val_metrics(ds, m1, tokens1, g_emb, names, k=G - 1, save_topk_path=p)
    assert len(out) == 7
    g1, g2, g3, r1, r5, r10, r50 = out
    assert 0 <= g1 <= g2 <= g3 <= 100 and 0 <= r1 <= r5 <= r10 <= r50 == 100.0      # k = G-1: every target is in the list
    f = cir.topk_file.load_topk(p, K=G - 1, split="val", index_names=names, target_names=ds.target_names)
    assert f["K_group_labels"].shape == (Q, 5) and (f["K_group_labels"].sum(1) == 1).all()
    assert (f["K_labels"].sum(1) == 1).all()
    # same lists from the oracle on the CUDA path's own embeddings
    _, q_emb = m1.encode_queries(tokens1, ref.int(), ids.clone().index_fill_(1, torch.tensor([0]), 30523), mask,
                                 want_z=False, want_emb=True, normalize_twice=True)
    noref, labels, gl = O.cirr_stage1_lists(q_emb.cpu(), g_emb.cpu(), ref.numpy(), tgt.numpy(), groups[:, 1:].numpy())
    assert np.array_equal(np.array(names)[noref.numpy()], f["K_sorted_index_names"])
    assert np.array_equal(gl.numpy(), f["K_group_labels"])
    assert (g1, g2, g3) == tuple(O.recall_at(gl, (1, 2, 3))) and (r1, r5, r10, r50) == tuple(O.recall_at(labels, (1, 5, 10, 50)))
    # Fashion-IQ flavour keeps the reference's 2-tuple
    ds.dress_types = ["dress"]
    r = cir.validate.compute_fiq_val_metrics(ds, m1, tokens1, g_emb, names, k=G)
    assert len(r) == 2


class _Classic:
    """'classic'-mode dataset stand-in (src/data_utils.py): item i -> (image_name, image tensor)."""

    def __init__(self, names, images):
        self.names, self.images = names, images

    def __len__(self):
        return len(self.names)

    def __getitem__(self, i):
        return self.names[i], self.images[i]


def test_extract_index_features_reference_signature():
    """utils.extract_index_features(dataset, model, blip_stage2= / blip_stage1=): src/utils.py:25-72, batches of 16."""
    g = load_golden("pipeline_small.npz")
    sd1, sd2 = golden_weights(g)
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd1, precision="bf16")
    m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision="bf16")
    G = 19                                              # 16 + 3: two batches, the second ragged
    images = syn.make_images(G, 384, seed=1)
    names = syn.index_names_for(G)
    ds = _Classic(names, images)
    feats2, names2 = cir.validate.extract_index_features(ds, m2, blip_stage2=True)
    assert names2 == names and feats2.shape == (G, 577, 768)
    direct = torch.cat([m2.img_embed(images[:16]), m2.img_embed(images[16:])])
    assert torch.equal(feats2, direct)
    # the first 6 images are the golden fixture's gallery: tokens against the reference's ViT output
    err = np.abs(feats2[:6].float().cpu()[:, ::48, ::16].numpy() - g["tokens2_sample"])
    assert err.max() < 0.15 and err.mean() < 0.02
    feats1, pooled, names1 = cir.validate.extract_index_features(ds, m1, blip_stage1=True)
    assert names1 == names and feats1.shape == (G, 577, 768) and pooled.shape == (G, 256) and pooled.dtype == torch.float32
    assert np.abs(pooled[:6].cpu().numpy() - g["g_emb"]).max() < 2e-2
    assert (pooled.norm(dim=1) - 1).abs().max() < 1e-5
    with pytest.raises(AssertionError):
        cir.validate.extract_index_features(ds, m2, blip_stage2=True, blip_stage1=True)
    with pytest.raises(RuntimeError):
        cir.validate.extract_index_features(ds, m2)
    e2, n2 = cir.validate.extract_index_features(_Classic([], images[:0]), m2, blip_stage2=True)
    assert e2.shape[0] == 0 and n2 == []


def test_checkpoint_files_load_through_the_factories(tmp_path):
    """Reference-layout checkpoint files (src/utils.py:135-150 save_model; BLIP base {'model': ...}) through
    blip_stage2(pretrained=...) / blip_stage1(pretrained=...): same scores as binding the state_dict directly, which the
    golden tests pin to the reference; the 224 px BLIP-base position table is interpolated like src/vit.py:281-305."""
    g = load_golden("stage2_L32.npz")
    sd1, sd2 = golden_weights(g)
    p2 = os.path.join(tmp_path, "tuned_nlvr.pt")
    torch.save({"epoch": 7, "BLIP_NLVR": sd2, "optimizer_state_dict": {}}, p2)
    m2 = cir.blip_stage2.blip_stage2(pretrained=p2, image_size=384, precision="bf16")
    tokens2 = m2.img_embed(syn.make_images(int(g["G"]), 384, seed=1))
    s = m2.score_triplets(torch.tensor(g["z_t"]).cuda().bfloat16(), torch.tensor(g["ids"]), torch.tensor(g["mask"]), tokens2, g["cand_idx"])
    assert np.abs(s.cpu().numpy() - g["scores"]).max() <= SCORE_TOL
    direct = cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision="bf16")
    s2 = direct.score_triplets(torch.tensor(g["z_t"]).cuda().bfloat16(), torch.tensor(g["ids"]), torch.tensor(g["mask"]),
                               direct.img_embed(syn.make_images(int(g["G"]), 384, seed=1)), g["cand_idx"])
    assert torch.equal(s, s2)
    # stage I from a BLIP-base-style file trained at 224 px: {'model': sd} with a 197-token position table
    sd224 = dict(sd1)
    gpos = torch.Generator().manual_seed(3)
    sd224["visual_encoder.pos_embed"] = torch.randn(1, 197, 768, generator=gpos) * 0.02
    p1 = os.path.join(tmp_path, "blip_base_224.pt")
    torch.save({"model": sd224}, p1)
    m1 = cir.blip_stage1.blip_stage1(pretrained=p1, image_size=384, precision="bf16")
    sd384 = dict(sd1)
    sd384["visual_encoder.pos_embed"] = cir.checkpoint.interpolate_pos_embed(sd224["visual_encoder.pos_embed"], 576)
    want = cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd384, precision="bf16")
    img = syn.make_images(2, 384, seed=4)
    assert torch.equal(m1.img_embed(img), want.img_embed(img))
    # a BLIP base file has no trained merge layers: stage II refuses it with a clear message instead of a KeyError
    base2 = {k: v for k, v in sd1.items() if k.startswith(("visual_encoder.", "text_encoder."))}
    pb = os.path.join(tmp_path, "blip_base_for_nlvr.pt")
    torch.save({"model": base2}, pb)
    with pytest.raises(cir.native.CirError, match="merge_layer"):
        cir.blip_stage2.blip_stage2(pretrained=pb, image_size=384, precision="bf16")


def test_engine_cache_respects_device_zero():
    eng0 = cir.engine.get_engine("cuda:0", "bf16")
    assert eng0.device.index == 0
    assert cir.engine.get_engine(torch.device("cuda", 0), "bf16") is eng0
    before = torch.cuda.current_device()
    cir.engine.Engine(torch.device("cuda", 0), "fp32")            # cir_create must not change the caller's current device
    assert torch.cuda.current_device() == before


def test_index_range_checks():
    g = load_golden("pipeline_small.npz")
    sd1, sd2 = golden_weights(g)
    m2 = cir.blip_stage2.blip_stage2(image_size=384, state_dict=sd2, precision="bf16")
    tok = torch.zeros(3, 577, 768, dtype=torch.bfloat16, device="cuda")
    z = torch.zeros(1, 8, 768, dtype=torch.bfloat16, device="cuda")
    ids, mask = torch.full((1, 8), 1000), torch.ones(1, 8, dtype=torch.long)
    with pytest.raises(cir.native.CirError, match="cand_idx"):
        m2.score_triplets(z, ids, mask, tok, np.array([[0, 3]]))             # row 3 of a 3-image gallery
    with pytest.raises(cir.native.CirError, match="token ids"):
        m2.score_triplets(z, torch.full((1, 8), 40000), mask, tok, np.array([[0, 1]]))
