"""CPU tests of the data formats either side of the hot path: top-K file (stage I -> stage II),
checkpoint ingestion, CIRR submission dicts."""
import json
import os

import numpy as np
import pytest
import torch

import cir_b200 as cir


def test_topk_file_roundtrip(tmp_path):
    T = cir.topk_file
    names = [f"img{i}" for i in range(12)]
    sorted_names = np.array([[names[(q + j) % 12] for j in range(8)] for q in range(5)])
    targets = [names[(q + 3) % 12] for q in range(5)]
    group_labels = torch.zeros(5, 5, dtype=torch.bool)
    d = T.make_topk_dict(sorted_names, names, "val", target_names=targets, group_labels=group_labels, k=8)
    assert d["labels"].shape == (5, 8) and d["labels"].sum() == 5
    p = os.path.join(tmp_path, "cirr_top_8_val.pt")
    T.save_topk(p, d)
    got = T.load_topk(p, K=4, split="val", index_names=names, target_names=targets)
    assert got["K"] == 4 and got["K_sorted_index_names"].shape == (5, 4)
    assert got["K_labels"].dtype == bool and got["K_labels"].sum() == 5
    assert got["K_group_labels"].shape == (5, 5)
    with pytest.raises(AssertionError):
        T.load_topk(p, K=9, split="val")              # K larger than the saved file
    with pytest.raises(AssertionError):
        T.load_topk(p, K=4, split="test1")            # wrong split
    with pytest.raises(AssertionError):
        T.load_topk(p, K=4, split="val", index_names=names[::-1])
    # Fashion-IQ flavour
    d2 = T.make_topk_dict(sorted_names, names, "val", target_names=targets, dress_types="dress")
    p2 = os.path.join(tmp_path, "fiq.pt")
    T.save_topk(p2, d2)
    assert T.load_topk(p2, K=8, split="val", dress_type="dress")["K_labels"].shape == (5, 8)
    with pytest.raises(AssertionError):
        T.load_topk(p2, K=8, split="val", dress_type="shirt")
    # the loaded fields feed the synthetic dataset object the drivers consume
    ds = cir.synthetic.SyntheticRelativeDataset(names, [0] * 5, [(q + 3) % 12 for q in range(5)], ["c"] * 5,
                                                np.array([[names.index(n) for n in row] for row in got["K_sorted_index_names"]]))
    assert np.array_equal(ds.K_labels, got["K_labels"])


def test_cirr_submission_dicts():
    T = cir.topk_file
    K_names = np.array([[f"c{q}_{j}" for j in range(60)] for q in range(3)])
    order = np.stack([np.random.default_rng(q).permutation(60) for q in range(3)])
    gm = np.array([[f"g{q}_{j}" for j in range(5)] for q in range(3)])
    gorder = np.stack([np.random.default_rng(10 + q).permutation(5) for q in range(3)])
    sub, gsub = T.cirr_submission_dicts([11, 12, 13], K_names, order, gm, gorder)
    assert sub["version"] == "rc2" and sub["metric"] == "recall" and gsub["metric"] == "recall_subset"
    assert len(sub["12"]) == 50 and sub["12"][0] == K_names[1, order[1, 0]]
    assert len(gsub["13"]) == 3 and gsub["13"] == [gm[2, i] for i in gorder[2, :3]]
    json.dumps(sub, sort_keys=True)


def test_checkpoint_ingestion(tmp_path):
    Cp = cir.checkpoint
    syn = cir.synthetic
    # fine-tuned checkpoint layout of src/utils.py:135-150
    sd = {"visual_encoder.pos_embed": torch.randn(1, 577, 768), "cls_head.0.weight": torch.randn(4, 4)}
    p = os.path.join(tmp_path, "tuned.pt")
    torch.save({"epoch": 3, "BLIP_NLVR": sd, "optimizer_state_dict": {}}, p)
    got = Cp.load_state_dict(p, "BLIP_NLVR", 384)
    assert torch.equal(got["cls_head.0.weight"], sd["cls_head.0.weight"])
    # BLIP base layout: twin duplication + pos-embed interpolation 224 -> 384
    base = {"visual_encoder.pos_embed": torch.randn(1, 197, 768),
            "text_encoder.encoder.layer.0.attention.self.query.weight": torch.randn(2, 2),
            "text_encoder.encoder.layer.0.crossattention.self.key.bias": torch.randn(2),
            "text_encoder.encoder.layer.0.attention.output.dense.weight": torch.randn(2, 2),
            "text_encoder.encoder.layer.0.crossattention.output.LayerNorm.weight": torch.randn(2),
            "text_encoder.encoder.layer.0.output.LayerNorm.weight": torch.randn(2)}
    p2 = os.path.join(tmp_path, "base.pt")
    torch.save({"model": base}, p2)
    got = Cp.load_state_dict(p2, "BLIP_NLVR", 384)
    assert got["visual_encoder.pos_embed"].shape == (1, 577, 768)
    assert torch.equal(got["visual_encoder.pos_embed"][:, 0], base["visual_encoder.pos_embed"][:, 0])
    k = "text_encoder.encoder.layer.0."
    for s in ("0", "1"):
        assert torch.equal(got[k + f"attention.self{s}.query.weight"], base[k + "attention.self.query.weight"])
        assert torch.equal(got[k + f"crossattention.self{s}.key.bias"], base[k + "crossattention.self.key.bias"])
        assert torch.equal(got[k + f"attention.output.dense{s}.weight"], base[k + "attention.output.dense.weight"])
    for s in ("A", "B"):
        assert torch.equal(got[k + f"crossattention.output.LayerNorm{s}.weight"], base[k + "crossattention.output.LayerNorm.weight"])
    assert k + "output.LayerNormA.weight" not in got                     # FFN LayerNorm stays shared
    # interpolation matches the reference formula on an identity-size input
    same = Cp.interpolate_pos_embed(sd["visual_encoder.pos_embed"], 576)
    assert same is sd["visual_encoder.pos_embed"]


def _load_golden(name):
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name))
    return {k: z[k] for k in z.files}


def test_interpolate_pos_embed_matches_reference_function():
    """224 px -> 384 px position table against the output of the reference's own ``vit.interpolate_pos_embed``
    (src/vit.py:281-305), generated by tests/golden/make_golden.py (interop.npz)."""
    g = _load_golden("interop.npz")
    pos224 = torch.randn(1, 197, 768, generator=torch.Generator().manual_seed(7)) * 0.02      # the input make_golden.py drew
    assert np.array_equal(pos224[:, 0].numpy(), g["pos224_cls"])
    got = cir.checkpoint.interpolate_pos_embed(pos224, 576)
    assert got.shape == (1, 577, 768)
    assert np.abs(got[..., g["pos384_channels"]].numpy() - g["pos384"]).max() <= 1e-6     # all 577 rows, seeded channel sample
    assert np.array_equal(got[:, 0].numpy(), g["pos224_cls"])             # class token kept


def test_cirr_topk_file_is_readable_by_the_reference_reader(tmp_path):
    """The dict shape the CIRR stage-I driver writes (src/validate.py:256-263) from the fixture the reference's own writer
    lines produced, through reader logic restated from src/data_utils.py:290-305 (``group_labels`` is read unconditionally)."""
    from oracle import cir_oracle as O
    T = cir.topk_file
    g = _load_golden("interop.npz")
    names = cir.synthetic.index_names_for(g["g_emb"].shape[0])
    ref_idx, tgt_idx, groups = g["ref_idx"], g["target_idx"], g["groups"]
    noref, labels, group_labels = O.cirr_stage1_lists(torch.tensor(g["q_emb"]), torch.tensor(g["g_emb"]), ref_idx, tgt_idx, groups[:, 1:])
    # the oracle's index bookkeeping == the reference's name bookkeeping
    assert np.array_equal(np.array(names)[noref.numpy()], g["sorted_index_names"])
    assert np.array_equal(labels.numpy(), g["labels"]) and np.array_equal(group_labels.numpy(), g["group_labels"])
    K = 10
    d = T.make_topk_dict(np.array(names)[noref.numpy()], names, "val", target_names=[names[i] for i in tgt_idx],
                         labels=labels, group_labels=group_labels, k=K)
    p = os.path.join(tmp_path, "cirr_top_10_val.pt")
    T.save_topk(p, d)
    # ---- src/data_utils.py:290-305, restated
    tmp_f = torch.load(p, weights_only=False)
    assert K <= tmp_f["sorted_index_names"].shape[-1]
    assert tmp_f["split"] == "val"
    K_sorted_index_names = tmp_f["sorted_index_names"][:, :K]
    assert tmp_f["index_names"] == names
    K_labels = tmp_f["labels"][:, :K].numpy()
    K_group_labels = tmp_f["group_labels"].numpy()
    assert tmp_f["target_names"] == [names[i] for i in tgt_idx]
    assert np.array_equal(K_sorted_index_names, g["sorted_index_names"][:, :K])
    assert np.array_equal(K_labels, g["labels"][:, :K]) and np.array_equal(K_group_labels, g["group_labels"])
    got = T.load_topk(p, K=K, split="val", index_names=names, target_names=[names[i] for i in tgt_idx])
    assert np.array_equal(got["K_group_labels"], g["group_labels"])
    # a CIRR file without group_labels is rejected exactly where the reference would fail (KeyError at :301)
    d.pop("group_labels")
    T.save_topk(p, d)
    with pytest.raises(KeyError):
        T.load_topk(p, K=K, split="val")


def test_tokenizer_is_never_silently_synthetic(monkeypatch):
    B = cir.blip
    monkeypatch.delenv("CIR_SYNTHETIC_TOKENIZER", raising=False)
    tok = B.init_tokenizer()
    if isinstance(tok, B.MissingTokenizer):                 # no vocabulary on disk (this container, the GPU box)
        assert tok.enc_token_id == 30523
        with pytest.raises(B.CirTokenizerError):
            tok(["a caption"])
        assert isinstance(B.init_tokenizer(synthetic=True), cir.synthetic.SyntheticTokenizer)
        monkeypatch.setenv("CIR_SYNTHETIC_TOKENIZER", "1")
        assert isinstance(B.init_tokenizer(), cir.synthetic.SyntheticTokenizer)
    else:
        assert not isinstance(tok, cir.synthetic.SyntheticTokenizer)
