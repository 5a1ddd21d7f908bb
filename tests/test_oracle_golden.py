"""The CPU oracle (oracle/cir_oracle.py) against the fixtures the UNMODIFIED reference
produced (tests/golden/make_golden.py).  This is the pin for every parity claim."""
import os

import numpy as np
import pytest
import torch

import cir_b200 as cir
from oracle import cir_oracle as O

syn = cir.synthetic
torch.set_num_threads(os.cpu_count() or 1)


def _load(golden_dir, name):
    z = np.load(os.path.join(golden_dir, name))
    return {k: z[k] for k in z.files}


@pytest.fixture(scope="module")
def small(golden_dir):
    g = _load(golden_dir, "pipeline_small.npz")
    sd1 = syn.make_stage1_state_dict(int(g["seed"]), 384, str(g["style"]))
    sd2 = syn.make_stage2_state_dict(int(g["seed"]), 384, str(g["style"]), head_gain=float(g["head_gain"]))
    images = syn.make_images(int(g["G"]), 384, seed=1)
    with torch.no_grad():
        tokens2 = O.vit_forward(sd2, images)
    return g, sd1, sd2, images, tokens2


def test_synthetic_inputs_reproduce(small):
    g = small[0]
    ref_idx, target_idx, ids, mask = syn.make_queries(int(g["Q"]), int(g["G"]), int(g["L"]), seed=3,
                                                       min_len=int(g["min_len"]))
    assert np.array_equal(ref_idx.numpy(), g["ref_idx"])
    assert np.array_equal(target_idx.numpy(), g["target_idx"])
    assert np.array_equal(ids.numpy(), g["ids"])
    assert np.array_equal(mask.numpy(), g["mask"])
    assert (g["mask"].sum(1) < g["mask"].shape[1]).any(), "fixture must contain ragged (padded) captions"


def test_vit_matches_reference(small):
    g, _, _, _, tokens2 = small
    assert np.abs(tokens2[:, ::48, ::16].numpy() - g["tokens2_sample"]).max() < 2e-5
    assert np.abs(tokens2[:, 0, :].numpy() - g["tokens2_cls"]).max() < 2e-5
    assert np.abs(tokens2.mean((1, 2)).numpy() - g["tokens2_mean"]).max() < 1e-6


def test_stage1_matches_reference(small):
    g, sd1, _, images, tokens2 = small
    ids, mask = torch.tensor(g["ids"]), torch.tensor(g["mask"])
    ref_idx = torch.tensor(g["ref_idx"])
    with torch.no_grad():
        tokens1 = O.vit_forward(sd1, images)
        assert np.abs(tokens1[:, 0, :].numpy() - g["tokens1_cls"]).max() < 2e-5
        g_emb = O.stage1_gallery_embedding(sd1, tokens1)
        assert np.abs(g_emb.numpy() - g["g_emb"]).max() < 1e-5
        q_emb = O.stage1_query_embedding(sd1, O.stage1_hidden(sd1, tokens1[ref_idx], ids, mask))
        q_emb = torch.nn.functional.normalize(q_emb)          # CIRR: src/validate.py:311
        assert np.abs(q_emb.numpy() - g["q_emb"]).max() < 1e-5
        # z_t uses the stage-II ViT's tokens: src/validate_stage2.py:243-244,293
        z = O.stage1_hidden(sd1, tokens2[ref_idx], ids, mask)
        assert np.abs(z.numpy() - g["z_t"]).max() < 5e-5
    # top-K from the reference's own fp32 embeddings must be bit-exact
    dist, idx = O.stage1_topk(torch.tensor(g["q_emb"]), torch.tensor(g["g_emb"]), ref_idx, int(g["K"]))
    assert np.array_equal(idx.numpy().astype(np.int32), g["cand_idx"])
    assert np.array_equal(dist.numpy(), g["distances_topk"])


def test_stage2_matches_reference(small):
    g, _, sd2, _, tokens2 = small
    ids, mask = torch.tensor(g["ids"]), torch.tensor(g["mask"])
    z_t = torch.tensor(g["z_t"])
    cand_idx = torch.tensor(g["cand_idx"]).long()
    with torch.no_grad():
        for q in range(int(g["Q"])):
            f = O.stage2_features(sd2, z_t[q:q + 1], ids[q:q + 1], mask[q:q + 1], tokens2[cand_idx[q]])
            assert np.abs(f.numpy() - g["feats"][q]).max() < 1e-4
            s = O.stage2_head(sd2, f)
            assert np.abs(s.numpy() - g["scores"][q]).max() < 1e-4


def test_rerank_and_recall_bit_exact_from_reference_scores(small):
    g = small[0]
    scores = torch.tensor(g["scores"])
    assert np.array_equal(O.rerank_order(scores).numpy().astype(np.int32), g["order"])
    lab = O.sorted_labels(scores, g["k_labels"])
    assert np.array_equal(lab.numpy(), g["sorted_labels"])
    assert O.recall_at(lab, (1, 2, 3, 4)) == list(g["recalls"])


def test_stage2_L32_reference_init(golden_dir):
    g = _load(golden_dir, "stage2_L32.npz")
    sd2 = syn.make_stage2_state_dict(int(g["seed"]), 384, str(g["style"]), head_gain=float(g["head_gain"]))
    images = syn.make_images(int(g["G"]), 384, seed=1)
    with torch.no_grad():
        tokens2 = O.vit_forward(sd2, images)
        s = O.stage2_score(sd2, torch.tensor(g["z_t"])[0:1], torch.tensor(g["ids"]), torch.tensor(g["mask"]),
                           tokens2[torch.tensor(g["cand_idx"][0]).long()])
    assert np.abs(s.numpy() - g["scores"][0]).max() < 1e-5


def test_empty_positive_rows_are_filled(small):
    g, sd1, sd2, _, tokens2 = small
    k_labels = np.zeros_like(g["k_labels"])
    out = O.stage2_predictions(sd1, sd2, tokens2, torch.tensor(g["ref_idx"]), torch.tensor(g["ids"]),
                               torch.tensor(g["mask"]), torch.tensor(g["cand_idx"]), k_labels)
    assert torch.all(out == O.NEG_FILL)


def test_training_shape_forward_matches_reference(small, golden_dir):
    """The in-batch B x B forward of both stages (train=True paths of src/blip_stage1.py:88-91 and
    src/blip_stage2.py:65-99) as run by the unmodified reference -> training_forward.npz."""
    g0, sd1, sd2, images, tokens2 = small
    g = _load(golden_dir, "training_forward.npz")
    assert int(g["seed"]) == int(g0["seed"]) and str(g["style"]) == str(g0["style"]) and int(g["G"]) == int(g0["G"])
    ids, mask = torch.tensor(g["ids"]), torch.tensor(g["mask"])
    ref_idx, target_idx = torch.tensor(g["ref_idx"]), torch.tensor(g["target_idx"])
    B = int(g["B"])
    with torch.no_grad():
        tokens1 = O.vit_forward(sd1, images)
        g_emb = O.stage1_gallery_embedding(sd1, tokens1)
        pred = O.stage1_query_embedding(sd1, O.stage1_hidden(sd1, tokens1[ref_idx], ids, mask))
        s1 = pred @ g_emb[target_idx].T / float(sd1["temp"])
        assert abs(float(sd1["temp"]) - float(g["temp"])) < 1e-7
        assert np.abs(s1.numpy() - g["s1_logits"]).max() < 2e-4                     # logits are O(1/temp) = O(14)
        z = O.stage1_hidden(sd1, tokens2[ref_idx], ids, mask)
        assert np.abs(z.numpy() - g["z_t"]).max() < 5e-5
        z_ref = torch.tensor(g["z_t"])
        s2 = torch.stack([O.stage2_score(sd2, z_ref[i:i + 1], ids[i:i + 1], mask[i:i + 1], tokens2[target_idx]) for i in range(B)])
        assert np.abs(s2.numpy() - g["s2_logits"]).max() < 1e-4


def test_config1_8x50_matches_reference(golden_dir):
    """BASELINE.json configs[0] (8 queries x top-50, L=32, reference-style init): the oracle against the reference's scores for
    two of the eight queries (the CPU budget of this suite), and the label / recall bookkeeping for all of them."""
    g = _load(golden_dir, "config1_8x50.npz")
    sd1 = syn.make_stage1_state_dict(int(g["seed"]), 384, "reference")
    sd2 = syn.make_stage2_state_dict(int(g["seed"]), 384, "reference", head_gain=1.0, cross_gain=float(g["cross_gain"]))
    assert str(g["images"]) == "diverse"
    images = syn.make_diverse_images(int(g["G"]), 384, seed=1)
    ids, mask = torch.tensor(g["ids"]), torch.tensor(g["mask"])
    with torch.no_grad():
        tokens2 = O.vit_forward(sd2, images)
        assert np.abs(tokens2[:, 0, :].numpy() - g["tokens2_cls"]).max() < 5e-5
        for i, q in enumerate(g["z_t_rows"].tolist()):                 # the fixture keeps z_t of queries 0 and 5
            z = O.stage1_hidden(sd1, tokens2[int(g["ref_idx"][q])][None], ids[q:q + 1], mask[q:q + 1])
            assert np.abs(z[0].numpy() - g["z_t"][i]).max() < 1e-4
            s = O.stage2_score(sd2, z, ids[q:q + 1], mask[q:q + 1], tokens2[torch.tensor(g["cand_idx"][q]).long()])
            assert np.abs(s.numpy() - g["scores"][q]).max() <= 1e-4
    sc = torch.tensor(g["scores"]).clone()
    sc[~torch.tensor(g["k_labels"]).any(1)] = O.NEG_FILL
    assert np.array_equal(O.rerank_order(torch.tensor(g["scores"])).numpy(), g["order"])
    assert O.recall_at(O.sorted_labels(sc, g["k_labels"]), (1, 5, 10, 50)) == g["recalls"].tolist()
    assert g["recalls"].tolist() == [12.5, 37.5, 62.5, 87.5]            # ranks 0 | [1,5) x2 | [5,10) x2 | [10,50) x2 | absent
    assert float(g["margins"].min()) > 3e-2          # > 3x the measured bf16 in-row ranking noise (profiles/r02_recall_margin_probe.txt)


def test_cirr_stage1_lists_match_reference_writer(golden_dir):
    g = _load(golden_dir, "interop.npz")
    names = np.array(syn.index_names_for(g["g_emb"].shape[0]))
    noref, labels, gl = O.cirr_stage1_lists(torch.tensor(g["q_emb"]), torch.tensor(g["g_emb"]), g["ref_idx"], g["target_idx"], g["groups"][:, 1:])
    assert np.array_equal(names[noref.numpy()], g["sorted_index_names"])
    assert np.array_equal(labels.numpy(), g["labels"]) and np.array_equal(gl.numpy(), g["group_labels"])
    assert O.recall_at(labels, (1, 5, 10, 50)) == g["recalls"].tolist()
    assert O.recall_at(gl, (1, 2, 3)) == g["group_recalls"].tolist()
