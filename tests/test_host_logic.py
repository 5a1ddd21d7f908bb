"""CPU tests of the host side: C-ABI library exports, scheduler, tokenizer, synthetic data."""
import os
import re

import numpy as np
import pytest
import torch

import cir_b200 as cir

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import ctypes
    from importlib import import_module
    native = import_module("candidate-reranking-cir_b200.native")
    hdr = open(os.path.join(ROOT, "include", "cir_b200.h")).read()
    declared = set(re.findall(r"\b(cir_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 25
    assert os.path.exists(native.LIB_PATH), "build the library first: python __graft_entry__.py"
    lib = ctypes.CDLL(native.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/cir_b200.h but not exported"
    assert declared == set(native.exported_symbols()), declared ^ set(native.exported_symbols())
    assert native.lib().cir_version() == 100


def test_no_gpu_means_loud_failure(monkeypatch):
    if torch.cuda.is_available():                                # on a GPU machine, torch is made to report none
        monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    from importlib import import_module
    native = import_module("candidate-reranking-cir_b200.native")
    engine = import_module("candidate-reranking-cir_b200.engine")
    with pytest.raises(native.CirError):
        engine.get_engine()
    with pytest.raises(native.CirError):
        cir.blip_stage2.BLIP_NLVR(image_size=384)


def test_plan_chunks_covers_every_triplet_once():
    from importlib import import_module
    sched = import_module("candidate-reranking-cir_b200.schedule")
    rng = np.random.default_rng(0)
    Q, K, G = 37, 11, 23
    cand = np.stack([rng.permutation(G)[:K] for _ in range(Q)]).astype(np.int32)
    active = rng.random(Q) < 0.8
    for mt, mc in ((2048, 64), (16, 3), (5, 1), (1, 1)):
        chunks = sched.plan_chunks(cand, active, mt, mc)
        seen = np.concatenate([c.flat_pos for c in chunks]) if chunks else np.zeros(0, np.int64)
        want = np.flatnonzero(np.repeat(active, K))
        assert np.array_equal(np.sort(seen), want)
        for c in chunks:
            assert len(c.flat_pos) <= mt and len(c.cand_list) <= mc
            assert np.array_equal(c.cand_list[c.trip_slot], cand.reshape(-1)[c.flat_pos])
            assert np.array_equal(c.query_list[c.trip_query], c.flat_pos // K)
            assert np.all(np.diff(c.cand_list) > 0)
    assert sched.plan_chunks(cand, np.zeros(Q, bool)) == []
    assert sched.plan_chunks(np.zeros((0, 4), np.int32)) == []


def test_plan_chunks_splits_an_oversized_candidate():
    from importlib import import_module
    sched = import_module("candidate-reranking-cir_b200.schedule")
    cand = np.zeros((10, 3), np.int32)         # one candidate, 30 triplets
    chunks = sched.plan_chunks(cand, None, max_triplets=8, max_candidates=4)
    assert [len(c.flat_pos) for c in chunks] == [8, 8, 8, 6]
    assert all(list(c.cand_list) == [0] for c in chunks)


def test_shard_rows_partitions():
    from importlib import import_module
    sched = import_module("candidate-reranking-cir_b200.schedule")
    for n in (0, 1, 7, 8, 4181):
        for w in (1, 2, 3, 8):
            got = [sched.shard_rows(n, r, w) for r in range(w)]
            assert got[0].start == 0 and got[-1].stop == n
            assert all(a.stop == b.start for a, b in zip(got, got[1:]))
            sizes = [s.stop - s.start for s in got]
            assert max(sizes) - min(sizes) <= 1


def test_synthetic_tokenizer_surface():
    tok = cir.synthetic.SyntheticTokenizer()
    enc = tok(["make the dog bigger", "a"], padding="longest", return_tensors="pt")
    assert enc.input_ids.shape == enc.attention_mask.shape == (2, 6)
    assert enc.input_ids[0, 0] == 101 and enc.input_ids[0, -1] == 102
    assert enc.attention_mask[1].tolist() == [1, 1, 1, 0, 0, 0]
    assert tok.enc_token_id == 30523
    again = tok(["make the dog bigger"])
    assert torch.equal(again.input_ids[0], enc.input_ids[0])


def test_random_topk_plants_targets():
    syn = cir.synthetic
    ref, tgt, ids, mask = syn.make_queries(50, 40, 8)
    cand, labels = syn.make_random_topk(50, 40, 10, ref, tgt, hit_rate=0.9)
    assert cand.shape == (50, 10) and labels.sum(1).max() <= 1
    assert not (cand.long() == ref[:, None]).any()
    assert all(len(set(r.tolist())) == 10 for r in cand)
    assert 0.7 < labels.any(1).float().mean() <= 1.0


def test_build_attn_work_units():
    from importlib import import_module
    sched = import_module("candidate-reranking-cir_b200.schedule")
    slot = np.array([0, 0, 0, 0, 0, 1, 3, 3], np.int32)
    for L, warps in ((32, 8), (12, 8), (40, 8), (32, 2)):
        mt = (L + 15) // 16
        w = sched.build_attn_work(slot, L, warps)
        covered = set()
        for b0, u0, nu, _ in w.tolist():
            for u in range(u0, min(u0 + warps, nu)):
                t, mi = b0 + u // mt, u % mt
                assert slot[t] == slot[b0]
                assert (t, mi) not in covered
                covered.add((t, mi))
        assert covered == {(t, mi) for t in range(len(slot)) for mi in range(mt)}
    assert sched.build_attn_work(np.zeros(0, np.int32), 32).shape == (0, 4)


def test_build_attn_tiles_cover():
    from importlib import import_module
    sched = import_module("candidate-reranking-cir_b200.schedule")
    slot = np.array([0, 0, 0, 0, 0, 1, 3, 3, 3, 3, 3, 3, 3, 3, 3], np.int32)
    for L in (1, 12, 32, 40, 64, 100, 300, 577):
        tiles = sched.build_attn_tiles(slot, L)
        rows = set()
        for b0, nb, row0, RB in tiles.tolist():
            assert nb * RB <= 256 and nb >= 1
            assert len({slot[b0 + i] for i in range(nb)}) == 1
            for i in range(nb):
                for r in range(row0, min(row0 + RB, L)):
                    assert (b0 + i, r) not in rows
                    rows.add((b0 + i, r))
        assert rows == {(t, r) for t in range(len(slot)) for r in range(L)}


def test_ctypes_structs_match_the_c_header(tmp_path):
    """The ctypes mirrors in native.py must have the size (and hence the layout rules) of the structs in
    include/cir_b200.h: compile a tiny C program against the header and compare sizeof."""
    import ctypes as C
    import os
    import subprocess
    N = cir.native
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pairs = {"cir_gemm_args": N.GemmArgs, "cir_attn_args": N.AttnArgs, "cir_qkv_attn_args": N.QkvAttnArgs, "cir_vit_weights": N.VitWeights,
             "cir_stage1_weights": N.Stage1Weights, "cir_stage2_weights": N.Stage2Weights, "cir_vit_state": N.VitState,
             "cir_text_embed_state": N.TextEmbedState, "cir_stage1_state": N.Stage1State, "cir_stage2_state": N.Stage2State}
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "cir_b200.h"\nint main(void) {\n' +
                   "".join(f'  printf("{n} %zu\\n", sizeof({n}));\n' for n in pairs) + "  return 0;\n}\n")
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    sizes = dict(line.split() for line in out.strip().splitlines())
    for name, ct in pairs.items():
        assert int(sizes[name]) == C.sizeof(ct), (name, sizes[name], C.sizeof(ct))


def test_candidate_partition_and_balanced_chunks():
    from importlib import import_module
    sched = import_module("candidate-reranking-cir_b200.schedule")
    rng = np.random.default_rng(1)
    Q, K, G = 301, 20, 97
    cand = np.stack([rng.permutation(G)[:K] for _ in range(Q)]).astype(np.int32)
    active = rng.random(Q) < 0.9
    want = np.flatnonzero(np.repeat(active, K))
    for world in (1, 2, 3, 8):
        seen, owners, infos = [], {}, []
        for r in range(world):
            info = {}
            chunks = sched.plan_chunks(cand, active, 512, 16, part=(r, world), info=info)
            infos.append(info["part_sizes"])
            assert sum(c.flat_pos.size for c in chunks) == info["part_sizes"][r]
            for c in chunks:
                assert c.flat_pos.size <= 512 and c.cand_list.size <= 16
                seen.append(c.flat_pos)
                for g in c.cand_list.tolist():
                    assert owners.setdefault(g, r) == r, "a candidate's triplets must stay on one rank"
        assert all(i == infos[0] for i in infos)                                     # every rank derives the same partition
        assert np.array_equal(np.sort(np.concatenate(seen)), want)
        sizes = np.array(infos[0])
        assert sizes.max() - sizes.min() <= 2 * np.bincount(cand[active].reshape(-1)).max()    # cut moved by at most one candidate run
    # balanced chunks: no small tail chunk
    chunks = sched.plan_chunks(cand, active, 512, 64)
    sizes = np.array([c.flat_pos.size for c in chunks])
    assert sizes.min() > 0.8 * sizes.max()
    greedy = sched.plan_chunks(cand, active, 512, 64, balance=False)
    assert np.array_equal(np.sort(np.concatenate([c.flat_pos for c in greedy])), want)
    # wide candidate ids (no 16-bit radix fast path)
    big = cand.astype(np.int64) * 1000
    a = sched.plan_chunks(big, active, 512, 16)
    assert np.array_equal(np.sort(np.concatenate([c.flat_pos for c in a])), want)
