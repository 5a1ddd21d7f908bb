"""Resident stage-I index (cir_stage1_index_*, engine.Stage1Index): a search returns exactly what cir_stage1_topk returns over the
same rows, bit for bit -- on the tensor-core filter path, the fp32 path, while the index grows, for queries that take the
per-query exact fallback, when replayed from a CUDA graph, through the validation drivers and sharded over ranks."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import cir_b200 as cir
from helpers import golden_weights, load_golden

pytestmark = pytest.mark.gpu
N = cir.native
syn = cir.synthetic


@pytest.fixture(scope="module")
def eng():
    return cir.engine.get_engine(precision="bf16")


def _unit(n, seed, dim=256):
    g = torch.Generator().manual_seed(seed)
    return torch.nn.functional.normalize(torch.randn(n, dim, generator=g), dim=-1)


def _index(eng, g, capacity=None):
    idx = eng.stage1_index(g.shape[0] if capacity is None else capacity)
    return idx.add(g)


def _fp32_path(eng, fn):
    eng.set_stage1_tensor_cores(False)
    try:
        return fn()
    finally:
        eng.set_stage1_tensor_cores(True)


def _same(a, b):
    return torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def _exclude(Q, G, seed):
    ex = torch.randint(0, G, (Q,), generator=torch.Generator().manual_seed(seed)).int()
    ex[::3] = -1
    return ex


def _adversarial(Q, G, seed):
    """Gallery sorted by increasing similarity to query 0: its candidate list overflows (the designed fallback path)."""
    q = _unit(Q, seed)
    base = _unit(G, seed + 1)
    return q, base[torch.argsort(base @ q[0])]


@pytest.mark.parametrize("Q,G,K", [(37, 20000, 50), (300, 70001, 200), (5, 16384, 1), (64, 33000, 1000), (23, 16383, 100)])
def test_index_equals_stage1_topk_and_fp32_path(eng, Q, G, K):
    q, g = _unit(Q, 1), _unit(G, 2)
    kw = dict(exclude=_exclude(Q, G, 3), col_offset=1000)
    idx = _index(eng, g)
    got = idx.topk(q, K, **kw)
    assert _same(got, eng.stage1_topk(q, g, K, **kw))
    assert _same(got, _fp32_path(eng, lambda: eng.stage1_topk(q, g, K, **kw)))
    assert _same(got, _fp32_path(eng, lambda: idx.topk(q, K, **kw)))
    assert not (got[1].cpu() == kw["exclude"][:, None]).any()
    assert int(got[1].min()) >= 1000 and int(got[1].max()) < 1000 + G


def test_ties_near_duplicates_and_unnormalised_rows(eng):
    Q, G, K = 16, 40000, 100
    q, g = _unit(Q, 5), _unit(G, 6)
    g[1000:1040] = g[999]                      # 41 identical rows
    g[20000:20030] = g[7] * (1 + 1e-4)         # near-duplicates of one row, distinguishable only in fp32
    g[30000] = q[3]
    got = _index(eng, g).topk(q, K)
    assert _same(got, eng.stage1_topk(q, g, K)) and _same(got, _fp32_path(eng, lambda: eng.stage1_topk(q, g, K)))
    assert int(got[1][3, 0]) == 30000
    Q, G, K = 32, 25000, 64
    q = _unit(Q, 11) * torch.linspace(0.1, 30, Q)[:, None]
    g = _unit(G, 12) * torch.rand(G, generator=torch.Generator().manual_seed(13))[:, None] * 5
    got = _index(eng, g).topk(q, K)
    assert _same(got, eng.stage1_topk(q, g, K)) and _same(got, _fp32_path(eng, lambda: eng.stage1_topk(q, g, K)))


def test_incremental_build_matches_one_shot(eng):
    """16-row appends (the extract_index_features batch), then one 50k block that crosses 16,384 rows (the search switches to
    the tensor-core filter); a search between appends sees exactly the rows added so far."""
    Q, K = 24, 50
    q, g = _unit(Q, 21), _unit(640 + 50000, 22)
    ex = _exclude(Q, g.shape[0], 23)
    idx = eng.stage1_index(g.shape[0])
    for b in range(40):
        idx.add(g[16 * b:16 * (b + 1)])
        if b in (0, 2, 39):                        # 16 rows (K > rows: empty slots), 48, 640
            n = idx.rows
            assert n == 16 * (b + 1)
            assert _same(idx.topk(q, K, exclude=ex), eng.stage1_topk(q, g[:n], K, exclude=ex))
    idx.add(g[640:])
    assert idx.rows == g.shape[0] and torch.equal(idx.g_f32.cpu(), g)
    got = idx.topk(q, K, exclude=ex)
    assert _same(got, _index(eng, g).topk(q, K, exclude=ex))
    assert _same(got, eng.stage1_topk(q, g, K, exclude=ex))
    assert _same(got, _fp32_path(eng, lambda: eng.stage1_topk(q, g, K, exclude=ex)))


@pytest.mark.parametrize("K", [1, 50, 1000])
def test_per_query_exact_fallback(eng, K):
    Q, G = 4, 60000
    q, g = _adversarial(Q, G, 8)
    ex = torch.tensor([G - 1, -1, 5, -1], dtype=torch.int32)
    rows = torch.full((Q,), -7, dtype=torch.int32, device=eng.device)
    got = _index(eng, g).topk(q, K, exclude=ex, exact_rows=rows)
    want = _fp32_path(eng, lambda: eng.stage1_topk(q, g, K, exclude=ex))
    assert _same(got, want) and _same(eng.stage1_topk(q, g, K, exclude=ex), want)
    assert int(got[1][0, 0]) == G - 2                        # its best row G - 1 is excluded
    rows = rows.cpu()
    assert rows[0] == 1 and set(rows.tolist()) <= {0, 1}


def test_cuda_graph_replay(eng):
    """index.topk captured once on static buffers, replayed for three query batches (one adversarial: the exact fallback runs
    inside the graph); and cir_stage1_topk itself is capturable at G >= 16,384 (it no longer reads a flag back)."""
    Q, G, K = 64, 60000, 50
    q_adv, g = _adversarial(Q, G, 31)
    batches = [_unit(Q, 33), q_adv, _unit(Q, 34)]
    ex = _exclude(Q, G, 35)
    dev = eng.device
    idx = _index(eng, g)
    q_s, ex_s = batches[0].to(dev), ex.to(dev)
    td, ti = torch.empty(Q, K, device=dev), torch.empty(Q, K, dtype=torch.int32, device=dev)
    rows = torch.zeros(Q, dtype=torch.int32, device=dev)
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):                            # warm-up: the index's workspace for (Q, K) exists before capture
        idx.topk(q_s, K, exclude=ex_s, out=(td, ti), exact_rows=rows)
    torch.cuda.current_stream(dev).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        idx.topk(q_s, K, exclude=ex_s, out=(td, ti), exact_rows=rows)
    for i, qb in enumerate(batches):
        q_s.copy_(qb)
        graph.replay()
        torch.cuda.synchronize(dev)
        assert _same((td, ti), eng.stage1_topk(qb, g, K, exclude=ex)), i
        assert (int(rows[0]) == 1) == (i == 1), (i, rows.tolist())
    # cir_stage1_topk under capture
    g_d, q_d = g.to(dev), batches[1].to(dev)
    want = eng.stage1_topk(q_d, g_d, K)
    torch.cuda.synchronize(dev)
    graph2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph2):
        out = eng.stage1_topk(q_d, g_d, K)
    graph2.replay()
    torch.cuda.synchronize(dev)
    assert _same(out, want)


def test_fp32_engine():
    e32 = cir.engine.get_engine(precision="fp32")
    Q, G, K = 20, 20000, 30
    q, g = _unit(Q, 41), _unit(G, 42)
    ex = _exclude(Q, G, 43)
    got = _index(e32, g).topk(q, K, exclude=ex)
    assert _same(got, e32.stage1_topk(q, g, K, exclude=ex))
    assert _same(got, cir.engine.get_engine(precision="bf16").stage1_topk(q, g, K, exclude=ex))


def test_rejected_input(eng):
    idx = _index(eng, _unit(60, 51), capacity=100)
    with pytest.raises(N.CirError, match=r"rc=-1\).*capacity"):
        idx.add(_unit(41, 52))
    assert idx.rows == 60
    q = _unit(3, 53).to(eng.device)
    for k in (0, 1025):
        with pytest.raises(N.CirError, match=r"rc=-1\).*out of range"):
            idx.topk(q, k)
    lib = N.lib()
    td, ti = torch.empty(3, 10, device=eng.device), torch.empty(3, 10, dtype=torch.int32, device=eng.device)
    ws = torch.empty(256, dtype=torch.uint8, device=eng.device)
    assert lib.cir_stage1_index_topk_workspace_bytes(eng.ctx, C.byref(idx._s), 3, 10) > ws.numel()
    eng._sync_stream()
    with pytest.raises(N.CirError, match=r"rc=-3\)"):
        N.check(lib.cir_stage1_index_topk(eng.ctx, C.byref(idx._s), N.ptr(q), 3, N.vp(0), 0, 10, N.ptr(td), N.ptr(ti), N.vp(0),
                                          N.ptr(ws), ws.numel()), "cir_stage1_index_topk")
    s = N.Stage1Index()
    with pytest.raises(N.CirError, match=r"rc=-3\)"):
        N.check(lib.cir_stage1_index_init(eng.ctx, N.ptr(ws), ws.numel(), 1000, C.byref(s)), "cir_stage1_index_init")


def _same_topk_dict(a, b):
    assert a.keys() == b.keys()
    for key in a:
        x, y = a[key], b[key]
        if isinstance(x, torch.Tensor):
            assert torch.equal(x, y), key
        elif isinstance(x, np.ndarray):
            assert np.array_equal(x, y), key
        else:
            assert x == y, key


def test_validate_drivers_with_index():
    g = load_golden("pipeline_small.npz")
    sd1, _ = golden_weights(g)
    m1 = cir.blip_stage1.blip_stage1(image_size=384, state_dict=sd1, precision="bf16")
    G = int(g["G"])
    names = syn.index_names_for(G)
    tokens1, g_emb = m1.img_embed(syn.make_images(G, 384, seed=1), return_pool_and_normalized=True)
    Q = 5
    ref, tgt, ids, mask = syn.make_queries(Q, G, 10, seed=9, min_len=6)
    groups = syn.make_group_members(ref, tgt, G, seed=11)
    tb = syn.TokenBatch(input_ids=ids, attention_mask=mask)
    ds = syn.SyntheticRelativeDataset(names, ref, tgt, ["x"] * Q, np.zeros((Q, 4), int), kind="cirr", group_idx=groups.numpy(), token_batch=tb)
    idx = _index(m1.engine, g_emb)
    V = cir.validate
    a = V.cirr_val_topk(ds, m1, tokens1, g_emb, names, k=G - 1)
    b = V.cirr_val_topk(ds, m1, tokens1, None, names, k=G - 1, index=idx)
    assert a[0] == b[0]
    _same_topk_dict(a[1], b[1])
    assert V.compute_cirr_val_metrics(ds, m1, tokens1, None, names, k=G - 1, index=idx) == a[0]
    ds.dress_types = ["dress"]
    a = V.fiq_val_topk(ds, m1, tokens1, g_emb, names, k=G)
    b = V.fiq_val_topk(ds, m1, tokens1, None, names, k=G, index=idx)
    assert a[0] == b[0]
    _same_topk_dict(a[1], b[1])
    assert V.compute_fiq_val_metrics(ds, m1, tokens1, None, names, k=G, index=idx) == a[0]


def test_shard_indexes_merge_to_the_whole_index(eng):
    Q, G, K = 40, 50001, 100
    q, g = _unit(Q, 61), _unit(G, 62)
    ex = _exclude(Q, G, 63)
    sched, D = cir.schedule, cir.distributed
    parts = []
    for r in range(2):
        s = sched.shard_rows(G, r, 2)
        parts.append(_index(eng, g[s]).topk(q, K, exclude=ex, col_offset=s.start))
    merged = eng.topk_merge(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]))
    whole = _index(eng, g).topk(q, K, exclude=ex)
    assert _same(merged, whole)
    assert _same(D.ShardedStage1Index(eng, G, lambda rows: g[rows]).topk(q, K, exclude=ex), whole)     # one process: one shard


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, ws, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=torch.device("cuda", rank))
    try:
        dev = torch.device("cuda", rank)
        eng = cir.engine.get_engine(dev, "bf16")
        Q, G, K = 33, 40001, 50
        q, g = _unit(Q, 71).to(dev), _unit(G, 72)
        ex = _exclude(Q, G, 73)
        sharded = cir.distributed.ShardedStage1Index(eng, G, lambda rows: g[rows])
        assert sharded.index.rows == sharded.block.stop - sharded.block.start < G
        got = sharded.topk(q, K, exclude=ex)
        assert _same(got, eng.stage1_topk(q, g, K, exclude=ex))
        ret[rank] = "ok"
    except Exception as e:  # pragma: no cover
        ret[rank] = f"{type(e).__name__}: {e}"
        raise
    finally:
        dist.destroy_process_group()


def test_two_gpu_sharded_index_matches_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    assert dict(ret) == {0: "ok", 1: "ok"}
