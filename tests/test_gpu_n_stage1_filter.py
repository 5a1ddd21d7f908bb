"""Filtered search over the resident stage-I index (cir_stage1_index_topk_filtered, Stage1Index.topk(tags=...)): row r is eligible
for query q iff (row_tag[r] & mask[q]) != 0.  The oracle is stage1_topk over the eligible rows only, one call per distinct mask,
indices mapped back and short lists padded with (+inf, -1); every comparison is bit for bit -- on the tensor-core filter path, the
fp32 path, in an fp32 engine and below 16,384 rows, for the per-query exact fallback, after removals, under CUDA-graph replay
while tags and masks change in place, and sharded over ranks."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import cir_b200 as cir

pytestmark = pytest.mark.gpu
N = cir.native
ALL = cir.engine.ALL_TAGS
MODES = ["tc", "fp32_path", "fp32_engine", "small"]


@pytest.fixture(scope="module")
def eng():
    return cir.engine.get_engine(precision="bf16")


def _unit(n, seed, dim=256):
    g = torch.Generator().manual_seed(seed)
    return torch.nn.functional.normalize(torch.randn(n, dim, generator=g), dim=-1)


def _setup(mode):
    """-> (engine, gallery rows, run(fn)): the path a mode exercises."""
    if mode == "fp32_engine":
        return cir.engine.get_engine(precision="fp32"), 20000, lambda fn: fn()
    e = cir.engine.get_engine(precision="bf16")
    if mode == "small":
        return e, 9000, lambda fn: fn()
    if mode == "fp32_path":
        def run(fn):
            e.set_stage1_tensor_cores(False)
            try:
                return fn()
            finally:
                e.set_stage1_tensor_cores(True)
        return e, 40000, run
    return e, 40000, lambda fn: fn()


def _bits(x):
    return torch.from_numpy(cir.engine.tag_bits(x)) if not isinstance(x, torch.Tensor) else x.cpu().int()


def _oracle(e, q, g, K, row_tags, masks, exclude=None, col_offset=0):
    """stage1_topk over g[eligible] per distinct mask; indices mapped back to col_offset + row; (+inf, -1) padding."""
    rt, m = _bits(row_tags), _bits(masks)
    Q = q.shape[0]
    td = torch.full((Q, K), float("inf"))
    ti = torch.full((Q, K), -1, dtype=torch.int32)
    ex = None if exclude is None else torch.as_tensor(exclude).long().cpu()
    for mv in torch.unique(m).tolist():
        qs = torch.nonzero(m == mv).flatten()
        elig = torch.nonzero((rt & mv) != 0).flatten()
        if elig.numel() == 0:
            continue
        ex_c = None
        if ex is not None:
            local = ex[qs] - col_offset
            pos = torch.searchsorted(elig, local.clamp(min=0))
            hit = (ex[qs] >= 0) & (pos < elig.numel()) & (elig[pos.clamp(max=elig.numel() - 1)] == local)
            ex_c = torch.where(hit, pos, torch.full_like(pos, -1)).int()
        d, i = e.stage1_topk(q[qs], g[elig], K, exclude=ex_c)
        d, i = d.cpu(), i.cpu().long()
        ti[qs] = torch.where(i >= 0, col_offset + elig[i.clamp(min=0)], torch.full_like(i, -1)).int()
        td[qs] = d
    return td, ti


def _same(got, want):
    return torch.equal(got[0].cpu(), want[0].cpu()) and torch.equal(got[1].cpu(), want[1].cpu())


def _index(e, g, tags=None, capacity=None):
    return e.stage1_index(g.shape[0] if capacity is None else capacity).add(g, tags=tags)


@pytest.mark.parametrize("mode", MODES)
def test_all_ones_equals_unfiltered(mode):
    e, G, run = _setup(mode)
    Q, K = 24, 100
    q, g = _unit(Q, 1), _unit(G, 2)
    ex = torch.randint(0, G, (Q,), generator=torch.Generator().manual_seed(3)).int()
    ex[::3] = -1
    idx = _index(e, g)
    plain = run(lambda: idx.topk(q, K, exclude=ex, col_offset=500))
    assert _same(run(lambda: idx.topk(q, K, exclude=ex, col_offset=500, tags=ALL)), plain)
    assert _same(run(lambda: idx.topk(q, K, exclude=ex, col_offset=500, tags=[ALL] * Q)), plain)
    assert _same(plain, e.stage1_topk(q, g, K, exclude=ex, col_offset=500))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("s", [2, 3, 64])
def test_selectivity(mode, s):
    """A fraction 1/s of the rows carries bit 0, the rest bit 1; queries mix mask 1 (selectivity 1/s), 2 and 3 (all rows)."""
    e, G, run = _setup(mode)
    Q, K = 24, 100
    q, g = _unit(Q, 10 + s), _unit(G, 20 + s)
    sel = torch.rand(G, generator=torch.Generator().manual_seed(30 + s)) < 1.0 / s
    tags = torch.where(sel, 1, 2).int()
    masks = torch.tensor([1, 1, 1, 2, 3, 1] * (Q // 6)).int()
    idx = _index(e, g, tags=tags)
    assert torch.equal(idx.row_tags.cpu(), tags)
    got = run(lambda: idx.topk(q, K, tags=masks))
    assert _same(got, _oracle(e, q, g, K, tags, masks))
    assert bool(sel[got[1][masks.to(got[1].device) == 1].long().cpu()].all())


@pytest.mark.parametrize("mode", ["tc", "fp32_path"])
def test_fashion_iq_categories(mode):
    """Three disjoint categories in one index (tags 1 / 2 / 4) == three per-category indexes searched with col_offset = the
    category's first row; the union mask 6 == one index over the two adjacent categories."""
    e, _, run = _setup(mode)
    sizes = [20000, 17000, 9000]
    starts = np.cumsum([0] + sizes)
    g = _unit(int(starts[-1]), 40)
    tags = torch.cat([torch.full((n,), 1 << c, dtype=torch.int32) for c, n in enumerate(sizes)])
    Q, K = 16, 200
    q = _unit(Q, 41)
    idx = _index(e, g, tags=tags)
    for c in range(3):
        got = run(lambda: idx.topk(q, K, tags=1 << c))
        lo, hi = int(starts[c]), int(starts[c + 1])
        want = run(lambda: _index(e, g[lo:hi]).topk(q, K, col_offset=lo))
        assert _same(got, want), c
    got = run(lambda: idx.topk(q, K, tags=6))
    lo = int(starts[1])
    assert _same(got, run(lambda: _index(e, g[lo:]).topk(q, K, col_offset=lo)))
    masks = torch.tensor([1, 2, 4, 6] * (Q // 4)).int()
    assert _same(run(lambda: idx.topk(q, K, tags=masks)), _oracle(e, q, g, K, tags, masks))


@pytest.mark.parametrize("mode", MODES)
def test_short_and_empty_lists(mode):
    e, G, run = _setup(mode)
    Q, K = 6, 100
    q, g = _unit(Q, 50), _unit(G, 51)
    tags = torch.ones(G, dtype=torch.int32)
    few = torch.randperm(G, generator=torch.Generator().manual_seed(52))[:30]
    tags[few] = 8
    masks = torch.tensor([8, 16, 0, 1, 9, 8]).int()        # 30 rows, none, none (mask 0), all but 30, all, 30
    idx = _index(e, g, tags=tags)
    got = run(lambda: idx.topk(q, K, tags=masks))
    assert _same(got, _oracle(e, q, g, K, tags, masks))
    d, i = got[0].cpu(), got[1].cpu()
    assert (i[0] >= 0).sum() == 30 and (i[0, 30:] == -1).all() and torch.isinf(d[0, 30:]).all()
    assert (i[1] == -1).all() and (i[2] == -1).all() and torch.isinf(d[2]).all()
    assert set(i[0, :30].tolist()) == set(few.tolist())


@pytest.mark.parametrize("mode", ["tc", "fp32_path"])
def test_exclude_eligible_and_ineligible_rows(mode):
    e, G, run = _setup(mode)
    Q, K = 4, 50
    q, g = _unit(Q, 60), _unit(G, 61)
    idx = _index(e, g)
    top1 = idx.topk(q, 1)[1].cpu().flatten()
    tags = torch.ones(G, dtype=torch.int32)
    tags[top1[1]] = 2                                      # query 1's nearest row is ineligible for mask 1
    idx.set_tags(torch.arange(G), tags)
    ex = torch.tensor([top1[0], top1[1], -1, top1[3]]).int()       # eligible (q0, q3), ineligible (q1)
    masks = torch.tensor([1, 1, 1, 3]).int()
    got = run(lambda: idx.topk(q, K, exclude=ex, tags=masks))
    assert _same(got, _oracle(e, q, g, K, tags, masks, exclude=ex))
    i = got[1].cpu()
    assert int(top1[0]) not in i[0].tolist() and int(top1[1]) not in i[1].tolist() and int(top1[3]) not in i[3].tolist()
    assert _same(run(lambda: idx.topk(q[1:2], K, tags=1)), (got[0][1:2], got[1][1:2]))   # excluding an ineligible row: no effect


@pytest.mark.parametrize("mode", ["tc", "fp32_path", "fp32_engine"])
def test_ties_with_ineligible_lowest_members(mode):
    e, G, run = _setup(mode)
    Q, K = 8, 60
    q, g = _unit(Q, 70), _unit(G, 71)
    g[1000:1040] = g[999]                                  # 41 identical rows 999..1039
    g[5000:5030] = g[7] * (1 + 1e-4)                       # near-duplicates of row 7
    q[0] = g[999]
    q[1] = g[7]
    tags = torch.ones(G, dtype=torch.int32)
    tags[999:1011] = 2                                     # the lowest members of the tie group are ineligible
    tags[7] = 2
    tags[5000:5010] = 2
    idx = _index(e, g, tags=tags)
    got = run(lambda: idx.topk(q, K, tags=1))
    assert _same(got, _oracle(e, q, g, K, tags, [1] * Q))
    i = got[1].cpu()
    assert i[0, :29].tolist() == list(range(1011, 1040))
    assert 7 not in i[1].tolist() and not (i[1] >= 5000).logical_and(i[1] < 5010).any()


@pytest.mark.parametrize("K", [50, 200])
def test_exact_fallback_with_filter(eng, K):
    """Gallery sorted by increasing similarity to query 0: its eligible candidate list overflows and the exact scan, which skips
    ineligible rows, produces its list."""
    Q, G = 4, 60000
    q = _unit(Q, 80)
    base = _unit(G, 81)
    g = base[torch.argsort(base @ q[0])]
    tags = torch.where(torch.rand(G, generator=torch.Generator().manual_seed(82)) < 0.5, 1, 2).int()
    masks = torch.tensor([1, 2, 1, 3]).int()
    ex = torch.tensor([-1, -1, 5, -1]).int()
    ex[0] = int(torch.nonzero(tags == 1).flatten()[-1])    # query 0's best eligible row
    rows = torch.full((Q,), -7, dtype=torch.int32, device=eng.device)
    got = _index(eng, g, tags=tags).topk(q, K, exclude=ex, tags=masks, exact_rows=rows)
    assert _same(got, _oracle(eng, q, g, K, tags, masks, exclude=ex))
    rows = rows.cpu()
    assert rows[0] == 1 and set(rows.tolist()) <= {0, 1}
    assert bool((tags[got[1][0].long().cpu()] == 1).all())


@pytest.mark.parametrize("mode", ["tc", "fp32_path"])
def test_removal_growth_and_restore(mode):
    e, G, run = _setup(mode)
    Q, K, extra = 16, 100, 6000
    q, g_all = _unit(Q, 90), _unit(G + extra, 91)
    g = g_all[:G]
    idx = _index(e, g, capacity=G + extra)
    top1 = idx.topk(q, 1)[1].cpu().flatten()
    rand10 = torch.randperm(G, generator=torch.Generator().manual_seed(92))[: G // 10]
    idx.remove(top1).remove(rand10.numpy())
    tags = torch.full((G,), -1, dtype=torch.int32)
    tags[top1.long()] = 0
    tags[rand10] = 0
    assert torch.equal(idx.row_tags.cpu(), tags)
    got = run(lambda: idx.topk(q, K, tags=ALL))
    assert _same(got, _oracle(e, q, g, K, tags, [ALL] * Q))
    assert not np.isin(got[1].cpu().numpy(), top1.numpy()).any()
    idx.add(g_all[G:])                                     # default tags: every bit
    tags = torch.cat([tags, torch.full((extra,), -1, dtype=torch.int32)])
    got = run(lambda: idx.topk(q, K, tags=ALL))
    assert _same(got, _oracle(e, q, g_all, K, tags, [ALL] * Q))
    idx.set_tags([int(top1[0])], 1)                        # restore one removed row
    tags[top1[0]] = 1
    got = run(lambda: idx.topk(q, K, tags=ALL))
    assert _same(got, _oracle(e, q, g_all, K, tags, [ALL] * Q))
    assert int(top1[0]) in got[1][0].tolist()


def test_cuda_graph_follows_tag_and_mask_edits(eng):
    Q, G, K = 32, 50000, 50
    q, g = _unit(Q, 100), _unit(G, 101)
    dev = eng.device
    idx = _index(eng, g)
    masks = torch.full((Q,), -1, dtype=torch.int32, device=dev)
    q_s = q.to(dev)
    td, ti = torch.empty(Q, K, device=dev), torch.empty(Q, K, dtype=torch.int32, device=dev)
    rows = torch.zeros(Q, dtype=torch.int32, device=dev)
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        idx.topk(q_s, K, out=(td, ti), exact_rows=rows, tags=masks)
    torch.cuda.current_stream(dev).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        idx.topk(q_s, K, out=(td, ti), exact_rows=rows, tags=masks)
    gen = torch.Generator().manual_seed(102)
    for step in range(4):
        if step > 0:                                       # rewrite masks and row tags in place between replays
            masks.copy_(torch.randint(0, 8, (Q,), generator=gen).int())
            chg = torch.randperm(G, generator=gen)[: G // 4]
            idx.set_tags(chg.to(dev), torch.randint(0, 8, (chg.numel(),), generator=gen).int().to(dev))
        if step == 3:
            prev = ti[:, 0].cpu().numpy()                  # the previous replay's top-1 rows
            idx.remove(prev[prev >= 0])
        graph.replay()
        torch.cuda.synchronize(dev)
        want = _oracle(eng, q, g, K, idx.row_tags.cpu(), masks.cpu())
        assert _same((td, ti), want), step


def test_two_shards_and_sharded_index(eng):
    Q, G, K = 20, 50001, 100
    q, g = _unit(Q, 110), _unit(G, 111)
    tags = (1 << torch.randint(0, 3, (G,), generator=torch.Generator().manual_seed(112))).int()
    masks = torch.tensor([1, 2, 4, 3, 7] * (Q // 5)).int()
    ex = torch.randint(0, G, (Q,), generator=torch.Generator().manual_seed(113)).int()
    sched, D = cir.schedule, cir.distributed
    parts = []
    for r in range(2):
        s = sched.shard_rows(G, r, 2)
        parts.append(_index(eng, g[s], tags=tags[s]).topk(q, K, exclude=ex, col_offset=s.start, tags=masks))
    merged = eng.topk_merge(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]))
    whole_idx = _index(eng, g, tags=tags)
    whole = whole_idx.topk(q, K, exclude=ex, tags=masks)
    assert _same(merged, whole)
    assert _same(whole, _oracle(eng, q, g, K, tags, masks, exclude=ex))
    sharded = D.ShardedStage1Index(eng, G, lambda rows: g[rows], tags_of=lambda rows: tags[rows])
    assert _same(sharded.topk(q, K, exclude=ex, tags=masks), whole)
    gone = whole[1][:, :3].flatten().cpu()
    gone = gone[gone >= 0]
    sharded.remove(gone)
    whole_idx.remove(gone.numpy())
    assert _same(sharded.topk(q, K, exclude=ex, tags=masks), whole_idx.topk(q, K, exclude=ex, tags=masks))
    with pytest.raises(ValueError):
        sharded.remove([G])


def test_rejected_input(eng):
    G = 20000
    idx = _index(eng, _unit(G, 120), capacity=G + 10)
    q = _unit(3, 121).to(eng.device)
    lib = N.lib()
    td, ti = torch.empty(3, 10, device=eng.device), torch.empty(3, 10, dtype=torch.int32, device=eng.device)
    ws = torch.empty(lib.cir_stage1_index_topk_workspace_bytes(eng.ctx, C.byref(idx._s), 3, 10), dtype=torch.uint8, device=eng.device)
    masks = torch.ones(3, dtype=torch.int32, device=eng.device)
    eng._sync_stream()
    for rt, qm in ((N.vp(0), N.ptr(masks)), (N.ptr(idx._tags), N.vp(0))):
        with pytest.raises(N.CirError, match=r"rc=-1\).*row_tags and query_masks"):
            N.check(lib.cir_stage1_index_topk_filtered(eng.ctx, C.byref(idx._s), N.ptr(q), 3, rt, qm, N.vp(0), 0, 10, N.ptr(td),
                                                       N.ptr(ti), N.vp(0), N.ptr(ws), ws.numel()), "cir_stage1_index_topk_filtered")
    with pytest.raises(N.CirError, match=r"rc=-1\).*out of range"):
        idx.topk(q, 0, tags=1)
    with pytest.raises(N.CirError, match=r"rc=-3\)"):
        N.check(lib.cir_stage1_index_topk_filtered(eng.ctx, C.byref(idx._s), N.ptr(q), 3, N.ptr(idx._tags), N.ptr(masks), N.vp(0), 0,
                                                   10, N.ptr(td), N.ptr(ti), N.vp(0), N.ptr(ws), 256), "cir_stage1_index_topk_filtered")
    with pytest.raises(ValueError, match="expected 3 tags"):
        idx.topk(q, 10, tags=torch.ones(4, dtype=torch.int32, device=eng.device))
    with pytest.raises(TypeError, match="int32"):
        idx.topk(q, 10, tags=torch.ones(3, dtype=torch.int64, device=eng.device))
    for bad in ([1, 2, -1], [1, 1 << 32, 1], 1 << 32, -1):
        with pytest.raises(ValueError, match=r"\[0, 2\^32\)"):
            idx.topk(q, 10, tags=bad)
    with pytest.raises(ValueError, match="expected 5 tags"):
        idx.add(_unit(5, 122), tags=[1, 2])
    assert idx.rows == G
    with pytest.raises(ValueError, match="expected 2 tags"):
        idx.set_tags([0, 1], torch.ones(3, dtype=torch.int32))
    with pytest.raises(N.CirError, match="outside"):
        idx.remove([G])


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
        q, g = _unit(Q, 130).to(dev), _unit(G, 131)
        tags = (1 << torch.randint(0, 3, (G,), generator=torch.Generator().manual_seed(132))).int()
        masks = (1 << torch.randint(0, 3, (Q,), generator=torch.Generator().manual_seed(133))).int()
        sharded = cir.distributed.ShardedStage1Index(eng, G, lambda rows: g[rows], tags_of=lambda rows: tags[rows])
        assert sharded.index.rows == sharded.block.stop - sharded.block.start < G
        gone = torch.arange(0, G, 97)
        sharded.remove(gone)
        got = sharded.topk(q, K, tags=masks)
        tags[gone] = 0
        assert _same(got, _oracle(eng, q.cpu(), g, K, tags, masks))
        ret[rank] = "ok"
    except Exception as e:  # pragma: no cover
        ret[rank] = f"{type(e).__name__}: {e}"
        raise
    finally:
        dist.destroy_process_group()


def test_two_gpu_sharded_filtered_index_matches_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    assert dict(ret) == {0: "ok", 1: "ok"}
