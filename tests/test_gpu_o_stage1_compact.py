"""Compaction and subsets of the resident stage-I index (cir_stage1_index_compact, cir_stage1_index_topk_ids, Stage1Index.compact /
.subset): rows keep permanent ids, so a compaction changes no search result.  The oracle is the same index with every compaction
left out (a twin that receives the same adds, tag edits and removals), or stage1_topk over the eligible rows as in
test_gpu_n_stage1_filter; every comparison is bit for bit -- on the tensor-core path, the fp32 path, in an fp32 engine and below
16,384 rows, across the threshold between the two, for the per-query exact fallback, under CUDA-graph replay and sharded over ranks."""
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


def _removed_layout(G, seed):
    """Tags in three categories (1 / 2 / 4) with 10 % of the rows removed (tag 0)."""
    gen = torch.Generator().manual_seed(seed)
    tags = (1 << torch.randint(0, 3, (G,), generator=gen)).int()
    gone = torch.randperm(G, generator=gen)[: G // 10]
    return tags, gone


@pytest.mark.parametrize("mode", MODES)
def test_compact_after_removals_equals_filtered_search(mode):
    e, G, run = _setup(mode)
    Q, K, off = 24, 100, 700
    q, g = _unit(Q, 1), _unit(G, 2)
    tags, gone = _removed_layout(G, 3)
    idx, twin = _index(e, g, tags=tags), _index(e, g, tags=tags)
    top1 = idx.topk(q, 1)[1].cpu().flatten()
    idx.remove(gone.numpy()).remove(top1)
    twin.remove(gone.numpy()).remove(top1)
    kept = torch.nonzero(twin.row_tags.cpu() != 0).flatten()
    ex = torch.randint(0, G, (Q,), generator=torch.Generator().manual_seed(4)).int() + off
    ex[0::4] = -1                                          # none
    ex[1::4] = off + top1[1::4]                            # removed rows
    ex[2::4] = off + kept[torch.randint(0, kept.numel(), (Q // 4,), generator=torch.Generator().manual_seed(5))].int()   # kept rows
    masks = torch.tensor([1, 2, 4, 6, 7, ALL & 0x7FFFFFFF] * (Q // 6)).int()
    before = run(lambda: idx.topk(q, K, exclude=ex, col_offset=off, tags=ALL))
    before_m = run(lambda: idx.topk(q, K, exclude=ex, col_offset=off, tags=masks))
    idx.compact()
    assert idx.rows == kept.numel() and idx.next_id == G
    assert torch.equal(idx.row_ids.cpu().long(), kept)
    assert torch.equal(idx.row_tags.cpu(), tags[kept])
    plain = run(lambda: idx.topk(q, K, exclude=ex, col_offset=off))
    assert _same(plain, before)
    assert _same(run(lambda: idx.topk(q, K, exclude=ex, col_offset=off, tags=ALL)), before)
    assert _same(run(lambda: idx.topk(q, K, exclude=ex, col_offset=off, tags=masks)), before_m)
    assert _same(before_m, run(lambda: twin.topk(q, K, exclude=ex, col_offset=off, tags=masks)))
    assert _same(before, _oracle(e, q, g, K, twin.row_tags, [ALL] * Q, exclude=ex, col_offset=off))
    i = plain[1].cpu()
    for r in range(2, Q, 4):                               # the excluded kept row is not returned; it would be without exclude
        assert int(ex[r]) not in i[r].tolist()


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_blob_equals_fresh_add_of_kept_rows(precision):
    e = cir.engine.get_engine(precision=precision)
    G, cap = 30000, 32000
    g = _unit(G, 10)
    g[123] *= 3.0                                          # the largest row norm: removed, so the rebuilt maxima must shrink
    tags, gone = _removed_layout(G, 11)
    gone = torch.cat([gone, torch.tensor([123])])
    idx = _index(e, g, tags=tags, capacity=cap).remove(gone.numpy())
    kept = torch.nonzero(idx.row_tags.cpu() != 0).flatten()
    old_gmax = idx._blob[idx._s.gmax - idx._blob.data_ptr():][:8].clone()
    idx.compact()
    fresh = _index(e, g[kept], capacity=cap)
    n = kept.numel()
    assert idx.rows == fresh.rows == n and idx.capacity == cap
    assert torch.equal(idx._blob[: n * 1024], fresh._blob[: n * 1024])                     # fp32 rows
    if precision == "bf16":
        o = idx._s.g_bf16 - idx._blob.data_ptr()
        assert o == fresh._s.g_bf16 - fresh._blob.data_ptr()
        assert torch.equal(idx._blob[o:o + n * 512], fresh._blob[o:o + n * 512])            # bf16 rows
    else:
        assert not idx._s.g_bf16 and not fresh._s.g_bf16
    o = idx._s.gmax - idx._blob.data_ptr()
    gmax = idx._blob[o:o + 8]
    assert torch.equal(gmax, fresh._blob[fresh._s.gmax - fresh._blob.data_ptr():][:8])     # gmax of the kept rows only
    if precision == "bf16":
        assert not torch.equal(gmax, old_gmax)
    assert torch.equal(idx.row_tags.cpu(), tags[kept])
    assert torch.equal(idx.row_ids.cpu().long(), kept)
    assert torch.equal(idx.g_f32.cpu(), g[kept])


@pytest.mark.parametrize("mode", ["tc", "fp32_path"])
def test_subsets_fashion_iq(mode):
    """Three categories (tags 1 / 2 / 4, rows assigned at random) and the union 6: each subset searched without tags equals the
    parent's filtered search; a narrower mask on a subset equals the oracle over rows eligible under both masks."""
    e, G, run = _setup(mode)
    Q, K = 16, 200
    q, g = _unit(Q, 20), _unit(G, 21)
    tags = (1 << torch.randint(0, 3, (G,), generator=torch.Generator().manual_seed(22))).int()
    idx = _index(e, g, tags=tags)
    idx.remove(np.arange(0, G, 50))
    ex = torch.randint(0, G, (Q,), generator=torch.Generator().manual_seed(23)).int()
    ex[::3] = -1
    rt = idx.row_tags.cpu()
    for mask in (1, 2, 4, 6):
        sub = idx.subset(mask)
        elig = torch.nonzero((rt & mask) != 0).flatten()
        assert sub.rows == elig.numel() and torch.equal(sub.row_ids.cpu().long(), elig)
        assert torch.equal(sub.row_tags.cpu(), rt[elig]) and sub.next_id == G and sub.capacity == idx.capacity
        want = run(lambda: idx.topk(q, K, exclude=ex, tags=mask))
        assert _same(run(lambda: sub.topk(q, K, exclude=ex)), want), mask
        assert _same(run(lambda: sub.topk(q, K, exclude=ex, tags=ALL)), want), mask
    sub6 = idx.subset(6, capacity=int(((rt & 6) != 0).sum()))
    assert _same(run(lambda: sub6.topk(q, K, tags=2)), run(lambda: idx.topk(q, K, tags=2)))      # 2 lies inside 6
    masks = torch.tensor([2, 4, 1, 7] * (Q // 4)).int()
    got = run(lambda: sub6.topk(q, K, exclude=ex, tags=masks))
    assert _same(got, _oracle(e, q, g, K, rt & 6, masks, exclude=ex))
    assert (got[1].cpu()[masks == 1] == -1).all()
    assert idx.rows == G and torch.equal(idx.row_tags.cpu(), rt)       # the parent is unchanged


@pytest.mark.parametrize("mode", ["tc", "fp32_path"])
def test_growth_removal_and_ids_across_compactions(mode):
    """idx (compacted twice, capacity shrunk) and twin (never compacted) receive the same adds, removals and tag edits by id."""
    e, G, run = _setup(mode)
    Q, K, extra = 16, 100, 6000
    q, g_all = _unit(Q, 30), _unit(G + 2 * extra, 31)
    gen = torch.Generator().manual_seed(32)
    idx, twin = _index(e, g_all[:G], capacity=G), _index(e, g_all[:G], capacity=G + 2 * extra)
    masks = torch.tensor([ALL & 0x7FFFFFFF, 1, 3, 2] * (Q // 4)).int()

    def check(tag):
        ex = torch.randint(0, twin.rows, (Q,), generator=gen).int() + 9
        ex[::4] = -1
        for m in (ALL, masks):
            assert _same(run(lambda: idx.topk(q, K, exclude=ex, col_offset=9, tags=m)),
                         run(lambda: twin.topk(q, K, exclude=ex, col_offset=9, tags=m))), tag

    def both(fn):
        fn(idx)
        fn(twin)

    gone = torch.randperm(G, generator=gen)[: G // 5].numpy()
    both(lambda x: x.remove(gone))
    idx.compact(capacity=G - 2000)                         # shrink: 32,000 rows now, 38,000 after the first growth
    assert idx.rows == G - gone.size and idx.next_id == G and idx.capacity == G - 2000
    check("first compaction")
    both(lambda x: x.add(g_all[G:G + extra], tags=[1, 2] * (extra // 2)))
    assert torch.equal(idx.row_ids[-extra:].cpu(), torch.arange(G, G + extra, dtype=torch.int32)) and idx.next_id == G + extra
    check("growth")
    ids = np.setdiff1d(np.arange(G + extra), gone)[::7]
    both(lambda x: x.remove(ids[:200]))
    both(lambda x: x.set_tags(ids[200:400], 2))
    both(lambda x: x.set_tags(torch.from_numpy(ids[400:600]).cuda(), torch.full((200,), 1, dtype=torch.int32).cuda()))
    check("edits by id")
    before = idx.row_tags.clone()
    idx.remove(gone[:50])                                  # ids a compaction dropped: nothing happens
    idx.set_tags(torch.from_numpy(gone[:50]).int().cuda(), torch.full((50,), 5, dtype=torch.int32).cuda())
    assert torch.equal(idx.row_tags, before)
    with pytest.raises(ValueError, match="no longer in the index"):
        idx.set_tags(gone[:3], 1)
    with pytest.raises(N.CirError, match="outside"):
        idx.remove([G + extra])
    idx.compact(capacity=G + extra)                        # second compaction, growing the capacity: drops ids[:200]
    assert idx.rows == twin.rows - gone.size - 200
    check("second compaction")
    both(lambda x: x.add(g_all[G + extra:], tags=4))
    assert idx.next_id == G + 2 * extra
    check("growth after the second compaction")
    assert torch.equal(idx.row_ids.cpu().long(), torch.nonzero(twin.row_tags.cpu() != 0).flatten())


def test_threshold_crossing_and_zero_rows(eng):
    """20,000 rows (tensor-core path) compacted to 14,000 (fp32 path: under 16,384), then to none."""
    Q, G, K = 12, 20000, 100
    q, g = _unit(Q, 40), _unit(G, 41)
    idx, twin = _index(eng, g), _index(eng, g)
    gone = torch.randperm(G, generator=torch.Generator().manual_seed(42))[:6000].numpy()
    idx.remove(gone)
    twin.remove(gone)
    ex = torch.tensor([-1, 5, 17, 19999] * 3).int()
    idx.compact()
    assert idx.rows == 14000
    assert _same(idx.topk(q, K, exclude=ex), twin.topk(q, K, exclude=ex, tags=ALL))
    assert _same(idx.topk(q, K, exclude=ex, tags=ALL), _oracle(eng, q, g, K, twin.row_tags, [ALL] * Q, exclude=ex))
    idx.remove(np.arange(G))                               # every id, present or not
    idx.compact()
    assert idx.rows == 0 and idx.next_id == G
    for t in (None, ALL):
        d, i = idx.topk(q, K, exclude=ex, tags=t)
        assert (i.cpu() == -1).all() and torch.isinf(d.cpu()).all() and (d.cpu() > 0).all()
    empty = idx.subset(1)
    assert empty.rows == 0 and (empty.topk(q, K)[1].cpu() == -1).all()
    idx.add(g[:50])                                        # an index compacted to nothing grows again, ids from next_id
    assert torch.equal(idx.row_ids.cpu(), torch.arange(G, G + 50, dtype=torch.int32))
    d, i = idx.topk(q, K)
    d0, i0 = eng.stage1_topk(q, g[:50], K, col_offset=G)
    assert torch.equal(d.cpu(), d0.cpu()) and torch.equal(i.cpu(), i0.cpu())


@pytest.mark.parametrize("K", [50, 200])
def test_exact_fallback_on_compacted_index(eng, K):
    """Gallery sorted by increasing similarity to query 0: its candidate list overflows on the compacted index too, and the exact
    scan of the kept rows gives the same list as the filtered search of the uncompacted one."""
    Q, G = 4, 60000
    q = _unit(Q, 50)
    base = _unit(G, 51)
    g = base[torch.argsort(base @ q[0])]
    gone = torch.randperm(G, generator=torch.Generator().manual_seed(52))[: G * 3 // 10]
    gone = torch.cat([gone, torch.tensor([G - 2])])       # one of query 0's best rows
    idx, twin = _index(eng, g), _index(eng, g)
    idx.remove(gone.numpy())
    twin.remove(gone.numpy())
    ex = torch.tensor([G - 1, -1, 5, G - 2]).int()
    rows = torch.full((Q,), -7, dtype=torch.int32, device=eng.device)
    want = twin.topk(q, K, exclude=ex, tags=ALL)
    idx.compact()
    got = idx.topk(q, K, exclude=ex, exact_rows=rows)
    assert _same(got, want)
    assert _same(want, _oracle(eng, q, g, K, twin.row_tags, [ALL] * Q, exclude=ex))
    rows = rows.cpu()
    assert rows[0] == 1 and set(rows.tolist()) <= {0, 1}


def test_cuda_graph_after_compaction(eng):
    Q, G, K = 32, 50000, 50
    q, g = _unit(Q, 60), _unit(G, 61)
    dev = eng.device
    idx, twin = _index(eng, g), _index(eng, g)
    gone = np.arange(0, G, 3)
    idx.remove(gone)
    twin.remove(gone)
    idx.compact()
    masks = torch.full((Q,), -1, dtype=torch.int32, device=dev)
    ex = torch.randint(0, G, (Q,), generator=torch.Generator().manual_seed(62)).int().to(dev)
    q_s = q.to(dev)
    td, ti = torch.empty(Q, K, device=dev), torch.empty(Q, K, dtype=torch.int32, device=dev)
    rows = torch.zeros(Q, dtype=torch.int32, device=dev)
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        idx.topk(q_s, K, exclude=ex, out=(td, ti), exact_rows=rows, tags=masks)
    torch.cuda.current_stream(dev).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        idx.topk(q_s, K, exclude=ex, out=(td, ti), exact_rows=rows, tags=masks)
    gen = torch.Generator().manual_seed(63)
    for step in range(4):
        if step > 0:                                       # rewrite masks and row tags (by id, on the device) between replays
            masks.copy_(torch.randint(0, 8, (Q,), generator=gen).int())
            chg = torch.randperm(G, generator=gen)[: G // 4].to(dev)
            new = torch.randint(0, 8, (chg.numel(),), generator=gen).int().to(dev)
            idx.set_tags(chg, new)
            twin.set_tags(chg[torch.from_numpy(~np.isin(chg.cpu().numpy(), gone)).to(dev)],
                          new[torch.from_numpy(~np.isin(chg.cpu().numpy(), gone)).to(dev)])
        if step == 3:
            prev = ti[:, 0].cpu().numpy()
            idx.remove(torch.from_numpy(prev[prev >= 0]).to(dev))
            twin.remove(prev[prev >= 0])
        graph.replay()
        torch.cuda.synchronize(dev)
        assert _same((td, ti), twin.topk(q, K, exclude=ex, tags=masks)), step


def test_two_shards_and_sharded_index(eng):
    Q, G, K = 20, 50001, 100
    q, g = _unit(Q, 70), _unit(G, 71)
    tags = (1 << torch.randint(0, 3, (G,), generator=torch.Generator().manual_seed(72))).int()
    masks = torch.tensor([1, 2, 4, 3, 7] * (Q // 5)).int()
    ex = torch.randint(0, G, (Q,), generator=torch.Generator().manual_seed(73)).int()
    gone = torch.randperm(G, generator=torch.Generator().manual_seed(74))[: G // 8]
    whole = _index(eng, g, tags=tags).remove(gone.numpy())
    want = whole.topk(q, K, exclude=ex, tags=masks)
    sched, D = cir.schedule, cir.distributed
    parts = []
    for r in range(2):                                     # two compacted shards on one GPU, ids local, col_offset = shard start
        s = sched.shard_rows(G, r, 2)
        mine = gone[(gone >= s.start) & (gone < s.stop)] - s.start
        shard = _index(eng, g[s], tags=tags[s]).remove(mine.numpy()).compact()
        parts.append(shard.topk(q, K, exclude=ex, col_offset=s.start, tags=masks))
    assert _same(eng.topk_merge(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts])), want)
    sharded = D.ShardedStage1Index(eng, G, lambda rows: g[rows], tags_of=lambda rows: tags[rows])     # world size 1
    sharded.remove(gone)
    before = sharded.topk(q, K, exclude=ex, tags=masks)
    sharded.compact()
    assert sharded.index.rows == G - gone.numel() and sharded.col_offset == 0
    assert _same(sharded.topk(q, K, exclude=ex, tags=masks), before)
    assert _same(before, want)
    more = want[1][:, :3].flatten().cpu()
    more = more[more >= 0]
    sharded.remove(more)
    whole.remove(more.numpy())
    assert _same(sharded.topk(q, K, exclude=ex, tags=masks), whole.topk(q, K, exclude=ex, tags=masks))
    sharded.compact()
    assert _same(sharded.topk(q, K, exclude=ex, tags=ALL), whole.topk(q, K, exclude=ex, tags=ALL))


def test_rejected_input(eng):
    lib = N.lib()
    G = 20000
    g = _unit(G, 80)
    src = _index(eng, g, capacity=G + 10).remove(np.arange(0, G, 2))
    ws = torch.empty(1 << 20, dtype=torch.uint8, device=eng.device)

    def compact(dst, dst_tags=None, dst_ids=None, ctx=None, nbytes=None):
        dt = dst._tags if dst_tags is None else dst_tags
        di = torch.full((dst.capacity + 1,), -7, dtype=torch.int32, device=eng.device) if dst_ids is None else dst_ids
        eng._sync_stream()
        N.check(lib.cir_stage1_index_compact(eng.ctx if ctx is None else ctx, C.byref(src._s), N.ptr(src._tags), N.vp(0), ALL,
                                             C.byref(dst._s), N.ptr(dt), N.ptr(di), N.ptr(ws), ws.numel() if nbytes is None else nbytes),
                "cir_stage1_index_compact")

    same_blob = N.Stage1Index(src._s.capacity, 0, src._s.g_f32, src._s.g_bf16, src._s.gmax)
    alias = eng.stage1_index(1)
    alias._s = same_blob
    with pytest.raises(N.CirError, match=r"rc=-1\).*overlap"):
        compact(alias)
    small = eng.stage1_index(100)
    small._blob.fill_(0x5A)
    ids = torch.full((101,), -7, dtype=torch.int32, device=eng.device)
    with pytest.raises(N.CirError, match=r"rc=-1\).*exceed the capacity 100"):
        compact(small, dst_ids=ids)
    assert small.rows == 0 and bool((small._blob == 0x5A).all()) and bool((small._tags == -1).all()) and bool((ids == -7).all())
    full = _index(eng, g[:10], capacity=G)
    with pytest.raises(N.CirError, match=r"rc=-1\).*must be an empty index"):
        compact(full)
    other = cir.engine.get_engine(precision="fp32").stage1_index(G)
    with pytest.raises(N.CirError, match=r"rc=-1\).*dtype"):
        compact(other)
    with pytest.raises(N.CirError, match=r"rc=-3\)"):
        compact(eng.stage1_index(G), nbytes=16)
    assert src.rows == G and src.next_id == G
    # ids that do not fit int32 indices
    idx = _index(eng, g[:100]).compact()
    q = _unit(3, 81).to(eng.device)
    with pytest.raises(N.CirError, match=r"rc=-1\).*do not fit int32"):
        idx.topk(q, 10, col_offset=(1 << 31) - 50)
    idx.topk(q, 10, col_offset=(1 << 31) - 100)            # the last id, 99, maps to 2^31 - 1
    td, ti = torch.empty(3, 10, device=eng.device), torch.empty(3, 10, dtype=torch.int32, device=eng.device)
    need = lib.cir_stage1_index_topk_ids_workspace_bytes(eng.ctx, C.byref(idx._s), 3, 10)
    assert need == -(-lib.cir_stage1_index_topk_workspace_bytes(eng.ctx, C.byref(idx._s), 3, 10) // 256) * 256 + 256
    for rt, qm in ((N.vp(0), N.ptr(idx._tags)), (N.ptr(idx._tags), N.vp(0))):
        with pytest.raises(N.CirError, match=r"rc=-1\).*both NULL"):
            N.check(lib.cir_stage1_index_topk_ids(eng.ctx, C.byref(idx._s), N.ptr(q), 3, N.ptr(idx._ids), idx.next_id, rt, qm, N.vp(0), 0,
                                                  10, N.ptr(td), N.ptr(ti), N.vp(0), N.ptr(ws), ws.numel()), "topk_ids")
    with pytest.raises(N.CirError, match=r"rc=-3\)"):
        N.check(lib.cir_stage1_index_topk_ids(eng.ctx, C.byref(idx._s), N.ptr(q), 3, N.ptr(idx._ids), idx.next_id, N.vp(0), N.vp(0),
                                              N.vp(0), 0, 10, N.ptr(td), N.ptr(ti), N.vp(0), N.ptr(ws), need - 256), "topk_ids")
    idx._next_id = (1 << 31) - 2
    with pytest.raises(N.CirError, match="do not fit int32"):
        idx.add(g[:5])
    assert idx.rows == 100


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
        q, g = _unit(Q, 90).to(dev), _unit(G, 91)
        tags = (1 << torch.randint(0, 3, (G,), generator=torch.Generator().manual_seed(92))).int()
        masks = (1 << torch.randint(0, 3, (Q,), generator=torch.Generator().manual_seed(93))).int()
        ex = torch.randint(0, G, (Q,), generator=torch.Generator().manual_seed(94)).int()
        sharded = cir.distributed.ShardedStage1Index(eng, G, lambda rows: g[rows], tags_of=lambda rows: tags[rows])
        gone = torch.arange(0, G, 7)
        sharded.remove(gone)
        before = sharded.topk(q, K, exclude=ex, tags=masks)
        sharded.compact()
        assert sharded.index.rows < sharded.block.stop - sharded.block.start
        got = sharded.topk(q, K, exclude=ex, tags=masks)
        assert _same(got, before)
        tags[gone] = 0
        assert _same(got, _oracle(eng, q.cpu(), g, K, tags, masks, exclude=ex))
        ret[rank] = "ok"
    except Exception as e:  # pragma: no cover
        ret[rank] = f"{type(e).__name__}: {e}"
        raise
    finally:
        dist.destroy_process_group()


def test_two_gpu_sharded_compaction_matches_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    assert dict(ret) == {0: "ok", 1: "ok"}
