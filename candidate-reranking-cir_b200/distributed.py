"""Multi-GPU sharding of the hot path: one process per GPU (torchrun), ``torch.distributed`` for the
plumbing.  The path shards without any data-path collective (SURVEY 8e): stage-II triplets are
independent, the stage-I gallery splits by rows; ranks exchange only (score, index) pairs:

  stage II : (a) candidate-range partition (default for N > 1): z_t is computed for a block of queries per rank and
             all-gathered; the candidate-sorted triplet list is cut into N contiguous candidate ranges
             (schedule.candidate_partition), so each gallery image's K/V projections are computed on ONE rank and the
             per-GPU K/V reuse does not fall with N; ranks all-gather (flat position, score) pairs -- 12 bytes per triplet --
             and every rank fills and re-sorts the [Q, K] matrix.
             (b) query partition: each rank scores its [Q_r, K] block (K/V of a candidate recomputed on every rank whose
             queries name it); one all-gather of the padded score blocks.
  stage I  : gallery rows block-partitioned; each rank computes a local top-K with global column ids
             (``col_offset``); one all-gather of [Q, K] (distance, index) lists; ``cir_topk_merge``.  ``ShardedStage1Index``
             keeps each rank's block resident (built once from that block only) for repeated query batches.

The compute steps are injected callables so the same code runs under ``gloo`` on CPU in the tests
(with the oracle standing in for the kernels) and under ``nccl`` on GPUs (with the engine).
"""
from __future__ import annotations

from typing import Callable, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

from .schedule import shard_rows


def world() -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def all_gather_rows(local: torch.Tensor, total_rows: int) -> torch.Tensor:
    """Concatenate per-rank row blocks produced by ``shard_rows`` (block sizes differ by at most one
    row: pad to the largest, gather, strip)."""
    rank, ws = world()
    if ws == 1:
        return local
    sizes = [shard_rows(total_rows, r, ws) for r in range(ws)]
    mx = max(s.stop - s.start for s in sizes)
    pad = torch.zeros((mx,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[: local.shape[0]] = local
    out = [torch.empty_like(pad) for _ in range(ws)]
    dist.all_gather(out, pad)
    return torch.cat([o[: s.stop - s.start] for o, s in zip(out, sizes)], dim=0)


def sharded_stage2_scores(score_fn: Callable[[slice], torch.Tensor], num_queries: int) -> torch.Tensor:
    """``score_fn(rows)`` -> fp32 [rows, K] scores of this rank's query block; returns the full [Q, K]
    matrix on every rank (8 bytes per triplet cross NVLink once sorted indices are added)."""
    rank, ws = world()
    rows = shard_rows(num_queries, rank, ws)
    local = score_fn(rows)
    assert local.shape[0] == rows.stop - rows.start
    return all_gather_rows(local, num_queries)


def sharded_stage2_scores_by_candidate(pairs_fn: Callable[[Optional[Tuple[int, int]]], Tuple[torch.Tensor, torch.Tensor, Sequence[int]]],
                                       num_queries: int, k: int, fill: float) -> torch.Tensor:
    """``pairs_fn(part)`` with ``part = (rank, world)`` (None when single-process) -> (flat_pos int64 [n], scores fp32 [n],
    part_sizes: triplets of EVERY rank, computable locally because the partition is deterministic).  One padded all-gather
    of positions and one of scores; every rank returns the full [Q, K] matrix, unscored slots = ``fill``."""
    rank, ws = world()
    pos, sc, sizes = pairs_fn((rank, ws) if ws > 1 else None)
    total = num_queries * k
    out = torch.full((total + 1,), fill, dtype=torch.float32, device=sc.device)     # slot `total` swallows the padding
    if ws == 1:
        out.index_copy_(0, pos, sc)
        return out[:total].view(num_queries, k)
    assert len(sizes) == ws and int(sizes[rank]) == pos.numel()
    mx = max(int(n) for n in sizes)
    ppos = torch.full((mx,), total, dtype=torch.int64, device=pos.device)
    psc = torch.zeros(mx, dtype=torch.float32, device=sc.device)
    ppos[: pos.numel()] = pos
    psc[: sc.numel()] = sc
    gpos = torch.empty(ws * mx, dtype=torch.int64, device=pos.device)
    gsc = torch.empty(ws * mx, dtype=torch.float32, device=sc.device)
    dist.all_gather_into_tensor(gpos, ppos)
    dist.all_gather_into_tensor(gsc, psc)
    out.index_copy_(0, gpos, gsc)
    out[total] = fill
    return out[:total].view(num_queries, k)


def sharded_stage1_topk(local_topk_fn: Callable[[slice], Tuple[torch.Tensor, torch.Tensor]],
                        merge_fn: Callable[[torch.Tensor, torch.Tensor], Tuple[torch.Tensor, torch.Tensor]],
                        gallery_rows: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """``local_topk_fn(rows)`` -> (dist [Q,K], idx [Q,K] with GLOBAL gallery ids) over this rank's gallery
    shard; ``merge_fn(dist [P,Q,K], idx [P,Q,K])`` -> merged lists.  Every rank gets the merged top-K."""
    rank, ws = world()
    rows = shard_rows(gallery_rows, rank, ws)
    d, i = local_topk_fn(rows)
    if ws == 1:
        return d, i
    ds = torch.empty((ws,) + tuple(d.shape), dtype=d.dtype, device=d.device)          # gathered straight into [P, Q, K]
    is_ = torch.empty((ws,) + tuple(i.shape), dtype=i.dtype, device=i.device)
    dist.all_gather_into_tensor(ds.view(-1, *d.shape[1:]), d.contiguous())            # (concatenation along dim 0: what gloo accepts too)
    dist.all_gather_into_tensor(is_.view(-1, *i.shape[1:]), i.contiguous())
    return merge_fn(ds, is_)


# ---- engine-backed convenience wrappers (GPU) ---------------------------------------------------------------

def encode_queries_sharded(m1, gallery_tokens, ref_idx, ids, mask) -> torch.Tensor:
    """z_t of all Q queries on every rank: each rank encodes its block of queries (stage-I encoder on the reference image's
    tokens), one all-gather of the [Q_r, L, 768] blocks (49 KB per query at L = 32)."""
    rank, ws = world()
    rows = shard_rows(len(ref_idx), rank, ws)
    z_loc, _ = m1.encode_queries(gallery_tokens, ref_idx[rows], ids[rows], mask[rows], want_z=True, want_emb=False)
    return all_gather_rows(z_loc, len(ref_idx))


def score_matrix_sharded(m2, gallery_tokens, z_all, ids, mask, cand_idx, row_active=None, kv_cache=None) -> torch.Tensor:
    """Stage-II scores of all Q*K triplets, candidate-range partitioned over the ranks -> [Q, K] on every rank.
    ``kv_cache``: this rank's Stage2KVCache; it must cover the candidates of the rank's share (e.g. the whole gallery)."""
    import numpy as np
    from .engine import NEG_FILL
    cand_np = cand_idx.cpu().numpy() if isinstance(cand_idx, torch.Tensor) else np.asarray(cand_idx)
    Q, K = cand_np.shape

    def pairs(part):
        pos, sc = m2.engine.stage2_score_pairs(m2._w, gallery_tokens, z_all, ids, mask, cand_np, row_active, part=part,
                                               kv_cache=kv_cache)
        return pos, sc, m2.engine.last_plan["part_sizes"]
    return sharded_stage2_scores_by_candidate(pairs, Q, K, NEG_FILL)


def stage2_scores_gpu(m1, m2, gallery_tokens, ref_idx, ids, mask, cand_idx, row_active=None, mode: str = "candidate") -> torch.Tensor:
    """z_t + stage-II scores of all Q*K triplets over the ranks of the default process group -> [Q, K] on every rank.
    mode "candidate": candidate-range partition (K/V of an image on one rank); "query": query-block partition."""
    import numpy as np
    cand_np = cand_idx.cpu().numpy() if isinstance(cand_idx, torch.Tensor) else np.asarray(cand_idx)
    if mode == "candidate":
        z_all = encode_queries_sharded(m1, gallery_tokens, ref_idx, ids, mask)
        return score_matrix_sharded(m2, gallery_tokens, z_all, ids, mask, cand_np, row_active)
    assert mode == "query"

    def score(rows: slice):
        z_t, _ = m1.encode_queries(gallery_tokens, ref_idx[rows], ids[rows], mask[rows], want_z=True, want_emb=False)
        act = None if row_active is None else np.asarray(row_active)[rows]
        return m2.score_triplets(z_t, ids[rows], mask[rows], gallery_tokens, cand_np[rows], act)
    return sharded_stage2_scores(score, cand_np.shape[0])


def stage1_topk_gpu(engine, q_emb, g_emb, k: int, exclude=None):
    def local(rows: slice):
        return engine.stage1_topk(q_emb, g_emb[rows], k, exclude=exclude, col_offset=rows.start)
    return sharded_stage1_topk(local, engine.topk_merge, g_emb.shape[0])


class ShardedStage1Index:
    """Resident stage-I index over the ranks of the default process group: each rank indexes only its ``shard_rows`` block of
    the gallery, searches it with ``col_offset = block.start`` (global row ids), and the lists meet in ``sharded_stage1_topk``
    + ``topk_merge``.  No rank holds the full gallery.  ``rows_of(block)`` -> fp32 [len(block), 256] gallery rows of that block
    (e.g. a slice of ``extract_index_features`` output, or rows read from storage); ``tags_of(block)`` (optional) -> their row
    tags (see ``Stage1Index.add``)."""

    def __init__(self, engine, gallery_rows: int, rows_of: Callable[[slice], torch.Tensor],
                 tags_of: Optional[Callable[[slice], object]] = None):
        rank, ws = world()
        self.engine, self.gallery_rows = engine, gallery_rows
        self.block = shard_rows(gallery_rows, rank, ws)
        self.index = engine.stage1_index(self.block.stop - self.block.start)
        self.index.add(rows_of(self.block), tags=None if tags_of is None else tags_of(self.block))
        self.col_offset = self.block.start        # global id of the rank's row id 0: block.start, 0 once compact() made ids global

    def topk(self, q_emb, k: int, exclude=None, tags=None) -> Tuple[torch.Tensor, torch.Tensor]:
        """-> merged (dist [Q,k], idx [Q,k]) on every rank; ``q_emb``, ``exclude`` (global row ids) and the query masks ``tags``
        (optional, see ``Stage1Index.topk``) cover all Q queries."""
        def local(rows: slice):
            assert rows == self.block
            return self.index.topk(q_emb, k, exclude=exclude, col_offset=self.col_offset, tags=tags)
        return sharded_stage1_topk(local, self.engine.topk_merge, self.gallery_rows)

    def remove(self, global_rows) -> None:
        """Remove gallery rows (global row ids, the same list on every rank): each rank removes those in its block."""
        g = global_rows.cpu() if isinstance(global_rows, torch.Tensor) else global_rows
        g = np.asarray(g, dtype=np.int64).reshape(-1)
        if g.size and (g.min() < 0 or g.max() >= self.gallery_rows):
            raise ValueError(f"remove: rows outside [0, {self.gallery_rows})")
        mine = g[(g >= self.block.start) & (g < self.block.stop)]
        self.index.remove(mine - self.col_offset)

    def compact(self) -> None:
        """Each rank drops the removed rows of its block (``Stage1Index.compact``).  The rank's row ids become the global rows
        (block.start + local row), so it then searches with col_offset 0; results, ``remove`` and the merge are unchanged."""
        self.index._compact(None, self.col_offset)
        self.col_offset = 0
