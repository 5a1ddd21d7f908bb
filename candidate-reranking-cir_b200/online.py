"""The online query path of a retrieve-then-re-rank system, entirely on the device:

    reference image + caption --stage-I encode--> (z_t, q_emb) --Stage1Index.topk--> top-k ids --stage2_rerank_cached--> re-ranked ids

Stage I encodes the query once (cir_stage1_encode returns both the token states z_t that stage II reads and the query embedding
q_emb), searches the resident gallery index (optionally filtered by per-query tag masks) and hands its device top-k list straight
to the stage-II re-ranker over the resident K/V gallery.  Nothing is read back to the host, so :meth:`OnlineReranker.capture`
can record the whole chain as one CUDA graph and replay it for new queries.
"""
from __future__ import annotations

from typing import List, Optional

import torch

from . import native as N
from .engine import Stage1Index, Stage2KVCache


class OnlineReranker:
    """``m1`` / ``m2``: the stage-I / stage-II models (BLIP_Retrieval, BLIP_NLVR) on one device; ``gallery_tokens`` act [G,N,768]:
    the tokens the query's reference image is read from (row ref_index[q]); ``index``: the stage-I gallery index searched with the
    query embeddings; ``kv_cache``: the stage-II K/V gallery of ``m2`` holding every row the index can return.  ``normalize_twice``
    as in cir_stage1_encode (src/validate.py:311)."""

    def __init__(self, m1, m2, gallery_tokens: torch.Tensor, index: Stage1Index, kv_cache: Stage2KVCache, normalize_twice: bool = False):
        m1._need_weights()
        m2._need_weights()
        if m1.engine.device != m2.engine.device or index.eng.device != m2.engine.device:
            raise N.CirError("OnlineReranker: the models, the index and the cache must share one device")
        kv_cache._check_use(m2.engine, m2._w, gallery_tokens.shape[1])
        self.m1, self.m2, self.tokens, self.index, self.kv_cache = m1, m2, gallery_tokens, index, kv_cache
        self.normalize_twice = normalize_twice
        self._ws: Optional[torch.Tensor] = None      # stage-I encode workspace, owned: Engine.workspace may be reallocated
        self._retired: List[torch.Tensor] = []       # outgrown workspaces stay alive: a captured graph may still point at one

    def _encode_ws(self, Q: int, L: int) -> torch.Tensor:
        eng = self.m1.engine
        need = eng._lib.cir_stage1_workspace_bytes(eng.ctx, Q, L, self.tokens.shape[1])
        if self._ws is None or self._ws.numel() < need:
            if self._ws is not None:
                self._retired.append(self._ws)
            self._ws = torch.empty(max(need, 256), dtype=torch.uint8, device=eng.device)
        return self._ws

    def __call__(self, ref_index, ids, mask, k: int, tags=None, out=None):
        """ref_index int [Q] (row of ``gallery_tokens``, excluded from the query's top-k), ids / mask int [Q,L], ``tags``: optional
        per-query masks for a filtered search (see Stage1Index.topk) -> (ranked ids int32 [Q,k], stage-II scores fp32 [Q,k] in
        stage-I order, stage-I distances fp32 [Q,k]).  A short filtered list pads with id -1, which scores -99999.99 and ranks last.
        ``out``: optional (ranked, scores, order, dist, idx) to fill.  Never synchronises."""
        eng1, eng2 = self.m1.engine, self.m2.engine
        ref_index, ids, mask = eng1._i32(ref_index), eng1._i32(ids), eng1._i32(mask)
        Q, L = ids.shape
        z_t, q_emb = eng1.stage1_encode(self.m1._w, self.tokens, ref_index, ids, mask, want_z=True, want_emb=True,
                                        normalize_twice=self.normalize_twice, workspace=self._encode_ws(Q, L))
        ranked, scores, order, dist, idx = (None,) * 5 if out is None else out
        dist, idx = self.index.topk(q_emb, k, exclude=ref_index, tags=tags, out=None if dist is None else (dist, idx))
        s2_out = None if ranked is None else (scores, order, ranked)
        scores, _, ranked = eng2.stage2_rerank_cached(self.m2._w, self.kv_cache, z_t, ids, mask, idx, out=s2_out)
        return ranked, scores, dist

    def capture(self, Q: int, L: int, k: int, tags: bool = False) -> "CapturedQuery":
        """Record the chain for Q queries of L tokens and top-k lists as one CUDA graph (see :class:`CapturedQuery`)."""
        return CapturedQuery(self, Q, L, k, tags)


class CapturedQuery:
    """The online chain of an :class:`OnlineReranker` recorded as one CUDA graph, with static input buffers ``ref_index`` int32 [Q],
    ``ids`` / ``mask`` int32 [Q,L] and, when captured with ``tags=True``, the per-query tag masks ``tags`` int32 [Q].  Calling it
    copies new inputs in, replays the graph and returns (ranked ids, stage-II scores, stage-I distances): views of static output
    buffers that the next replay overwrites.

    Like a captured index search, the graph sees the rows and tags the index holds at replay; rows added after the capture are not
    searched.  After ``index.compact()`` (a new blob) the graph must be captured again, as must one whose model weights or cache
    were replaced."""

    def __init__(self, chain: OnlineReranker, Q: int, L: int, k: int, tags: bool = False):
        dev = chain.m2.engine.device
        self.chain, self.k = chain, k
        self.ref_index = torch.zeros(Q, dtype=torch.int32, device=dev)
        self.ids = torch.zeros(Q, L, dtype=torch.int32, device=dev)
        self.mask = torch.ones(Q, L, dtype=torch.int32, device=dev)
        self.tags = torch.full((Q,), -1, dtype=torch.int32, device=dev) if tags else None
        i32 = dict(dtype=torch.int32, device=dev)
        self._out = (torch.empty(Q, k, **i32), torch.empty(Q, k, dtype=torch.float32, device=dev), torch.empty(Q, k, **i32),
                     torch.empty(Q, k, dtype=torch.float32, device=dev), torch.empty(Q, k, **i32))
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):             # warm-up: workspaces, kernel attributes and lazy module loads before capture
            self._run()
        torch.cuda.current_stream(dev).wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._result = self._run()

    def _run(self):
        return self.chain(self.ref_index, self.ids, self.mask, self.k, tags=self.tags, out=self._out)

    def __call__(self, ref_index, ids, mask, tags=None):
        """Copy the new inputs into the static buffers, replay -> (ranked ids int32 [Q,k], scores fp32 [Q,k], dist fp32 [Q,k])."""
        self.ref_index.copy_(torch.as_tensor(ref_index).reshape(self.ref_index.shape), non_blocking=True)
        self.ids.copy_(torch.as_tensor(ids).reshape(self.ids.shape), non_blocking=True)
        self.mask.copy_(torch.as_tensor(mask).reshape(self.mask.shape), non_blocking=True)
        if self.tags is not None:
            if tags is None:
                raise ValueError("CapturedQuery: captured with tags, so every call needs the per-query masks")
            self.tags.copy_(self.chain.index._tag_tensor(tags, self.tags.numel(), "CapturedQuery tags"), non_blocking=True)
        elif tags is not None:
            raise ValueError("CapturedQuery: captured without tags")
        self.graph.replay()
        return self._result
