"""Row-sharded corpus search across the GPUs of one box (SURVEY.md §8e).

Rank g owns documents [g*ceil(N/G), (g+1)*ceil(N/G)); every rank scans its own shard (no data-path communication),
then ONE collective — an all-gather of the per-shard top-(k+1) ``(score fp32, global id int64)`` lists,
Q*(k+1)*12 bytes per rank — followed by the same merge kernel the single-GPU chunk loop uses.  This is the reference's
sequential "chunk, top-k, heapq.nlargest merge" (exact_search.py:80-132) with "chunk" = "shard".  The only collective
the reference itself has is the padded embedding all-gather of sentence_transformers/util.py:326-347, whose role
(combine per-rank partial results) this takes over.  Works with the ``nccl`` backend on GPUs and — for the host-side
logic tests — with ``gloo`` on CPU tensors when a ``local_search`` callable is supplied.
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import torch
import torch.distributed as dist


def shard_range(n_docs: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous row range of `rank`: [rank*ceil(N/G), min(N, (rank+1)*ceil(N/G)))."""
    per = (n_docs + world - 1) // world
    lo = min(n_docs, rank * per)
    return lo, min(n_docs, lo + per)


def all_gather_topk(scores: torch.Tensor, ids: torch.Tensor, group=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """[Q,k] per rank -> [G,Q,k] on every rank (scores fp32, ids int64): the two-tensor form used with CPU stand-ins
    (gloo tests) and by callers that hold unpacked lists.  The GPU path uses ONE exchange of packed 8-byte entries
    (`all_gather_packed` over NCCL, or no collective at all: `PeerGather`)."""
    world = dist.get_world_size(group)
    Q, k = scores.shape
    # concatenated-along-dim-0 output layout is the one both nccl and gloo accept
    gs = torch.empty((world * Q, k), dtype=scores.dtype, device=scores.device)
    gi = torch.empty((world * Q, k), dtype=ids.dtype, device=ids.device)
    dist.all_gather_into_tensor(gs, scores.contiguous(), group=group)
    dist.all_gather_into_tensor(gi, ids.contiguous(), group=group)
    return gs.view(world, Q, k), gi.view(world, Q, k)


def all_gather_packed(packed: torch.Tensor, group=None) -> torch.Tensor:
    """Packed per-shard top-k int64 [Q,k] (CorpusShard.search_packed) -> [G,Q,k] on every rank: the single
    Q*(k+1)*8-byte-per-rank all-gather of SURVEY.md §8e."""
    world = dist.get_world_size(group)
    Q, k = packed.shape
    out = torch.empty((world * Q, k), dtype=packed.dtype, device=packed.device)
    dist.all_gather_into_tensor(out, packed.contiguous(), group=group)
    return out.view(world, Q, k)


class PeerGather:
    """Cross-GPU exchange of the per-shard top-k WITHOUT a collective call (include/sgpt_b200.h: sgpt_gather_*): every
    rank's final selection kernel stores its list into every rank's gather buffer through NVLink peer mappings and
    signals per query; the merge kernel waits on those signals.  torch.distributed only carries the 64-byte CUDA IPC
    handles at construction time.  Every rank must call `search` with the same number of queries, in the same order."""

    def __init__(self, nq_cap: int, k: int, device, group=None):
        import ctypes as C

        from . import _lib

        self.group, self.device = group, torch.device(device)
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.nq_cap, self.k = int(nq_cap), int(k)
        self._lib = _lib.lib()
        handle = C.c_void_p()
        mine = C.create_string_buffer(_lib.IPC_HANDLE_BYTES)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.sgpt_gather_create(self.rank, self.world, self.nq_cap, self.k, C.byref(handle), mine),
                       "sgpt_gather_create")
            self._handle = handle
            if self.world > 1:
                every = [None] * self.world
                dist.all_gather_object(every, bytes(mine.raw), group=group)
                blob = C.create_string_buffer(b"".join(every), _lib.IPC_HANDLE_BYTES * self.world)
                _lib.check(self._lib.sgpt_gather_connect(self._handle, blob), "sgpt_gather_connect")
                dist.barrier(group)  # nobody pushes into a buffer its owner has not finished mapping/zeroing

    def search(self, shard, queries: torch.Tensor, k: int, score_function: str = "cos_sim",
               exclude_ids: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """Local exact top-k of `shard` (CorpusShard) -> push to all ranks -> merge.  Identical (scores fp32 [Q,k], ids
        int64 [Q,k]) on every rank."""
        from . import _lib

        qb, q_scale, c_scale = shard._prepare(queries, k, score_function)
        nq = qb.shape[0]
        out_s = torch.empty((nq, k), dtype=torch.float32, device=self.device)
        out_i = torch.empty((nq, k), dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self._lib.sgpt_search_gather_ex(self._handle, qb.data_ptr(), shard.vectors.data_ptr(),
                                                 _lib.ptr(q_scale), c_scale, nq, shard.n, shard.dim, k, shard.id_base,
                                                 _lib.ptr(exclude_ids), out_s.data_ptr(), out_i.data_ptr(),
                                                 shard._ws.data_ptr(), shard._ws.numel(), shard._elem,
                                                 _lib.current_stream())
        _lib.check(rc, "sgpt_search_gather_ex")
        return out_s, out_i

    def close(self):
        if getattr(self, "_handle", None):
            torch.cuda.synchronize(self.device)
            if self.world > 1:
                dist.barrier(self.group)  # no peer is still storing into this rank's buffer
            self._lib.sgpt_gather_destroy(self._handle)
            self._handle = None


def sharded_search(query_emb: torch.Tensor, shard, k: int, score_function: str = "cos_sim",
                   exclude_ids: Optional[torch.Tensor] = None, group=None,
                   merge: Optional[Callable] = None, gather: Optional["PeerGather"] = None
                   ) -> Tuple[torch.Tensor, torch.Tensor]:
    """Every rank: local exact top-k over its shard -> exchange -> merge.  Returns identical (scores, ids) [Q,k] on all
    ranks, ids being global document rows.  `shard` is a CorpusShard (or anything with .search(q, k, score_function)).
    Exchange: `gather` (PeerGather: kernel-to-kernel over NVLink, no collective) when given; otherwise one NCCL
    all-gather of packed 8-byte entries + the packed merge kernel; with an injected `merge` (CPU stand-ins on gloo)
    the two-tensor all-gather."""
    if gather is not None:
        return gather.search(shard, query_emb, k, score_function, exclude_ids)
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    if merge is None and hasattr(shard, "search_packed"):
        from .index import merge_topk_packed

        packed = shard.search_packed(query_emb, k, score_function)
        return merge_topk_packed(all_gather_packed(packed, group) if multi else packed.unsqueeze(0), exclude_ids)
    local_s, local_i = shard.search(query_emb, k, score_function)
    gs, gi = all_gather_topk(local_s, local_i, group) if multi else (local_s.unsqueeze(0), local_i.unsqueeze(0))
    if merge is None:
        from .index import merge_topk as merge
    return merge(gs, gi, exclude_ids)


class ShardedDenseRetrievalExactSearch:
    """``DenseRetrievalExactSearch.search`` (exact_search.py:34-134) across the ranks of one ``torch.distributed`` group.

    Every rank holds a replica of the embedder.  Queries are encoded by every rank (cheap, and it keeps the result
    available everywhere); the corpus is sorted by length like the reference (XS:66-70) and dealt out ``i mod G`` over
    the ranks, so every rank encodes the same mix of long and short documents (SURVEY.md §8e).  Rank g encodes only its
    documents into one resident ``CorpusShard``, scans it once, and the per-rank top-(k+1) lists meet in one all-gather
    followed by the merge kernel — the reference's "chunk, top-k, heapq merge" with chunk = rank.  Every rank returns the
    same ``Dict[qid, Dict[cid, float]]``.  ``shard_factory(dim, capacity)`` / ``merge`` default to ``CorpusShard`` and the
    CUDA merge kernel; the CPU tests inject stand-ins and run it on ``gloo``.
    """

    def __init__(self, model, batch_size: int = 128, corpus_chunk_size: int = 50000, group=None,
                 shard_factory: Optional[Callable] = None, merge: Optional[Callable] = None, peer_gather: bool = False,
                 corpus_dtype: str = "bf16", **kwargs):
        self.model, self.batch_size, self.corpus_chunk_size = model, batch_size, corpus_chunk_size
        self.corpus_dtype = corpus_dtype  # element type of the resident shards: "bf16" or "int8" (CorpusShard dtype)
        self.group, self.shard_factory, self.merge = group, shard_factory, merge
        self.peer_gather = peer_gather  # exchange through NVLink peer mappings (PeerGather) instead of one NCCL all-gather
        self.show_progress_bar, self.convert_to_tensor = True, True
        self.results = {}
        self.device = getattr(model, "device", torch.device("cuda:0"))

    def _world(self):
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(self.group), dist.get_world_size(self.group)
        return 0, 1

    def search(self, corpus, queries, top_k: int, score_function: str, return_sorted: bool = False, **kwargs):
        from .index import _check_score_function

        _check_score_function(score_function)
        rank, world = self._world()
        query_ids = list(queries.keys())
        self.results = {qid: {} for qid in query_ids}
        q_emb = torch.as_tensor(self.model.encode_queries(
            [(qid, queries[qid]) for qid in query_ids], batch_size=self.batch_size,
            show_progress_bar=self.show_progress_bar, convert_to_tensor=self.convert_to_tensor)).to(self.device).float()
        corpus_ids = sorted(corpus, key=lambda k: len(corpus[k].get("title", "") + corpus[k].get("text", "")),
                            reverse=True)
        row_of = {cid: i for i, cid in enumerate(corpus_ids)}
        mine = corpus_ids[rank::world]  # global sorted row of local row j is rank + j * world
        cap = max((len(corpus_ids) + world - 1) // world, 1)  # rows per rank (the longest deal)
        gpu_path = self.shard_factory is None
        if gpu_path:
            from .index import CorpusShard

            # the shard numbers its rows rank * cap + j, so a merged id still names its owner: (id // cap, id % cap)
            shard = CorpusShard(q_emb.shape[1], max(len(mine), 1), device=self.device, id_base=rank * cap,
                                dtype=self.corpus_dtype)
        else:
            shard = self.shard_factory(q_emb.shape[1], max(len(mine), 1))
        for batch_num, start in enumerate(range(0, len(mine), self.corpus_chunk_size)):
            chunk = [(cid, corpus[cid]) for cid in mine[start:start + self.corpus_chunk_size]]
            shard.add(torch.as_tensor(self.model.encode_corpus(
                chunk, batch_size=self.batch_size, show_progress_bar=self.show_progress_bar,
                convert_to_tensor=self.convert_to_tensor, batch_num=f"{rank}_{batch_num}")).to(self.device).float())
        kk = top_k + 1
        if gpu_path and self.merge is None:
            rows = [row_of.get(qid, -1) for qid in query_ids]  # self match (XS:118) in the shard id space
            exclude = torch.tensor([(r % world) * cap + r // world if r >= 0 else -1 for r in rows], dtype=torch.int64,
                                   device=self.device)
            gather = PeerGather(len(query_ids), kk, self.device, self.group) if (self.peer_gather and world > 1) else None
            s, i = sharded_search(q_emb, shard, kk, score_function, exclude_ids=exclude, group=self.group, gather=gather)
            if gather is not None:
                gather.close()
            to_row = lambda sid: (sid % cap) * world + sid // cap  # noqa: E731
        else:
            exclude = torch.tensor([row_of.get(qid, -1) for qid in query_ids], dtype=torch.int64, device=self.device)
            s, i = shard.search(q_emb, kk, score_function)
            i = torch.where(i >= 0, i * world + rank, i)  # local row -> row in the global length-sorted order
            if world > 1:
                gs, gi = all_gather_topk(s, i, self.group)
            else:
                gs, gi = s.unsqueeze(0), i.unsqueeze(0)
            merge = self.merge
            if merge is None:
                from .index import merge_topk as merge
            s, i = merge(gs, gi, exclude)
            to_row = lambda sid: sid  # noqa: E731
        for qi, (srow, irow) in enumerate(zip(s.cpu().tolist(), i.cpu().tolist())):
            res = self.results[query_ids[qi]]
            for score, sid in zip(srow, irow):
                if sid >= 0:
                    res[corpus_ids[to_row(sid)]] = score
        return self.results
