"""Corpus shard in HBM + exact top-k search over it (rows S1–S3 of SURVEY.md §8a).

A shard holds the embeddings of a contiguous range of documents as a bf16 matrix [n, D] (read once per search at
HBM speed) plus fp32 1/||row|| of the STORED rows, so cosine scores are exactly ``cos_sim`` of the stored vectors
(sentence_transformers/util.py:24-43) and dot scores are exactly ``dot_score`` (:46-63).

``dtype="int8"`` stores every row as int8 codes with one fp32 scale per row (symmetric per-row quantization,
include/sgpt_b200.h ``sgpt_quantize_rows_i8``): half the HBM and half the bytes every search reads.  Queries are quantized
the same way, and the scores are exactly cos_sim / dot_score of the dequantized rows ``scale * codes``.
"""
from __future__ import annotations

import json
import os
from typing import Dict, List, Optional, Tuple, Union

import numpy as np
import torch

from . import _lib

SCORE_FUNCTIONS = ("cos_sim", "dot")


def _check_score_function(score_function: str) -> None:
    if score_function not in SCORE_FUNCTIONS:
        # same message as biencoder/beir/custommodels/exact_search.py:46-51
        raise ValueError(
            "score function: {} must be either (cos_sim) for cosine similarity or (dot) for dot product".format(
                score_function))


def to_bf16_rows(x: torch.Tensor) -> torch.Tensor:
    """fp32 [n, D] (device) -> bf16 [n, D] (round-to-nearest-even) with the library's conversion kernel."""
    x = x.contiguous()
    assert x.dtype == torch.float32 and x.is_cuda and x.numel() % 4 == 0
    out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().sgpt_f32_to_bf16(x.data_ptr(), out.data_ptr(), x.numel(), _lib.current_stream()))
    return out


def quantize_rows_i8(x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """fp32 or bf16 rows [n, D] (device) -> (int8 codes [n, D], scale fp32 [n], 1/||codes|| fp32 [n]) with the library's
    quantization kernel (per row: scale = max|x| / 127, codes = clamp(rint(x / scale), -127, 127))."""
    x = x.contiguous()
    assert x.is_cuda and x.dtype in (torch.float32, torch.bfloat16) and x.dim() == 2
    n, D = x.shape
    out = torch.empty((n, D), dtype=torch.int8, device=x.device)
    scale = torch.empty(n, dtype=torch.float32, device=x.device)
    inv = torch.empty(n, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().sgpt_quantize_rows_i8(x.data_ptr(), int(x.dtype == torch.bfloat16), n, D, out.data_ptr(),
                                                    scale.data_ptr(), inv.data_ptr(), _lib.current_stream()),
                   "sgpt_quantize_rows_i8")
    return out, scale, inv


def row_inv_norms(x_bf16: torch.Tensor) -> torch.Tensor:
    n, D = x_bf16.shape
    out = torch.empty(n, dtype=torch.float32, device=x_bf16.device)
    with torch.cuda.device(x_bf16.device):
        _lib.check(_lib.lib().sgpt_row_inv_norms(x_bf16.data_ptr(), out.data_ptr(), n, D, _lib.current_stream()))
    return out


DTYPES = ("bf16", "int8")


class CorpusShard:
    """Documents [id_base, id_base + n) of a corpus, resident in the HBM of one GPU.

    ``dtype="bf16"``: ``vectors`` bf16 [capacity, D] and ``inv_norms`` fp32.  ``dtype="int8"``: ``vectors`` int8 codes
    [capacity, D], ``scales`` fp32 (one per row) and ``inv_norms`` fp32 = 1/||codes||; D must be a multiple of 16."""

    def __init__(self, dim: int, capacity: int, device="cuda:0", id_base: int = 0, dtype: str = "bf16"):
        if dtype not in DTYPES:
            raise ValueError(f"shard dtype must be one of {DTYPES}, got {dtype!r}")
        if dim % 8 != 0:
            raise ValueError("embedding dimension must be a multiple of 8")
        if dtype == "int8" and (dim % 16 != 0 or dim > 65536):
            raise ValueError("an int8 shard needs an embedding dimension that is a multiple of 16 and at most 65536")
        self.dim, self.capacity, self.id_base, self.dtype = int(dim), int(capacity), int(id_base), dtype
        self.device = torch.device(device)
        self.vectors = torch.empty((self.capacity, self.dim), dtype=torch.int8 if dtype == "int8" else torch.bfloat16,
                                   device=self.device)
        self.inv_norms = torch.empty(self.capacity, dtype=torch.float32, device=self.device)
        self.scales = torch.empty(self.capacity, dtype=torch.float32, device=self.device) if dtype == "int8" else None
        self.n = 0
        self._ws: Optional[torch.Tensor] = None

    @property
    def _elem(self) -> int:
        return _lib.ELEM_I8 if self.dtype == "int8" else _lib.ELEM_BF16

    @classmethod
    def from_embeddings(cls, emb: torch.Tensor, device=None, id_base: int = 0, dtype: str = "bf16") -> "CorpusShard":
        device = device or emb.device
        shard = cls(emb.shape[1], emb.shape[0], device=device, id_base=id_base, dtype=dtype)
        shard.add(emb)
        return shard

    def add(self, emb: torch.Tensor) -> None:
        """Append fp32 (or bf16) embeddings [m, D]; they are stored bf16-rounded, or quantized to int8 rows (an int8 shard
        rejects non-finite values with ValueError: such a row has no scale)."""
        m = emb.shape[0]
        if self.n + m > self.capacity:
            raise ValueError(f"shard capacity {self.capacity} exceeded ({self.n} + {m})")
        emb = emb.to(self.device)
        if self.dtype == "int8":
            if not bool(torch.isfinite(emb).all()):
                raise ValueError("an int8 shard cannot store non-finite embedding values (NaN / inf)")
            codes, scale, inv = quantize_rows_i8(emb if emb.dtype == torch.bfloat16 else emb.float())
            self.vectors[self.n:self.n + m].copy_(codes)
            self.scales[self.n:self.n + m].copy_(scale)
            self.inv_norms[self.n:self.n + m].copy_(inv)
            self.n += m
            return
        rows = emb if emb.dtype == torch.bfloat16 else to_bf16_rows(emb.float())
        self.vectors[self.n:self.n + m].copy_(rows)
        self.inv_norms[self.n:self.n + m].copy_(row_inv_norms(self.vectors[self.n:self.n + m]))
        self.n += m

    def stored(self) -> torch.Tensor:
        return self.vectors[:self.n]

    # ---- persistence (replaces the pickle-per-chunk embedding cache of BDR:311-323, 336-342) ----------------------
    def save(self, path: str) -> None:
        """Write the shard as ``path/{vectors.npy (bf16 bit patterns as uint16), inv_norms.npy, meta.json}``; one
        directory per rank for a sharded corpus.  An int8 shard writes int8 ``vectors.npy`` plus ``scales.npy``."""
        os.makedirs(path, exist_ok=True)
        if self.dtype == "int8":
            np.save(os.path.join(path, "vectors.npy"), self.stored().cpu().numpy())
            np.save(os.path.join(path, "scales.npy"), self.scales[:self.n].cpu().numpy())
        else:
            np.save(os.path.join(path, "vectors.npy"), self.stored().view(torch.int16).cpu().numpy().view(np.uint16))
        np.save(os.path.join(path, "inv_norms.npy"), self.inv_norms[:self.n].cpu().numpy())
        with open(os.path.join(path, "meta.json"), "w") as f:
            json.dump({"format": "sgpt_b200.CorpusShard/1", "dtype": self.dtype, "dim": self.dim, "n": self.n,
                       "id_base": self.id_base}, f)

    @classmethod
    def load(cls, path: str, device="cuda:0", capacity: Optional[int] = None) -> "CorpusShard":
        """Reload a shard written by ``save`` (bit-identical vectors and norms, so identical search results)."""
        with open(os.path.join(path, "meta.json")) as f:
            meta = json.load(f)
        dtype = meta.get("dtype")
        if meta.get("format") != "sgpt_b200.CorpusShard/1" or dtype not in DTYPES:
            raise ValueError(f"{path}: not a CorpusShard directory ({meta})")
        vec = np.load(os.path.join(path, "vectors.npy"), mmap_mode="r")
        inv = np.load(os.path.join(path, "inv_norms.npy"))
        n, dim = int(meta["n"]), int(meta["dim"])
        want = np.int8 if dtype == "int8" else np.uint16
        if vec.shape != (n, dim) or vec.dtype != want or inv.shape != (n,):
            raise ValueError(f"{path}: array shapes {vec.shape}/{inv.shape} do not match meta {meta}")
        shard = cls(dim, max(n, capacity or n), device=device, id_base=int(meta["id_base"]), dtype=dtype)
        if dtype == "int8":
            scales = np.load(os.path.join(path, "scales.npy"))
            if scales.shape != (n,):
                raise ValueError(f"{path}: scales.npy shape {scales.shape} does not match meta {meta}")
            shard.vectors[:n].copy_(torch.from_numpy(np.array(vec)))
            shard.scales[:n].copy_(torch.from_numpy(scales))
        else:
            shard.vectors[:n].copy_(torch.from_numpy(np.array(vec).view(np.int16)).view(torch.bfloat16))
        shard.inv_norms[:n].copy_(torch.from_numpy(inv))
        shard.n = n
        return shard

    def _prepare(self, queries: torch.Tensor, k: int, score_function: str):
        """Queries -> rows of the shard's element type + their scale factor + the shard's (device address) + a workspace
        large enough for this search.  bf16: 1/||q|| and 1/||d|| for cos_sim, none for dot.  int8: 1/||codes|| for
        cos_sim, the quantization scales for dot."""
        _check_score_function(score_function)
        q = queries.to(self.device)
        cos = score_function == "cos_sim"
        if self.dtype == "int8":
            if not bool(torch.isfinite(q).all()):
                raise ValueError("queries against an int8 shard must be finite")
            qb, q_s, q_inv = quantize_rows_i8(q if q.dtype == torch.bfloat16 else q.float())
            q_scale, c_scale = (q_inv, self.inv_norms) if cos else (q_s, self.scales)
        else:
            qb = q.contiguous() if q.dtype == torch.bfloat16 else to_bf16_rows(q.float())
            q_scale = row_inv_norms(qb) if cos else None
            c_scale = self.inv_norms if cos else None
        need = _lib.lib().sgpt_search_workspace_bytes(qb.shape[0], self.n, k)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        return qb, q_scale, _lib.ptr(c_scale)

    def search(self, queries: torch.Tensor, k: int, score_function: str = "cos_sim") -> Tuple[torch.Tensor, torch.Tensor]:
        """Exact top-k of this shard for fp32/bf16 queries [Q, D] (device).

        Returns (scores fp32 [Q,k] descending, global ids int64 [Q,k]); when the shard has fewer than k documents the
        tail is (-inf, -1).  Queries are rounded to bf16 (the tensor-core input type); their 1/||q|| is taken from the
        rounded rows so the result equals cos_sim of the stored/rounded vectors evaluated in fp32.  Against an int8
        shard the queries are quantized like the corpus rows and the scores are those of the dequantized rows.
        """
        qb, q_scale, c_scale = self._prepare(queries, k, score_function)
        nq = qb.shape[0]
        out_s = torch.empty((nq, k), dtype=torch.float32, device=self.device)
        out_i = torch.empty((nq, k), dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            rc = _lib.lib().sgpt_search_ex(qb.data_ptr(), self.vectors.data_ptr(), _lib.ptr(q_scale), c_scale, nq,
                                           self.n, self.dim, k, self.id_base, out_s.data_ptr(), out_i.data_ptr(),
                                           self._ws.data_ptr(), self._ws.numel(), self._elem, _lib.current_stream())
        _lib.check(rc, "sgpt_search_ex")
        return out_s, out_i

    def search_packed(self, queries: torch.Tensor, k: int, score_function: str = "cos_sim") -> torch.Tensor:
        """The same search with the result as ONE tensor of packed 8-byte entries, int64 [Q,k] whose low 32 bits are the
        fp32 score and high 32 bits the int32 global id (-inf / -1 = empty): what a rank contributes to the single
        all-gather of a sharded search (SURVEY.md §8e).  Needs id_base + n < 2^31."""
        qb, q_scale, c_scale = self._prepare(queries, k, score_function)
        nq = qb.shape[0]
        out = torch.empty((nq, k), dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            rc = _lib.lib().sgpt_search_packed_ex(qb.data_ptr(), self.vectors.data_ptr(), _lib.ptr(q_scale), c_scale,
                                                  nq, self.n, self.dim, k, self.id_base, out.data_ptr(),
                                                  self._ws.data_ptr(), self._ws.numel(), self._elem,
                                                  _lib.current_stream())
        _lib.check(rc, "sgpt_search_packed_ex")
        return out


def unpack_topk(packed: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Packed entries int64[...] -> (scores fp32[...], ids int64[...]) (host-side convenience for tests and tools)."""
    halves = packed.contiguous().view(torch.int32).view(*packed.shape, 2)
    return halves[..., 0].contiguous().view(torch.float32), halves[..., 1].to(torch.int64)


def merge_topk_packed(packed: torch.Tensor, exclude_ids: Optional[torch.Tensor] = None
                      ) -> Tuple[torch.Tensor, torch.Tensor]:
    """Merge G packed candidate lists per query: int64 [G,Q,k] -> (scores fp32 [Q,k], ids int64 [Q,k]) descending;
    empty slots and ids == exclude_ids[q] (XS:118) are dropped."""
    G, Q, k = packed.shape
    packed = packed.contiguous()
    out_s = torch.empty((Q, k), dtype=torch.float32, device=packed.device)
    out_i = torch.empty((Q, k), dtype=torch.int64, device=packed.device)
    with torch.cuda.device(packed.device):
        rc = _lib.lib().sgpt_topk_merge_packed(packed.data_ptr(), G, Q, k, out_s.data_ptr(), out_i.data_ptr(),
                                               _lib.ptr(exclude_ids), _lib.current_stream())
    _lib.check(rc, "sgpt_topk_merge_packed")
    return out_s, out_i


def merge_topk(scores: torch.Tensor, ids: torch.Tensor, exclude_ids: Optional[torch.Tensor] = None
               ) -> Tuple[torch.Tensor, torch.Tensor]:
    """Merge G candidate lists per query: scores fp32 [G,Q,k], ids int64 [G,Q,k] -> ([Q,k], [Q,k]) descending.
    Entries with id < 0, or id == exclude_ids[q] (int64 [Q], the XS:118 self-match rule), are dropped."""
    G, Q, k = scores.shape
    scores, ids = scores.contiguous(), ids.contiguous()
    out_s = torch.empty((Q, k), dtype=torch.float32, device=scores.device)
    out_i = torch.empty((Q, k), dtype=torch.int64, device=scores.device)
    with torch.cuda.device(scores.device):
        rc = _lib.lib().sgpt_topk_merge(scores.data_ptr(), ids.data_ptr(), G, Q, k, out_s.data_ptr(), out_i.data_ptr(),
                                        _lib.ptr(exclude_ids), None, _lib.current_stream())
    _lib.check(rc, "sgpt_topk_merge")
    return out_s, out_i


def semantic_search(query_embeddings: torch.Tensor, corpus_embeddings: Union[torch.Tensor, CorpusShard],
                    query_chunk_size: int = 100, corpus_chunk_size: int = 500000, top_k: int = 10,
                    score_function="cos_sim", device="cuda:0") -> List[List[Dict[str, Union[int, float]]]]:
    """``sentence_transformers.util.semantic_search`` (ST/util.py:197-258) on the fused exact search: for every query
    the ``top_k`` corpus entries as ``{"corpus_id", "score"}`` dicts, best first.  ``score_function`` is "cos_sim" /
    "dot" or the reference's ``cos_sim`` / ``dot_score`` callables (recognised by name); the chunk sizes of the reference
    are accepted and ignored — the kernel streams the whole shard once and needs no score-matrix chunks."""
    del query_chunk_size, corpus_chunk_size
    if callable(score_function):
        score_function = {"cos_sim": "cos_sim", "pytorch_cos_sim": "cos_sim", "dot_score": "dot"}.get(
            getattr(score_function, "__name__", ""), None)
    _check_score_function(score_function)
    q = torch.as_tensor(query_embeddings)
    if q.dim() == 1:
        q = q.unsqueeze(0)  # ST/util.py:214-217
    shard = corpus_embeddings if isinstance(corpus_embeddings, CorpusShard) else CorpusShard.from_embeddings(
        torch.as_tensor(corpus_embeddings).to(device))
    k = min(int(top_k), shard.n)
    scores, ids = shard.search(q.to(shard.device), k, score_function)
    scores, ids = scores.cpu().tolist(), ids.cpu().tolist()
    return [[{"corpus_id": int(i), "score": float(s)} for s, i in zip(srow, irow) if i >= 0]
            for srow, irow in zip(scores, ids)]
