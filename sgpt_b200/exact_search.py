"""DenseRetrievalExactSearch — drop-in for biencoder/beir/custommodels/exact_search.py:22-134 ("XS").

Same constructor, attributes and ``search`` contract (``Dict[qid, Dict[cid, float]]`` with up to top_k+1 entries per
query, ValueError on an unknown score function), but the per-chunk work — scores, NaN fix, top-(k+1), self-match drop
and the cross-chunk merge — stays on the GPU: one Python dict is built at the very end instead of Q x chunks x 1001
Python-level dict operations and a ``heapq.nlargest`` per query per chunk (XS:112-132).
"""
from __future__ import annotations

import logging
from typing import Dict, List, Optional

import numpy as np
import torch

from .index import CorpusShard, _check_score_function, merge_topk

logger = logging.getLogger(__name__)


class DenseRetrievalExactSearch:
    def __init__(self, model, batch_size: int = 128, corpus_chunk_size: int = 50000, plain_lists: bool = False,
                 corpus_dtype: str = "bf16", **kwargs):
        """model is any class that provides encode_corpus() and encode_queries() (XS:24).  ``plain_lists=False`` is the
        reference's custom convention — ``[(id, text)]`` / ``[(id, {title, text})]`` tuples and a ``batch_num`` keyword
        (XS:56-62, 87-93); ``plain_lists=True`` is upstream beir's DRES convention — ``List[str]`` /
        ``List[{title, text}]`` — which the ST-path wrappers (SentenceBERTBOSEOS / SentenceBERTAsym, used with
        ``beir.retrieval.search.dense.DenseRetrievalExactSearch`` at BDR:405-412) expect.  ``corpus_dtype`` is the
        element type the corpus chunks are searched in: "bf16" or "int8" (per-row int8 rows, see CorpusShard)."""
        self.model = model
        self.corpus_dtype = corpus_dtype
        self.plain_lists = plain_lists
        self.batch_size = batch_size
        self.score_functions = {"cos_sim": "cos_sim", "dot": "dot"}
        self.score_function_desc = {"cos_sim": "Cosine Similarity", "dot": "Dot Product"}
        self.corpus_chunk_size = corpus_chunk_size
        self.show_progress_bar = True
        self.convert_to_tensor = True
        self.results: Dict[str, Dict[str, float]] = {}
        self.device = getattr(model, "device", torch.device("cuda:0"))

    def _as_device(self, emb) -> torch.Tensor:
        if isinstance(emb, np.ndarray):
            emb = torch.from_numpy(emb)
        return emb.to(self.device, dtype=torch.float32)

    def search(self, corpus: Dict[str, Dict[str, str]], queries: Dict[str, str], top_k: int, score_function: str,
               return_sorted: bool = False, **kwargs) -> Dict[str, Dict[str, float]]:
        _check_score_function(score_function)  # XS:46-51
        logger.info("Encoding Queries...")
        query_ids = list(queries.keys())
        self.results = {qid: {} for qid in query_ids}
        query_list = [queries[qid] if self.plain_lists else (qid, queries[qid]) for qid in queries]  # XS:56
        q_emb = self._as_device(self.model.encode_queries(
            query_list, batch_size=self.batch_size, show_progress_bar=self.show_progress_bar,
            convert_to_tensor=self.convert_to_tensor))

        logger.info("Sorting Corpus by document length (Longest first)...")
        corpus_ids = sorted(corpus, key=lambda k: len(corpus[k].get("title", "") + corpus[k].get("text", "")),
                            reverse=True)  # XS:66-70
        corpus_list = [corpus[cid] if self.plain_lists else (cid, corpus[cid]) for cid in corpus_ids]
        # XS:118 drops corpus_id == query_id: as a per-query global row index (or -1) so the GPU merge can apply it
        row_of = {cid: i for i, cid in enumerate(corpus_ids)}
        exclude = torch.tensor([row_of.get(qid, -1) for qid in query_ids], dtype=torch.int64, device=self.device)

        logger.info("Encoding Corpus in batches... Warning: This might take a while!")
        logger.info("Scoring Function: {} ({})".format(self.score_function_desc[score_function], score_function))
        kk = top_k + 1
        nq = len(query_ids)
        run_s = torch.full((nq, kk), float("-inf"), dtype=torch.float32, device=self.device)
        run_i = torch.full((nq, kk), -1, dtype=torch.int64, device=self.device)
        starts = range(0, len(corpus_list), self.corpus_chunk_size)
        for batch_num, start in enumerate(starts):
            logger.info("Encoding Batch {}/{}...".format(batch_num + 1, len(starts)))
            end = min(start + self.corpus_chunk_size, len(corpus_list))
            extra = {} if self.plain_lists else {"batch_num": batch_num}
            sub = self._as_device(self.model.encode_corpus(
                corpus_list[start:end], batch_size=self.batch_size, show_progress_bar=self.show_progress_bar,
                convert_to_tensor=self.convert_to_tensor, **extra))
            shard = CorpusShard.from_embeddings(sub, device=self.device, id_base=start, dtype=self.corpus_dtype)
            # XS:96-108: scores, NaN -> -1, top-(k+1) of this chunk
            s, i = shard.search(q_emb, kk, score_function)
            # XS:112-132: drop self matches, merge with the running lists, keep the best k+1
            run_s, run_i = merge_topk(torch.stack([run_s, s]), torch.stack([run_i, i]), exclude)
        scores = run_s.cpu().tolist()
        ids = run_i.cpu().tolist()
        for qi, qid in enumerate(query_ids):
            res = self.results[qid]
            for cid_idx, score in zip(ids[qi], scores[qi]):
                if cid_idx >= 0:
                    res[corpus_ids[cid_idx]] = score
        return self.results


def search_shard_embeddings(query_emb: torch.Tensor, shard: CorpusShard, top_k: int, score_function: str = "cos_sim"):
    """Top-(k+1) of pre-computed embeddings against one resident shard (the inner step of ``search``)."""
    return shard.search(query_emb, top_k + 1, score_function)
