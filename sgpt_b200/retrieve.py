"""`python -m sgpt_b200.retrieve` — the retrieval run of biencoder/beir/beir_dense_retriever.py:352-498 on the B200 path.

Same flags (BDR:31-96), same flow (load BEIR split -> drop empty documents -> build the embedder + exact search ->
retrieve top-1000 -> write ``results_<model>_<method>_<dataset>.json`` -> NDCG/MAP/Recall/P into
``beir_embeddings_ndcgs.json`` incl. the CQADupStack average), with ``sgpt_b200.CustomEmbedder`` /
``DenseRetrievalExactSearch`` in place of the reference classes and ``sgpt_b200.beir_compat`` in place of the absent
``beir`` package.  Not carried over: dataset download (no network here: the dataset directory must exist) and the two
result-post-processing modes ``--computeavg`` / ``--selectbest`` (BDR:506-640; offline JSON aggregation, not part of
the retrieval path).
"""
from __future__ import annotations

import argparse
import json
import logging
import os

from .beir_compat import EvaluateRetrieval, GenericDataLoader

logger = logging.getLogger(__name__)

CQADUPSTACK_DATASETS = ["android", "english", "gaming", "gis", "mathematica", "physics", "programmers", "stats",
                        "wordpress", "webmasters", "unix", "tex"]  # BDR:469-482


def parse_args(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--dataset", type=str, default="scifact", help="Dataset to embed.")
    p.add_argument("--modelname", type=str, default="bert-base-uncased", help="Model to use.")
    p.add_argument("--method", type=str, default="mean", help="Method to use.")
    p.add_argument("--device", type=str, default="cuda:0", help="Device to use.")
    p.add_argument("--layeridx", type=int, default=-1, help="Layer to use: -1 is the last.")
    p.add_argument("--usest", action="store_const", default=False, const=True, help="Load a sentence-transformers model")
    p.add_argument("--datapath", type=str, default="./datasets/", help="Path to folder with datasets")
    p.add_argument("--overwrite", action="store_const", default=False, const=True,
                   help="Whether to recompute & overwrite existing results")
    p.add_argument("--batchsize", type=int, default=250, help="How many requests to batch")
    p.add_argument("--saveemb", action="store_const", default=False, const=True, help="Whether to save embeddings")
    p.add_argument("--speca", action="store_const", default=False, const=True, help="Use special token a encoding method")
    p.add_argument("--specb", action="store_const", default=False, const=True, help="Use special brackets encoding method")
    p.add_argument("--maxseqlen", type=int, default=None, help="Sequence length to use; SGPT-msmarco-specb models use 300")
    p.add_argument("--outdir", type=str, default=".", help="Where the result JSON files are written (reference: cwd)")
    p.add_argument("--corpusdtype", type=str, default="bf16", choices=["bf16", "int8"],
                   help="Element type of the searched corpus embeddings: bf16, or int8 rows with one scale per row")
    return p.parse_args(argv)


def clean_titles(corpus):  # BDR:500-504
    for k in corpus:
        if "title" in corpus[k] and corpus[k]["title"] is None:
            corpus[k]["title"] = ""
    return corpus


def build_retriever(args):
    """BDR:392-430: the ST path wraps the model for upstream beir's call convention, the HF path uses CustomEmbedder."""
    from . import CustomEmbedder, DenseRetrievalExactSearch, SentenceBERTAsym, SentenceBERTBOSEOS, SentenceEncoder

    if args.usest:
        model = SentenceEncoder.from_pretrained(args.modelname, device=args.device, batch_capacity=max(args.batchsize, 1),
                                                max_seq_length=args.maxseqlen)
        if "asym" in args.modelname:
            logger.info("Using asymmetric model.")
            wrapped = SentenceBERTAsym(model)
        elif args.speca or args.specb:
            wrapped = SentenceBERTBOSEOS(model, speca=args.speca, specb=args.specb)
        else:
            wrapped = _PlainSentenceBERT(model)
        wrapped.device = model.device
        return DenseRetrievalExactSearch(wrapped, batch_size=args.batchsize, plain_lists=True,
                                         corpus_dtype=args.corpusdtype)
    if args.speca:
        raise ValueError("speca is only supported with use_st")  # BDR:415-416
    return DenseRetrievalExactSearch(CustomEmbedder(
        model_name=args.modelname, method=args.method, device=args.device, batch_size=args.batchsize,
        save_emb=args.saveemb, layeridx=args.layeridx, specb=args.specb, maxseqlen=args.maxseqlen, dataset=args.dataset),
        corpus_dtype=args.corpusdtype)


class _PlainSentenceBERT:
    """beir.retrieval.models.SentenceBERT (BDR:412): plain texts, title + sep + text."""

    def __init__(self, model, sep: str = " "):
        self.model, self.sep = model, sep

    def encode_queries(self, queries, batch_size: int = 16, **kwargs):
        return self.model.encode(queries, batch_size=batch_size, **kwargs)

    def encode_corpus(self, corpus, batch_size: int = 8, **kwargs):
        sentences = [(doc["title"] + self.sep + doc["text"]).strip() if "title" in doc else doc["text"].strip()
                     for doc in corpus]
        return self.model.encode(sentences, batch_size=batch_size, **kwargs)


def update_scores_json(path: str, model_name: str, dataset: str, ndcg, _map, recall, precision) -> dict:
    """BDR:448-496: merge this run into beir_embeddings_ndcgs.json, adding the CQADupStack average once complete."""
    if os.path.exists(path):
        with open(path) as f:
            js = json.load(f)
    else:
        js = {"ndcgs": {}, "maps": {}, "recalls": {}, "precisions": {}}
    for key, val in (("ndcgs", ndcg), ("maps", _map), ("recalls", recall), ("precisions", precision)):
        js.setdefault(key, {}).setdefault(model_name, {})[dataset] = val
    have = js["ndcgs"][model_name]
    if "cqadupstack" in dataset and all(f"cqadupstack_{d}" in have for d in CQADUPSTACK_DATASETS):
        avg = {}
        for d in CQADUPSTACK_DATASETS:
            for k, v in have[f"cqadupstack_{d}"].items():
                avg[k] = avg.get(k, 0) + v / len(CQADUPSTACK_DATASETS)
        have["cqadupstack"] = avg
    with open(path, "w") as f:
        json.dump(js, f)
    return js


def main(args) -> dict:
    data_path = f"{args.datapath}/{args.dataset}"
    if not os.path.exists(data_path):
        raise FileNotFoundError(f"{data_path} not found (the reference would download it, BDR:370-377; there is no "
                                "network here — unpack the BEIR dataset under --datapath)")
    split = "dev" if args.dataset == "msmarco" else "test"  # BDR:380-381
    corpus, queries, qrels = GenericDataLoader(data_path).load(split=split)
    corpus = clean_titles(corpus) if "robust04" in data_path else corpus
    empty_keys = [k for k, v in corpus.items() if not v["text"]]
    logger.info(f"Found {len(empty_keys)} empty keys in corpus. Removing...")
    assert len(empty_keys) < len(corpus), "Too many empty keys..."
    for k in empty_keys:
        del corpus[k]
    empty_keys = [k for k, v in queries.items() if not v]
    assert not empty_keys, f"Contains {len(empty_keys)} empty queries"

    dataset = args.dataset.replace("/", "_")
    model_name = args.modelname.rstrip("/").replace("/", "_")
    out_path = os.path.join(args.outdir, f"results_{model_name}_{args.method}_{dataset}.json")
    if os.path.exists(out_path) and not args.overwrite:
        logger.info(f"Found {out_path} - Skipping ...")
        return {}
    retriever = EvaluateRetrieval(build_retriever(args), k_values=[1, 3, 5, 10, 100, 1000])
    results = retriever.retrieve(corpus, queries)
    with open(out_path, "w") as fp:
        json.dump(results, fp)
    ndcg, _map, recall, precision = retriever.evaluate(qrels, results, retriever.k_values)
    update_scores_json(os.path.join(args.outdir, "beir_embeddings_ndcgs.json"), model_name, dataset, ndcg, _map, recall,
                       precision)
    return {"ndcg": ndcg, "map": _map, "recall": recall, "precision": precision}


if __name__ == "__main__":
    logging.basicConfig(format="%(asctime)s - %(message)s", datefmt="%Y-%m-%d %H:%M:%S", level=logging.INFO)
    main(parse_args())
