"""SURVEY.md §8f row 1 / VERDICT r01 item 9: the retrieval run of the original project's
biencoder/beir/beir_dense_retriever.py (its ``main``, BDR:352-498) against ``sgpt_b200.retrieve.main`` on one toy BEIR
dataset.  tests/golden/reference_main_toyset.json holds the two files the original ``main`` wrote when it ran unmodified
on the stand-in ``beir`` package and ``custommodels`` of sgpt_b200/compat (tests/golden/make_reference_main.py), and
every name the script imports from those two packages.  The test checks that those imports resolve in the stand-in
packages through ``load_reference_script``, and that ``sgpt_b200.retrieve.main`` writes the same result file (same
documents and scores per query) and the same metrics file.  In both runs the two classes that launch CUDA kernels are
replaced by CPU stand-ins that keep their interfaces (a toy embedder with CustomEmbedder's constructor keywords; the
oracle's restatement of the search loop behind DenseRetrievalExactSearch's ``search``); everything else — argument
parsing, GenericDataLoader, empty-text filtering, EvaluateRetrieval.retrieve/evaluate, the result and metric files — is
the code under comparison.  (The same flow with the real classes is covered by tests/test_gpu_heads.py.)"""
import json
import os
import sys
import zlib

import numpy as np
import torch

from tests.conftest import GOLDEN

GOLDEN_FILE = os.path.join(GOLDEN, "reference_main_toyset.json")
# command line of both runs; --datapath (and --outdir for sgpt_b200.retrieve) are added per run
ARGV = ["--dataset", "toyset", "--modelname", "toy/model", "--method", "weightedmean", "--device", "cpu",
        "--batchsize", "16", "--specb"]


class _ToyEmbedder:
    """CustomEmbedder's protocol (BDR:107-120, 316-348) with a deterministic bag-of-words embedding on the CPU."""

    def __init__(self, model_name, batch_size=250, device="cpu", save_emb=False, reinit=False, layeridx=-1, method="mean",
                 dataset="scifact", specb=False, maxseqlen=None, **kwargs):
        self.kw = dict(model_name=model_name, batch_size=batch_size, device=device, method=method, specb=specb,
                       layeridx=layeridx, maxseqlen=maxseqlen, save_emb=save_emb)
        self.device = torch.device("cpu")

    @staticmethod
    def _vec(text, dim=32):
        v = torch.zeros(dim)
        for w in text.lower().split():
            g = torch.Generator().manual_seed(zlib.crc32(w.encode()))
            v += torch.randn(dim, generator=g)
        return v

    def encode_queries(self, queries, batch_size=None, **kwargs):
        return torch.stack([self._vec(t) for _, t in queries])

    def encode_corpus(self, corpus, batch_size=None, **kwargs):
        return torch.stack([self._vec((d["title"] + " " + d["text"]).strip() if "title" in d else d["text"].strip())
                            for _, d in corpus])


class _CpuDRES:
    """DenseRetrievalExactSearch's interface (XS:22-42) on the oracle's restatement of XS:44-134."""

    def __init__(self, model, batch_size=128, corpus_chunk_size=50000, **kwargs):
        self.model, self.batch_size, self.corpus_chunk_size = model, batch_size, corpus_chunk_size
        self.results = {}

    def search(self, corpus, queries, top_k, score_function, return_sorted=False, **kwargs):
        from oracle import search as osearch

        if score_function not in ("cos_sim", "dot"):
            raise ValueError("score function: {} must be either (cos_sim) for cosine similarity or (dot) for dot product"
                             .format(score_function))
        qids = list(queries)
        cids = sorted(corpus, key=lambda k: len(corpus[k].get("title", "") + corpus[k].get("text", "")), reverse=True)
        q = self.model.encode_queries([(i, queries[i]) for i in qids], batch_size=self.batch_size)
        c = self.model.encode_corpus([(i, corpus[i]) for i in cids], batch_size=self.batch_size, batch_num=0)
        self.results = osearch.search_embeddings(qids, q, cids, c, top_k, score_function,
                                                 corpus_chunk_size=self.corpus_chunk_size)
        return self.results


def write_toyset(datasets_dir):
    """Toy BEIR directory ``<datasets_dir>/toyset``: the relevant document of every query repeats the query's words, and
    one document has an empty text.  Returns the queries."""
    rs = np.random.RandomState(0)
    words = [f"w{i}" for i in range(200)]
    root = os.path.join(datasets_dir, "toyset")
    os.makedirs(os.path.join(root, "qrels"))
    corpus = {f"d{i}": {"title": " ".join(rs.choice(words, 2)), "text": " ".join(rs.choice(words, rs.randint(3, 30)))}
              for i in range(60)}
    corpus["d_empty"] = {"title": "t", "text": ""}  # removed by the script (BDR:382-388)
    queries = {f"q{i}": corpus[f"d{i}"]["text"] for i in range(8)}
    with open(os.path.join(root, "corpus.jsonl"), "w") as f:
        for k, v in corpus.items():
            f.write(json.dumps({"_id": k, **v}) + "\n")
    with open(os.path.join(root, "queries.jsonl"), "w") as f:
        for k, v in queries.items():
            f.write(json.dumps({"_id": k, "text": v}) + "\n")
    with open(os.path.join(root, "qrels", "test.tsv"), "w") as f:
        f.write("query-id\tcorpus-id\tscore\n")
        for i in range(8):
            f.write(f"q{i}\td{i}\t1\n")
    return queries


def _assert_close(got, want, path="scores"):
    """Same nested keys; numbers within 1e-6 (metrics are rounded to 5 decimals, scores are fp32 cosines)."""
    if isinstance(want, dict):
        assert isinstance(got, dict) and set(got) == set(want), f"{path}: keys {sorted(got)} != {sorted(want)}"
        for k in want:
            _assert_close(got[k], want[k], f"{path}/{k}")
    else:
        assert abs(got - want) <= 1e-6, f"{path}: {got} != {want}"


def test_retrieve_main_matches_reference_main_on_the_stand_in_packages(tmp_path, monkeypatch):
    import sgpt_b200
    from sgpt_b200 import compat, retrieve
    from sgpt_b200.compat.run_reference import load_reference_script

    with open(GOLDEN_FILE) as f:
        want = json.load(f)
    queries = write_toyset(str(tmp_path / "datasets"))

    # the original script's imports from `beir` / `custommodels`, loaded the way run_reference loads the script
    script = tmp_path / "imports_of_the_reference_script.py"
    script.write_text("".join(f"from {mod} import {name}\n" for mod, names in want["imports"] for name in names)
                      + "\n\nclass CustomEmbedder:\n    pass\n")
    monkeypatch.setattr(sys, "path", list(sys.path))
    mod = load_reference_script(str(script), embedder_cls=_ToyEmbedder, module_name="ref_bdr_imports_under_test")
    assert mod.CustomEmbedder is _ToyEmbedder
    import beir
    import custommodels

    assert os.path.dirname(os.path.dirname(beir.__file__)) == compat.COMPAT_DIR  # the stand-in, not an installed beir
    assert custommodels.DenseRetrievalExactSearch.__module__ == "sgpt_b200.exact_search"

    # the project's retrieval run, with the same two CPU stand-ins the original run had
    monkeypatch.setattr(sgpt_b200, "CustomEmbedder", _ToyEmbedder)
    monkeypatch.setattr(sgpt_b200, "DenseRetrievalExactSearch", _CpuDRES)
    out = tmp_path / "out"
    out.mkdir()
    args = retrieve.parse_args(ARGV + ["--datapath", str(tmp_path / "datasets"), "--outdir", str(out)])
    retrieve.main(args)

    assert sorted(os.listdir(out)) == sorted([want["result_file"], "beir_embeddings_ndcgs.json"])
    with open(out / want["result_file"]) as f:
        results = json.load(f)
    _assert_close(results, want["results"], "results")
    with open(out / "beir_embeddings_ndcgs.json") as f:
        nd = json.load(f)
    _assert_close(nd, want["scores"])
    assert set(results) == set(queries)
    for i in range(8):
        assert max(results[f"q{i}"], key=results[f"q{i}"].get) == f"d{i}"  # the planted document ranks first
        assert "d_empty" not in results[f"q{i}"]
    assert nd["ndcgs"]["toy_model"]["toyset"]["NDCG@1"] == 1.0
    assert nd["recalls"]["toy_model"]["toyset"]["Recall@10"] == 1.0
    assert set(nd) >= {"ndcgs", "maps", "recalls", "precisions"}
    # a second run finds the result file and skips (BDR:433-436)
    assert retrieve.main(args) == {}
