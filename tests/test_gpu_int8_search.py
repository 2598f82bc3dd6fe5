"""int8 corpus shards on the GPU: the quantization kernel, the kind::i8 scan (dense, two-pass, CTA-pair paths), packed
results and their merge, persistence, the DRES surface and the retrieval quality of the format.  The kernels reproduce
the CPU oracle of tests/int8_oracle.py bit for bit, so scores are compared for equality and ids exactly (ties at the cut
as sets)."""
import os

import numpy as np
import pytest
import torch

from tests.helpers import ToyTokenizer, planted_corpus
from tests.int8_oracle import assert_same_topk, quantize_rows, scores

pytestmark = pytest.mark.gpu


def _gpu_quant(x):
    from sgpt_b200.index import quantize_rows_i8

    c, s, inv = quantize_rows_i8(x.cuda())
    return c.cpu().numpy(), s.cpu().numpy(), inv.cpu().numpy()


@pytest.mark.parametrize("D", [64, 768, 4096])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_quantizer_bit_identical_to_oracle(D, dtype):
    g = torch.Generator().manual_seed(D)
    x = torch.randn(300, D, generator=g) * torch.rand(300, 1, generator=g) * 4
    x[3] = 0.0  # all-zero row: s = 0, codes 0, inv = 1e12
    # rows whose values sit exactly on .5 after the division: max = 127 -> s = 1, x = k + 0.5
    x[5] = (torch.arange(D) % 50 - 25).float() + 0.5
    x[5, 0] = 127.0
    x[6] = -x[5]
    x[7, :] = 1e-3
    x[7, 1] = -200.0
    x = x.to(dtype)
    got, want = _gpu_quant(x), quantize_rows(x)
    for a, b, what in zip(got, want, ("codes", "scale", "inv_norm")):
        assert a.dtype == b.dtype and np.array_equal(a, b), what
    assert got[1][3] == 0 and np.all(got[0][3] == 0)
    assert got[1][5] == np.float32(1.0) and got[0][5, 1] == -24  # -23.5 -> -24 (half to even)


def _oracle_full(q, c, fn):
    return scores(quantize_rows(q), quantize_rows(c), fn)


SHAPES = [(128, 20000, 768, 1001), (16, 5003, 2048, 1001), (1, 3000, 768, 1001), (7, 600, 64, 1001),
          # two-pass path; 130 queries = two query blocks; ragged last tile
          (130, 320001, 64, 1001), (5, 310000, 128, 10),
          # CTA-pair scans (M = 256): one pair block + a 44-query block; a full pair
          (300, 320001, 64, 100), (256, 150001, 128, 1001)]


@pytest.mark.parametrize("fn", ["cos_sim", "dot"])
@pytest.mark.parametrize("nq,n,D,k", SHAPES)
def test_int8_search_identical_to_oracle(nq, n, D, k, fn):
    from sgpt_b200 import CorpusShard

    q, c = planted_corpus(n, D, nq, seed=4321)
    shard = CorpusShard.from_embeddings(c.cuda(), device="cuda:0", id_base=1000, dtype="int8")
    s, i = shard.search(q.cuda(), k, fn)
    full = _oracle_full(q, c, fn)
    assert_same_topk(s, i, full, k, id_base=1000)
    if n < k:
        assert torch.all(i[:, n:] == -1) and torch.all(torch.isinf(s[:, n:]))


@pytest.mark.parametrize("k_hi", ["1", "1001"])
def test_int8_two_pass_front_and_back_lists(k_hi, monkeypatch):
    """SGPT_SEARCH_K_HI=1 forces every query through the back lists, = k puts everything at the front (no split)."""
    from sgpt_b200 import CorpusShard

    monkeypatch.setenv("SGPT_SEARCH_K_HI", k_hi)
    nq, n, D, k = 37, 130001, 128, 1001
    q, c = planted_corpus(n, D, nq, seed=77)
    shard = CorpusShard.from_embeddings(c.cuda(), device="cuda:0", id_base=7, dtype="int8")
    for fn in ("cos_sim", "dot"):
        s, i = shard.search(q.cuda(), k, fn)
        assert_same_topk(s, i, _oracle_full(q, c, fn), k, id_base=7)


def test_int8_packed_and_merge_equal_search():
    from sgpt_b200 import CorpusShard, merge_topk_packed

    dev = torch.device("cuda:0")
    q, c = planted_corpus(200000, 256, 40, seed=11)
    whole = CorpusShard.from_embeddings(c.to(dev), device=dev, dtype="int8")
    k = 500
    for fn in ("cos_sim", "dot"):
        s, i = whole.search(q.to(dev), k, fn)
        a = CorpusShard.from_embeddings(c[:90000].to(dev), device=dev, id_base=0, dtype="int8")
        b = CorpusShard.from_embeddings(c[90000:].to(dev), device=dev, id_base=90000, dtype="int8")
        sm, im = merge_topk_packed(torch.stack([a.search_packed(q.to(dev), k, fn), b.search_packed(q.to(dev), k, fn)]))
        assert torch.equal(sm, s) and torch.equal(im, i), fn


def test_int8_shard_save_load_roundtrip(tmp_path):
    from sgpt_b200 import CorpusShard

    q, c = planted_corpus(5000, 128, 9, seed=5)
    shard = CorpusShard.from_embeddings(c.cuda(), id_base=1000, dtype="int8")
    s0, i0 = shard.search(q.cuda(), 50, "dot")
    shard.save(str(tmp_path / "s"))
    again = CorpusShard.load(str(tmp_path / "s"), device="cuda:0")
    assert again.dtype == "int8" and again.n == shard.n and again.id_base == 1000
    assert torch.equal(again.vectors[:again.n], shard.vectors[:shard.n])
    s1, i1 = again.search(q.cuda(), 50, "dot")
    assert torch.equal(s0, s1) and torch.equal(i0, i1)
    s2, i2 = again.search(q.cuda(), 50, "cos_sim")
    assert torch.equal(s2, shard.search(q.cuda(), 50, "cos_sim")[0])


def test_int8_add_rejects_non_finite_rows():
    from sgpt_b200 import CorpusShard

    shard = CorpusShard(64, 10, device="cuda:0", dtype="int8")
    for bad in (float("nan"), float("inf")):
        x = torch.randn(3, 64)
        x[1, 7] = bad
        with pytest.raises(ValueError, match="non-finite"):
            shard.add(x.cuda())
    assert shard.n == 0


def test_int8_dres_matches_oracle_search_loop(golden_dir):
    """DenseRetrievalExactSearch(corpus_dtype="int8") on the tiny encoder == the XS search loop over the oracle's int8
    scores of the same embeddings (self match dropped, up to top_k + 1 entries, bit-identical scores)."""
    from oracle import gpt_neo
    from sgpt_b200 import CustomEmbedder, DenseRetrievalExactSearch
    from tests.test_gpu_parity import _cfg_from_spec, _spec_from

    z = np.load(os.path.join(golden_dir, "neo_tiny.npz"))
    spec = _spec_from(z)
    w = gpt_neo.init_weights(spec, seed=int(z["weight_seed"]))
    emb = CustomEmbedder("toy-gpt-neo", batch_size=16, device="cuda:0", method="weightedmean", specb=True, maxseqlen=40,
                         config=_cfg_from_spec(spec), state_dict=w, tokenizer=ToyTokenizer(vocab=spec.vocab))
    rs = np.random.RandomState(0)
    words = [f"w{i}" for i in range(300)]
    corpus = {f"d{i}": {"title": " ".join(rs.choice(words, 3)), "text": " ".join(rs.choice(words, rs.randint(1, 60)))}
              for i in range(130)}
    queries = {f"q{i}": " ".join(rs.choice(words, rs.randint(1, 12))) for i in range(9)}
    queries["d5"] = corpus["d5"]["text"]
    top_k = 20
    for fn in ("cos_sim", "dot"):
        res = DenseRetrievalExactSearch(emb, batch_size=16, corpus_chunk_size=50, corpus_dtype="int8").search(
            corpus, queries, top_k, fn)
        corpus_ids = sorted(corpus, key=lambda k: len(corpus[k].get("title", "") + corpus[k].get("text", "")),
                            reverse=True)
        q_emb = emb.encode_queries([(qid, queries[qid]) for qid in queries], convert_to_tensor=True).float()
        c_emb = emb.encode_corpus([(cid, corpus[cid]) for cid in corpus_ids], convert_to_tensor=True).float()
        full = _oracle_full(q_emb.cpu(), c_emb.cpu(), fn)
        for qi, qid in enumerate(queries):
            # XS:96-132: per chunk of 50 the top-(k+1), self match dropped, running nlargest(k+1)
            want = {}
            for start in range(0, len(corpus_ids), 50):
                sc = full[qi, start:start + 50]
                for j in torch.argsort(-sc.double(), stable=True)[:top_k + 1].tolist():
                    if corpus_ids[start + j] != qid:
                        want[corpus_ids[start + j]] = sc[j].item()
                keep = sorted(want, key=lambda cid: -want[cid])[:top_k + 1]
                want = {cid: want[cid] for cid in keep}
            assert "d5" not in res["d5"] and len(res[qid]) == len(want)
            cut = min(want.values())
            assert {c for c in want if want[c] > cut} <= set(res[qid]), qid
            for cid, score in res[qid].items():
                assert score == full[qi, corpus_ids.index(cid)].item() and score >= cut, (qid, cid)


def test_int8_retrieval_quality_on_planted_corpus():
    """Top-k overlap of the int8 shard against fp32 cos_sim on the planted 200 k x 768 corpus (64 queries).  The GPU
    equals the oracle, so the figure is deterministic; a CPU fp64 simulation of the format gives 0.973 / 0.985 / 0.988."""
    from sgpt_b200 import CorpusShard

    q, c = planted_corpus(200000, 768, 64, seed=4321)
    shard = CorpusShard.from_embeddings(c.cuda(), device="cuda:0", dtype="int8")
    _, i = shard.search(q.cuda(), 1000, "cos_sim")
    qn, cn = q.cuda() / q.cuda().norm(dim=1, keepdim=True), c.cuda() / c.cuda().norm(dim=1, keepdim=True)
    ref = torch.topk(qn @ cn.T, 1000, dim=1).indices
    for k, bar in ((10, 0.96), (100, 0.98), (1000, 0.98)):
        overlap = sum(len(set(a[:k]) & set(b[:k])) for a, b in zip(i.tolist(), ref.tolist())) / (64 * k)
        assert overlap >= bar, (k, overlap)


def _two_rank_worker(rank, world, port, q):
    import sys

    import torch.distributed as dist

    from tests.conftest import ROOT

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    torch.cuda.set_device(rank)
    dev = torch.device(f"cuda:{rank}")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from sgpt_b200 import CorpusShard, PeerGather, sharded_search
        from sgpt_b200.dist import shard_range

        for case, (nq, n, D, k, fn) in enumerate([(130, 40001, 64, 101, "cos_sim"), (9, 700_000, 64, 1001, "dot")]):
            qv, cv = planted_corpus(n, D, nq, seed=77 + case)
            lo, hi = shard_range(n, rank, world)
            shard = CorpusShard.from_embeddings(cv[lo:hi].to(dev), device=dev, id_base=lo, dtype="int8")
            exclude = torch.full((nq,), -1, dtype=torch.int64)
            exclude[0], exclude[nq - 1] = 0, 97
            full = _oracle_full(qv, cv, fn)
            for qi in range(nq):
                if exclude[qi] >= 0:
                    full[qi, exclude[qi]] = float("-inf")
            s, i = sharded_search(qv.to(dev), shard, k, fn, exclude_ids=exclude.to(dev))
            assert_same_topk(s, i, full, k)
            gather = PeerGather(nq, k, dev)
            for _ in range(2):
                s2, i2 = gather.search(shard, qv.to(dev), k, fn, exclude_ids=exclude.to(dev))
                assert torch.equal(s2, s) and torch.equal(i2, i)
            gather.close()
        q.put((rank, "ok", None))
    except Exception as e:  # noqa: BLE001 - reported to the parent
        import traceback

        q.put((rank, "error", traceback.format_exc()[-3000:] + repr(e)))
    finally:
        dist.destroy_process_group()


def test_int8_two_rank_nccl_and_peer_gather_match_whole_corpus_oracle():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 25000 + os.getpid() % 2000
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    res = [q.get(timeout=600) for _ in procs]
    [p.join(120) for p in procs]
    for rank, status, payload in res:
        assert status == "ok", f"rank {rank}: {payload}"
