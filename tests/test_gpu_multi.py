"""Multi-GPU correctness of the sharded search ON GPUs (VERDICT r01 item 1b): two NCCL ranks, each scanning its row range
of one planted corpus; the merged result of (a) the single packed NCCL all-gather + merge kernel and (b) the peer-memory
push/merge (PeerGather: no collective) must equal the oracle's top-k over the WHOLE corpus on every rank.  Skipped on a
one-GPU box; bench.py repeats the same check under the driver's own multi-GPU launch (`merge_verified`)."""
import os
import sys

import pytest
import torch

from tests.conftest import ROOT
from tests.helpers import planted_corpus

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    torch.cuda.set_device(rank)
    dev = torch.device(f"cuda:{rank}")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from oracle import search as osearch
        from sgpt_b200 import CorpusShard, PeerGather, sharded_search
        from sgpt_b200.dist import shard_range
        from tests.test_gpu_parity import _assert_same_topk

        out = {}
        for case, (nq, n, D, k, fn) in enumerate([(130, 40001, 64, 101, "cos_sim"), (9, 700_000, 64, 1001, "dot")]):
            qv, cv = planted_corpus(n, D, nq, seed=77 + case)
            lo, hi = shard_range(n, rank, world)
            shard = CorpusShard.from_embeddings(cv[lo:hi].to(dev), device=dev, id_base=lo)
            exclude = torch.full((nq,), -1, dtype=torch.int64)
            exclude[0], exclude[nq - 1] = 0, 97  # planted near-duplicates of those queries: must be dropped (XS:118)
            full = osearch.SCORE_FUNCTIONS[fn](qv.to(torch.bfloat16).float(), cv.to(torch.bfloat16).float())
            for qi in range(nq):
                if exclude[qi] >= 0:
                    full[qi, exclude[qi]] = float("-inf")
            s, i = sharded_search(qv.to(dev), shard, k, fn, exclude_ids=exclude.to(dev))  # one packed NCCL all-gather
            _assert_same_topk(s, i, full, k)
            gather = PeerGather(nq, k, dev)
            for rep in range(3):  # both buffer parities and their reuse
                s2, i2 = gather.search(shard, qv.to(dev), k, fn, exclude_ids=exclude.to(dev))
                _assert_same_topk(s2, i2, full, k)
                assert torch.equal(s2, s) and torch.equal(i2, i), f"peer gather != NCCL gather (rep {rep})"
            # every rank holds the identical merged list
            ref_i = i.clone()
            dist.broadcast(ref_i, src=0)
            assert torch.equal(ref_i, i)
            gather.close()
            out[case] = True
        q.put((rank, "ok", out))
    except Exception as e:  # noqa: BLE001 - reported to the parent
        import traceback

        q.put((rank, "error", traceback.format_exc()[-3000:] + repr(e)))
    finally:
        dist.destroy_process_group()


def test_two_rank_nccl_and_peer_gather_match_whole_corpus_oracle():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 23000 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    res = [q.get(timeout=600) for _ in procs]
    [p.join(120) for p in procs]
    for rank, status, payload in res:
        assert status == "ok", f"rank {rank}: {payload}"


def test_packed_search_and_merge_single_gpu():
    """The packed entry format and the packed merge on ONE GPU: two half shards searched with search_packed and merged
    == the whole shard searched directly (ids, scores), incl. the (-inf, -1) tail of a shard smaller than k."""
    from sgpt_b200 import CorpusShard, PeerGather, merge_topk_packed, unpack_topk

    dev = torch.device("cuda:0")
    qv, cv = planted_corpus(5000, 128, 7, seed=3)
    whole = CorpusShard.from_embeddings(cv.to(dev), device=dev)
    k = 300
    s, i = whole.search(qv.to(dev), k, "cos_sim")
    a = CorpusShard.from_embeddings(cv[:200].to(dev), device=dev, id_base=0)  # fewer than k documents
    b = CorpusShard.from_embeddings(cv[200:].to(dev), device=dev, id_base=200)
    pa, pb = a.search_packed(qv.to(dev), k, "cos_sim"), b.search_packed(qv.to(dev), k, "cos_sim")
    sa, ia = unpack_topk(pa)
    assert torch.all(ia[:, 200:] == -1) and torch.all(torch.isinf(sa[:, 200:])) and torch.all(ia[:, :200] >= 0)
    sm, im = merge_topk_packed(torch.stack([pa, pb]))
    assert torch.equal(im, i) and torch.equal(sm, s)
    ex = torch.full((7,), -1, dtype=torch.int64, device=dev)
    ex[2] = i[2, 0]
    sm, im = merge_topk_packed(torch.stack([pa, pb]), ex)
    assert int(i[2, 0]) not in im[2].tolist() and torch.equal(im[2, :k - 1], i[2, 1:])
    # world-size-1 peer gather == plain search
    g = PeerGather(7, k, dev)
    for _ in range(3):
        s1, i1 = g.search(whole, qv.to(dev), k, "cos_sim")
        assert torch.equal(s1, s) and torch.equal(i1, i)
    g.close()
