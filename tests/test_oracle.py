"""Pin the oracle (oracle/) against the golden fixtures produced by the REFERENCE code (tests/golden/make_golden.py:
HF GPTNeoModel + the reference's Pooling.py + the reference's util.py), and re-run the reference's own property tests
for the scoring stage (sentence-transformers/tests/test_util.py:9-53) with fixed seeds.  CPU only."""
import os

import numpy as np
import pytest
import torch

from oracle import gpt_neo, pooling, search


def _spec_from(npz):
    L, d, H, ff, vocab, max_pos, window = [int(x) for x in npz["spec"]]
    return gpt_neo.NeoSpec(n_layer=L, d_model=d, n_head=H, d_ff=ff, vocab=vocab, max_pos=max_pos, window=window)


@pytest.fixture(scope="module")
def tiny(golden_dir):
    z = np.load(os.path.join(golden_dir, "neo_tiny.npz"))
    spec = _spec_from(z)
    w = gpt_neo.init_weights(spec, seed=int(z["weight_seed"]))
    ids = torch.from_numpy(z["input_ids"]).long()
    mask = torch.from_numpy(z["attention_mask"]).long()
    with torch.no_grad():
        hs = gpt_neo.forward(spec, w, ids, mask)
    return z, spec, ids, mask, hs


def test_forward_matches_hf_hidden_states(tiny):
    """Every hidden state of the restated forward == HF GPTNeoModel's, at the real (unpadded) positions.
    The tiny spec has window 16 < S 48, so the local-attention layers are exercised."""
    z, spec, ids, mask, hs = tiny
    ref = torch.from_numpy(z["hidden_states"])
    assert len(hs) == spec.n_layer + 1 == ref.shape[0]
    m = mask.bool()
    for i in range(len(hs)):
        diff = (hs[i] - ref[i]).abs()[m].max().item()
        assert diff < 2e-5, (i, diff)


def test_pooling_matches_reference_pooling(tiny):
    z, spec, ids, mask, hs = tiny
    last = hs[-1]
    for clamp in (False, True):
        np.testing.assert_allclose(pooling.weighted_mean(last, mask, clamp).numpy(), z["pooled_weightedmean"], atol=2e-5)
        np.testing.assert_allclose(pooling.mean(last, mask, clamp).numpy(), z["pooled_mean"], atol=2e-5)
    np.testing.assert_allclose(pooling.last_token(last, mask, st_variant=True).numpy(), z["pooled_lasttoken"], atol=2e-5)
    # script semantics agree with Pooling.py wherever the row is padded (Pooling.py's argmin trick breaks on full rows)
    padded = (mask.sum(1) < mask.shape[1]).numpy()
    assert padded.any() and (~padded).any()
    np.testing.assert_allclose(pooling.last_token(last, mask).numpy()[padded], z["pooled_lasttoken"][padded], atol=2e-5)
    mid = int(z["mid_layer"])
    np.testing.assert_allclose(pooling.weighted_mean(hs[mid], mask).numpy(), z["pooled_weightedmean_mid"], atol=2e-5)


def test_config1_sgpt125m_pooled_embeddings(golden_dir):
    """BASELINE.json configs[0]: SGPT-125M-weightedmean, 32 sentences, seq_len 64 — pooled-embedding parity of the
    oracle vs the reference path (HF forward + Pooling.py)."""
    z = np.load(os.path.join(golden_dir, "neo_125m_b32_s64.npz"))
    spec = _spec_from(z)
    assert (spec.n_layer, spec.d_model, spec.n_head) == (12, 768, 12)
    w = gpt_neo.init_weights(spec, seed=int(z["weight_seed"]))
    ids = torch.from_numpy(z["input_ids"]).long()
    mask = torch.from_numpy(z["attention_mask"]).long()
    with torch.no_grad():
        hs = gpt_neo.forward(spec, w, ids, mask)
    emb = pooling.weighted_mean(hs[-1], mask)
    ref = torch.from_numpy(z["pooled_weightedmean"])
    cos = torch.nn.functional.cosine_similarity(emb, ref, dim=1)
    assert cos.min().item() > 1 - 1e-6
    assert (emb - ref).abs().max().item() < 1e-4
    np.testing.assert_allclose(pooling.mean(hs[-1], mask).numpy(), z["pooled_mean"], atol=1e-4)
    mid = int(z["mid_layer"])
    np.testing.assert_allclose(pooling.weighted_mean(hs[mid], mask).numpy(), z["pooled_weightedmean_mid"], atol=1e-4)


def test_ragged_equals_padded(tiny):
    """Right-padded rows never influence real rows under causal attention (SURVEY §8a F-note): running each sequence
    alone, unpadded, gives the same hidden states — the legality argument for the ragged CUDA layout."""
    z, spec, ids, mask, hs = tiny
    w = gpt_neo.init_weights(spec, seed=int(z["weight_seed"]))
    for b in range(ids.shape[0]):
        n = int(mask[b].sum())
        with torch.no_grad():
            alone = gpt_neo.forward(spec, w, ids[b:b + 1, :n], None)
        assert (alone[-1][0] - hs[-1][b, :n]).abs().max().item() < 2e-5


def test_scoring_matches_reference_util(golden_dir):
    z = np.load(os.path.join(golden_dir, "scoring.npz"))
    q, c = torch.from_numpy(z["queries"]), torch.from_numpy(z["corpus"])
    np.testing.assert_allclose(search.cos_sim(q, c).numpy(), z["cos"], atol=1e-6)
    np.testing.assert_allclose(search.dot_score(q, c).numpy(), z["dot"], atol=1e-5)
    assert np.all(search.cos_sim(q, c).numpy()[:, 3] == 0.0)  # zero vector: x / max(||x||, 1e-12) = 0
    hits = search.semantic_search(q, c, query_chunk_size=5, corpus_chunk_size=17, top_k=10)
    ids = np.array([[h["corpus_id"] for h in row] for row in hits])
    np.testing.assert_array_equal(ids, z["hit_ids"])
    np.testing.assert_allclose(np.array([[h["score"] for h in row] for row in hits]), z["hit_scores"], atol=1e-6)


# --- the reference's own property tests for this stage, seeded (sentence-transformers/tests/test_util.py) ---------
def test_ref_property_normalize_embeddings():
    """tests/test_util.py:9-18: rows of normalize() have unit length (±1e-4)."""
    g = torch.Generator().manual_seed(0)
    x = torch.randn(50, 16, generator=g)
    n = pooling.normalize(x)
    assert (n.norm(dim=1) - 1).abs().max().item() < 1e-4


def test_ref_property_cos_sim_vs_numpy():
    """tests/test_util.py:21-30: cos_sim vs an independent cosine (sklearn there, numpy fp64 here), |d| < 1e-3."""
    rs = np.random.RandomState(1)
    a, b = rs.randn(50, 100), rs.randn(50, 100)
    ref = (a / np.linalg.norm(a, axis=1, keepdims=True)) @ (b / np.linalg.norm(b, axis=1, keepdims=True)).T
    got = search.cos_sim(torch.tensor(a, dtype=torch.float32), torch.tensor(b, dtype=torch.float32)).numpy()
    assert np.abs(got - ref).max() < 1e-3


def test_ref_property_semantic_search_chunking():
    """tests/test_util.py:33-53: chunked search (5 x 17) returns the un-chunked top-10 ids, scores within 1e-3."""
    rs = np.random.RandomState(2)
    q = torch.tensor(rs.randn(20, 100), dtype=torch.float32)
    c = torch.tensor(rs.randn(1000, 100), dtype=torch.float32)
    hits = search.semantic_search(q, c, query_chunk_size=5, corpus_chunk_size=17, top_k=10)
    full = search.cos_sim(q, c)
    vals, idx = full.topk(10, dim=1)
    for qi in range(20):
        assert [h["corpus_id"] for h in hits[qi]] == idx[qi].tolist()
        assert np.abs(np.array([h["score"] for h in hits[qi]]) - vals[qi].numpy()).max() < 1e-3


def test_search_embeddings_merge_equals_global_topk():
    """XS:80-134 restatement: chunked top-(k+1) + heapq merge == global top-(k+1) minus self matches; unknown score
    function raises ValueError like XS:46-51."""
    g = torch.Generator().manual_seed(3)
    q = torch.randn(7, 32, generator=g)
    c = torch.randn(500, 32, generator=g)
    qids = [f"q{i}" for i in range(7)]
    cids = [f"d{i}" for i in range(500)]
    cids[10] = "q0"  # a corpus doc that IS query 0 -> dropped for q0 only (XS:118)
    k = 20
    res = search.search_embeddings(qids, q, cids, c, k, "cos_sim", corpus_chunk_size=64)
    full = search.cos_sim(q, c)
    for qi, qid in enumerate(qids):
        order = torch.argsort(-full[qi]).tolist()
        expect = [cids[j] for j in order[:k + 1] if cids[j] != qid]
        got = sorted(res[qid], key=res[qid].get, reverse=True)
        assert got[:len(expect)] == expect[:len(got)]
        assert len(res[qid]) <= k + 1
    with pytest.raises(ValueError):
        search.search_embeddings(qids, q, cids, c, k, "euclid")


# --- GPT-J (SGPT-5.8B family) and BLOOM (sgpt-bloom-7b1 family) oracles vs HF GPTJModel / BloomModel fixtures ---------
def _family(golden_dir, name):
    from oracle import bloom, gptj

    z = np.load(os.path.join(golden_dir, name + ".npz"))
    a = [int(x) for x in z["spec"]]
    if name.startswith("gptj"):
        spec = gptj.GPTJSpec(n_layer=a[0], d_model=a[1], n_head=a[2], d_ff=a[3], vocab=a[4], max_pos=a[5], rotary_dim=a[6])
        mod = gptj
    else:
        spec = bloom.BloomSpec(n_layer=a[0], d_model=a[1], n_head=a[2], vocab=a[3])
        mod = bloom
    w = mod.init_weights(spec, seed=int(z["weight_seed"]))
    return z, spec, mod, w


@pytest.mark.parametrize("name", ["gptj_tiny", "bloom_tiny"])
def test_gptj_bloom_oracle_matches_hf(golden_dir, name):
    """Restated GPT-J (rotary, parallel residual) / BLOOM (ALiBi, embedding LayerNorm, fused qkv) forward == HF model."""
    z, spec, mod, w = _family(golden_dir, name)
    ids = torch.from_numpy(z["input_ids"]).long()
    mask = torch.from_numpy(z["attention_mask"]).long()
    with torch.no_grad():
        hs = mod.forward(spec, w, ids, mask)
    ref = torch.from_numpy(z["hidden_states"])
    for i in range(len(hs)):
        assert (hs[i] - ref[i]).abs()[mask.bool()].max().item() < 2e-5, i
    np.testing.assert_allclose(pooling.weighted_mean(hs[-1], mask).numpy(), z["pooled_weightedmean"], atol=2e-5)
    np.testing.assert_allclose(pooling.mean(hs[-1], mask).numpy(), z["pooled_mean"], atol=2e-5)


@pytest.mark.parametrize("name", ["neo_tiny", "gptj_tiny", "bloom_tiny"])
def test_script_pooling_modes_match_executed_reference_block(golden_dir, name):
    """All five script-path pooling modes (BDR:238-301) of the oracle vs fixtures produced by EXECUTING the reference's
    own pooling block on the HF hidden states (tests/golden/make_script_pooling.py)."""
    from oracle import pooling

    fx = np.load(os.path.join(golden_dir, name + ".npz"))
    ref = np.load(os.path.join(golden_dir, f"script_pooling_{name}.npz"))
    hs = [torch.from_numpy(h) for h in fx["hidden_states"]]
    mask = torch.from_numpy(fx["attention_mask"].astype(np.int64))
    got = {
        "mean": pooling.mean(hs[-1], mask),
        "weightedmean": pooling.weighted_mean(hs[-1], mask),
        "lasttoken": pooling.last_token(hs[-1], mask),
        "meanmean": pooling.mean_mean(hs, mask),
        "lasttokenmean": pooling.last_token_mean(hs, mask),
    }
    for mode, val in got.items():
        np.testing.assert_allclose(val.numpy(), ref["pooled_" + mode], rtol=1e-5, atol=1e-6, err_msg=mode)


def _ce_requests(z):
    co, qo = z["ctx_off"], z["cont_off"]
    return [(i, z["ctx_flat"][co[i]:co[i + 1]].tolist(), z["cont_flat"][qo[i]:qo[i + 1]].tolist())
            for i in range(len(co) - 1)]


def test_lm_score_oracle_matches_executed_reference_functions(golden_dir):
    """oracle.lm_score vs the output of the reference's own _loglikelihood_tokens (crossencoder/beir/sgptce.py:150-262,
    executed by tests/golden/make_ce.py on HF GPTNeoForCausalLM with the st_tiny weights): left truncation after the
    instruction, the duplicate request, a 1-token context and a 1-token continuation are all in the fixture."""
    from oracle import lm_score
    from sgpt_b200.st_loader import load_torch_weights

    z = np.load(os.path.join(golden_dir, "ce_tiny.npz"))
    # the fixture stores its bf16-exact 2-D weights as bf16; the oracle computes in fp32
    w = {k: v.float() for k, v in load_torch_weights(os.path.join(golden_dir, "st_tiny")).items()}
    spec = gpt_neo.NeoSpec(n_layer=2, d_model=128, n_head=2, d_ff=256, vocab=300, max_pos=64, window=8)
    reqs = _ce_requests(z)
    assert any(len(c) + len(q) > int(z["max_length"]) + 1 for _, c, q in reqs)  # truncation is exercised
    got = lm_score.loglikelihood(spec, w, reqs, int(z["max_length"]), int(z["instruction_len"]))
    np.testing.assert_allclose(got, z["loglik"], atol=2e-4)
    assert got[0] == got[-1]  # the duplicated request
    assert lm_score.model_input([1, 2, 3, 4, 5, 6], [7, 8], max_length=4, instruction_len=2) == [1, 2, 6, 7]


def _gptj_head(vocab, d, seed):
    g = torch.Generator().manual_seed(seed)  # same construction as tests/golden/make_ce.py:gptj_lm_head
    w = (torch.randn(vocab, d, generator=g) * 0.05).to(torch.bfloat16).float()
    return w, (torch.randn(vocab, generator=g) * 0.5).float()


def test_lm_score_oracle_gptj_untied_head_with_bias(golden_dir):
    """Same for HF GPTJForCausalLM (rotary, parallel residual, untied LM head + bias: the SGPT-CE 6.1B architecture)."""
    from oracle import gptj as ogptj
    from oracle import lm_score

    z = np.load(os.path.join(golden_dir, "ce_gptj_tiny.npz"))
    L, d, H, ff, vocab, max_pos, rd = [int(x) for x in z["spec"]]
    spec = ogptj.GPTJSpec(n_layer=L, d_model=d, n_head=H, d_ff=ff, vocab=vocab, max_pos=max_pos, rotary_dim=rd)
    w = ogptj.init_weights(spec, int(z["weight_seed"]))
    hw, hb = _gptj_head(vocab, d, int(z["head_seed"]))
    got = lm_score.loglikelihood(spec, w, _ce_requests(z), int(z["max_length"]), int(z["instruction_len"]), arch="gptj",
                                 lm_head=hw, lm_bias=hb)
    np.testing.assert_allclose(got, z["loglik"], atol=5e-4)
