#!/usr/bin/env python
"""bench.py — the reference's headline hot path on B200: SGPT-125M bi-encoder, batch 256 x seq_len 128 encode
(GPT-Neo forward + weighted-mean pool) and exact top-1001 cosine retrieval of 128 queries over a 1M-doc corpus shard.

One "step" = encode one batch of 256 synthetic documents  +  search 128 synthetic queries against the resident
1M x 768 shard (N>1: every rank encodes its own batch and scans its own 1M-doc shard — weak scaling — then the per-shard
top-1001 lists are exchanged ONCE (kernel-to-kernel over NVLink peer mappings; NCCL all-gather of packed entries as the
other transport) and merged on every rank; the merged result is verified against a single-rank search of the whole of
a small planted corpus: `merge_verified`).  Extra keys (N=1): BASELINE configs 3-5 at full size, the fp32 top-k overlap,
the 10M-doc strong-scaling legs.  Prints ONE JSON line (rank 0).

  python bench.py --gpus 1 --steps 10 --warmup 3
  python bench.py --gpus 1 --steps 10 --warmup 3 --dump-outputs DIR   # + the last timed step's outputs as DIR/*.npy
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
  python bench.py --impl reference ...      # the reference's CPU path (HF GPTNeoModel fp32 + pooling + cos_sim/topk)
"""
import argparse
import ctypes
import gc
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "embeddings/sec (SGPT-125M, batch 256, seq 128) + queries/sec@top-1000 (1M-doc corpus)"
B, S, NQ, NDOCS, TOPK = 256, 128, 128, 1_000_000, 1000
CFG = dict(n_layer=12, d_model=768, n_head=12, d_ff=3072, vocab=50257, max_pos=2048)


def synthetic_weights(seed=0):
    """Random-init SGPT-125M (GPT-Neo-125M architecture) weights, HF state_dict keys, bf16-representable values."""
    g = torch.Generator().manual_seed(seed)
    d, ff, L = CFG["d_model"], CFG["d_ff"], CFG["n_layer"]

    def rnd(*shape, sd=0.02, mean=0.0):
        return (torch.randn(*shape, generator=g) * sd + mean).to(torch.bfloat16).float()

    w = {"wte.weight": rnd(CFG["vocab"], d), "wpe.weight": rnd(CFG["max_pos"], d, sd=0.01)}
    for i in range(L):
        p = f"h.{i}."
        w[p + "ln_1.weight"], w[p + "ln_1.bias"] = rnd(d, sd=0.1, mean=1.0), rnd(d, sd=0.05)
        for n in ("q_proj", "k_proj", "v_proj"):
            w[p + f"attn.attention.{n}.weight"] = rnd(d, d)
        w[p + "attn.attention.out_proj.weight"], w[p + "attn.attention.out_proj.bias"] = rnd(d, d), rnd(d)
        w[p + "ln_2.weight"], w[p + "ln_2.bias"] = rnd(d, sd=0.1, mean=1.0), rnd(d, sd=0.05)
        w[p + "mlp.c_fc.weight"], w[p + "mlp.c_fc.bias"] = rnd(ff, d), rnd(ff)
        w[p + "mlp.c_proj.weight"], w[p + "mlp.c_proj.bias"] = rnd(d, ff), rnd(d)
    w["ln_f.weight"], w["ln_f.bias"] = rnd(d, sd=0.1, mean=1.0), rnd(d, sd=0.05)
    return w


def token_batches(n_batches, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, CFG["vocab"], (B, S), generator=g, dtype=torch.int64) for _ in range(n_batches)]


def encoder_flops_per_seq(S_):
    """SURVEY.md §8d: S*2*L*(4d^2 + 2*d*ff) linear FLOPs + L*2*S*(S+1)*d causal attention FLOPs."""
    L, d, ff = CFG["n_layer"], CFG["d_model"], CFG["d_ff"]
    return S_ * 2 * L * (4 * d * d + 2 * d * ff), L * 2 * S_ * (S_ + 1) * d


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        z = json.load(open(p))
        return dict(hbm=z["hbm_gbs"], tf_burst=z["bf16_tflops"], tf_sustained=z["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, reasons = [], set()
        for r in rows:
            try:
                sm.append(float(r[0]))
                out["sm_max_mhz"] = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


# ----------------------------------------------------------------------------------------------------------------------
def reference_cpu_model(weights):
    """The reference's encoder on CPU: HF GPTNeoModel fp32 (what AutoModel.from_pretrained resolves to at
    beir_dense_retriever.py:123); falls back to the oracle's restatement if transformers is unavailable."""
    try:
        from transformers import GPTNeoConfig, GPTNeoModel

        cfg = GPTNeoConfig(vocab_size=CFG["vocab"], max_position_embeddings=CFG["max_pos"], hidden_size=CFG["d_model"],
                           num_layers=CFG["n_layer"], num_heads=CFG["n_head"], intermediate_size=CFG["d_ff"],
                           window_size=256, attention_types=[[["global", "local"], CFG["n_layer"] // 2]],
                           embed_dropout=0.0, attention_dropout=0.0, resid_dropout=0.0)
        m = GPTNeoModel(cfg)
        m.load_state_dict(weights, strict=False)
        m = m.float().eval()

        def fwd(ids, mask):
            with torch.no_grad():
                return m(input_ids=ids, attention_mask=mask, output_hidden_states=True).hidden_states[-1]
        return fwd, "HF GPTNeoModel fp32 + oracle.pooling/oracle.search (ports of Pooling.py / exact_search.py)"
    except Exception:
        from oracle import gpt_neo

        spec = gpt_neo.NeoSpec()

        def fwd(ids, mask):
            with torch.no_grad():
                return gpt_neo.forward(spec, weights, ids, mask)[-1]
        return fwd, "oracle.gpt_neo restatement + oracle.pooling/oracle.search"


_REF_MODEL = {}


def usable_cores():
    """Host threads this process may really use: CPU affinity mask capped by the cgroup CPU quota (os.cpu_count() alone
    over-counts inside a container and oversubscribed MKL threads make the CPU baseline unrealistically slow)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                quota = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    n = min(n, max(1, quota // period))
            break
        except Exception:
            continue
    return max(1, n)


def cpu_model_name():
    """CPU model string of the box the CPU baseline ran on (SURVEY.md §8d asks for it next to the core count)."""
    try:
        for line in open("/proc/cpuinfo"):
            if line.lower().startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_reference_times(weights, enc_batch=32, n_enc=2, search_docs=100_000, warm=True):
    """Bounded sample of the reference CPU path: encode `n_enc` batches of `enc_batch` x 128 tokens, and cos_sim +
    topk(1001) of 128 queries over `search_docs` docs in 50k chunks with the heapq merge (XS:80-132)."""
    from oracle import pooling, search

    torch.set_num_threads(usable_cores())
    if "m" not in _REF_MODEL:
        _REF_MODEL["m"] = reference_cpu_model(weights)  # built once per process
    fwd, how = _REF_MODEL["m"]
    ids = token_batches(1, seed=77)[0]
    mask = torch.ones_like(ids)
    if warm:
        pooling.weighted_mean(fwd(ids[:2], mask[:2]), mask[:2])
    t0 = time.perf_counter()
    for i in range(n_enc):
        sl = slice((i * enc_batch) % B, (i * enc_batch) % B + enc_batch)
        pooling.weighted_mean(fwd(ids[sl], mask[sl]), mask[sl])
    t_enc = time.perf_counter() - t0
    g = torch.Generator().manual_seed(4321)
    q, c = torch.randn(NQ, CFG["d_model"], generator=g), torch.randn(search_docs, CFG["d_model"], generator=g)
    qids, cids = [f"q{i}" for i in range(NQ)], [f"d{i}" for i in range(search_docs)]
    t0 = time.perf_counter()
    search.search_embeddings(qids, q, cids, c, TOPK, "cos_sim", corpus_chunk_size=50000)
    t_search = time.perf_counter() - t0
    emb_s = n_enc * enc_batch / t_enc
    qps_1m = NQ / (t_search * (NDOCS / search_docs))
    return dict(emb_s=emb_s, qps_1m=qps_1m, how=how, t_enc=t_enc, t_search=t_search,
                sample=f"encode {n_enc}x{enc_batch} seqs of {S} tokens; search {NQ} queries over {search_docs} docs in "
                       f"50k chunks incl. python heapq merge, scaled x{NDOCS / search_docs:g} to 1M docs")


def calibrate_reference(weights, enc_seconds, search_seconds):
    """Pick sample sizes so that one reference step costs about enc_seconds + search_seconds on this host."""
    r = cpu_reference_times(weights, enc_batch=8, n_enc=1, search_docs=10_000, warm=True)
    enc_batch = int(min(64, max(4, round(r["emb_s"] * enc_seconds))))
    docs = int(min(200_000, max(10_000, round(10_000 * search_seconds / max(r["t_search"], 1e-3) / 10_000) * 10_000)))
    return enc_batch, docs


def run_reference(args, rank):
    """`--impl reference`: the reference's CPU path (HF GPTNeoModel fp32 on all host cores + Pooling / exact-search ports),
    each step a bounded sample of the workload (~3 s), throughput in the same unit as the B200 arm."""
    if rank != 0:
        return
    w = synthetic_weights(0)
    enc_batch, docs = calibrate_reference(w, enc_seconds=2.0, search_seconds=1.0)
    vals = []
    for _ in range(args.warmup):
        cpu_reference_times(w, enc_batch=enc_batch, n_enc=1, search_docs=docs, warm=False)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        vals.append(cpu_reference_times(w, enc_batch=enc_batch, n_enc=1, search_docs=docs, warm=False))
    wall = time.perf_counter() - t0
    emb_s = float(sum(enc_batch for _ in vals) / sum(v["t_enc"] for v in vals))
    qps = float(NQ * len(vals) / (sum(v["t_search"] for v in vals) * (NDOCS / docs)))
    cores = usable_cores()
    line = {"impl": "reference", "metric": METRIC, "value": emb_s, "unit": "embeddings/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000 * wall / max(1, args.steps),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": workload_config(args.gpus), "search": {"value": qps, "unit": "queries/s"},
            "cpu_baseline": {"value": emb_s, "unit": "embeddings/s", "cores": cores, "cpu_model": cpu_model_name(), "kind": "port",
                             "sample": vals[-1]["sample"] + " per step", "how": vals[-1]["how"], "search_qps_1m": qps},
            "e2e": {"value": emb_s, "unit": "embeddings/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def measured_traffic():
    """DRAM bytes per launch by kernel class from the newest committed ncu capture (profiles/*dram_traffic.json,
    written by tools/ncu_traffic.py); {} when there is none."""
    import glob

    files = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "*dram_traffic.json")))
    if not files:
        return {}, None
    try:
        with open(files[-1]) as f:
            return json.load(f), os.path.relpath(files[-1], os.path.dirname(os.path.abspath(__file__)))
    except (OSError, ValueError):
        return {}, None


def workload_config(n):
    return {"workload": "SGPT-125M (GPT-Neo-125M arch, random-init bf16) bi-encoder: encode batch 256 x seq_len 128 "
                        "(full-length rows) + weighted-mean pool; cos_sim top-1001 of 128 queries over a 1M x 768 bf16 "
                        "corpus shard per GPU", "batch": B, "seq_len": S, "queries": NQ, "docs_per_gpu": NDOCS,
            "top_k": TOPK, "parallelism": f"dp{n} (corpus row-sharded, per-shard top-k exchanged once, merged on every rank)",
            "l2": "inputs larger than L2 (activations 0.55 GB, shard 1.5 GB)"}


CATS = ["embed", "layernorm", "linear_gemm", "attention", "pool", "similarity_gemm", "topk", "misc"]


def fill_shard(shard, n, D, g, dev, queries=None, slab=100_000):
    """Synthetic corpus generated on the device in slabs; with `queries`, 1 % of the rows are planted near-duplicates
    (query + 0.5 noise) so that the top of every ranking is meaningful (SURVEY.md §8d)."""
    for s0 in range(0, n, slab):
        m = min(slab, n - s0)
        c = torch.randn(m, D, generator=g, device=dev)
        if queries is not None:
            idx = torch.arange(0, m, 100, device=dev)
            c[idx] = queries[((s0 + idx) // 100) % queries.shape[0]] + 0.5 * c[idx]
        shard.add(c)
        del c


def time_search(fn, steps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def dump_outputs(out_dir, arrays):
    """`--dump-outputs DIR`: one DIR/<name>.npy per array (float32 / float64), so that two builds can be compared output
    for output on the same seeded inputs."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def other_config_legs(dev, pk, lib, steps):
    """BASELINE.json configs[2..4] at full size on ONE GPU (VERDICT r01 item 7): the encoder of each model at its batch x
    seq_len (random-init bf16 weights drawn on the GPU, inputs resident) and the exact top-1001 search over the shard
    shape the config puts on one GPU.  Extra keys of the JSON line; the headline stays configs[1]."""
    from sgpt_b200 import CorpusShard, Encoder, preset
    from tools.bench_models import SHAPES, rand_weights

    out = {}
    ms_cat, n_cat = (ctypes.c_double * 8)(), (ctypes.c_int64 * 8)()
    for key, name, shard_shape in (("config3_sgpt_1.3b", "sgpt-1.3b", (1_000_000, 2048, "1M x 2048 on one GPU")),
                                   ("config4_sgpt_5.8b_gptj", "sgpt-5.8b", (125_000, 4096, "1M x 4096 over 8 GPUs: 125k per GPU")),
                                   ("config5_sgpt_bloom_7b1", "sgpt-bloom-7b1", (1_250_000, 4096, "10M x 4096 over 8 GPUs: 1.25M per GPU"))):
        leg = {}
        try:
            cfg = preset(name)
            Bm, Sm = SHAPES[name]
            sd = rand_weights(cfg, dev)
            enc = Encoder(cfg, sd, device=dev, max_tokens=Bm * Sm, max_batch=Bm)
            del sd
            g = torch.Generator().manual_seed(1)
            ids = torch.randint(0, cfg.vocab, (Bm, Sm), generator=g).numpy()
            mask = np.ones((Bm, Sm), dtype=np.int8)
            for _ in range(2):
                o = enc.encode_tokens(ids, mask)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                o = enc.encode_tokens(ids, mask)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            lib.sgpt_profile_read(None, None, None)
            lib.sgpt_profile_enable(1)
            for _ in range(steps):
                enc.encode_tokens(ids, mask)
            torch.cuda.synchronize()
            lib.sgpt_profile_enable(0)
            lib.sgpt_profile_read(ms_cat, n_cat, None)
            L, d, ff = cfg.n_layer, cfg.d_model, cfg.d_ff
            lin = Bm * Sm * 2 * L * (4 * d * d + 2 * d * ff)
            att = Bm * L * 2 * Sm * (Sm + 1) * d
            gemm_tf = lin / (ms_cat[2] / steps / 1e3) / 1e12 if ms_cat[2] > 0 else None
            att_tf = att / (ms_cat[3] / steps / 1e3) / 1e12 if ms_cat[3] > 0 else None
            leg["encode"] = {
                "model": name, "batch": Bm, "seq_len": Sm, "ms_per_batch": ms, "embeddings_per_s": Bm / (ms / 1e3),
                "model_tflops": (lin + att) / (ms / 1e3) / 1e12, "finite": bool(torch.isfinite(o).all()),
                "e2e": "Encoder.encode_tokens(host ids): pinned H2D of ids/positions inside the timed region, embeddings stay on the device",
                "kernel_ms_per_batch": {c: ms_cat[i] / steps for i, c in enumerate(CATS) if ms_cat[i] > 0},
                "roofline": {"kernel": "gemm_bf16_tn_kernel (linear layers)", "bound": "tensor", "achieved": gemm_tf,
                             "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": gemm_tf / pk["tf_sustained"] if gemm_tf else None,
                             "traffic": None},
                "roofline_attention": {"kernel": "attention kernel", "bound": "tensor", "achieved": att_tf,
                                       "peak": pk["tf_sustained"], "unit": "TFLOP/s (causal FLOPs 2*S*(S+1)*d per layer per sequence)",
                                       "frac": att_tf / pk["tf_sustained"] if att_tf else None, "traffic": None}}
            enc.close()
            del enc, o
            torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001 - an extra leg must never cost the headline
            leg["encode"] = {"error": repr(e)[:300]}
        try:
            n, D, what = shard_shape
            g = torch.Generator(device=dev).manual_seed(11)
            q = torch.randn(NQ, D, generator=g, device=dev)
            sh = CorpusShard(D, n, device=dev)
            fill_shard(sh, n, D, g, dev, queries=q, slab=125_000)
            ms = time_search(lambda: sh.search(q, TOPK + 1, "cos_sim"), max(steps, 10))
            byts = n * D * 2 + n * 4 + NQ * D * 2
            leg["search"] = {"shard": what, "docs": n, "dim": D, "queries": NQ, "top_k": TOPK, "ms_per_search": ms,
                             "queries_per_s": NQ / (ms / 1e3),
                             "roofline": {"kernel": "whole search (similarity scan x2 + radix selects)", "bound": "hbm",
                                          "achieved": byts / (ms / 1e3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                                          "frac": byts / (ms / 1e3) / 1e9 / pk["hbm"], "traffic": None,
                                          "fits_l2": n * D * 2 < 126e6}}
            del sh
            torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001
            leg["search"] = {"error": repr(e)[:300]}
        out[key] = leg
    return out


def cublas_same_shapes(dev):
    """CALIBRATION ONLY (not a product path): what the vendor library reaches on the four linear shapes of one SGPT-125M
    block at batch 256 x 128 (torch.nn.functional.linear, bf16, bias only — no gelu, no residual), each shape looped back
    to back for ~0.3 s so that it runs under the same sustained power state as the bench step.  MEASURED_PEAKS.json's
    cuBLAS figure is an 8192^3 GEMM; K = 768 shapes cannot reach it in any implementation, so this is the like-for-like
    denominator for `roofline.achieved`."""
    M, d, ff = B * S, CFG["d_model"], CFG["d_ff"]
    out, tot_flops, tot_s = {}, 0.0, 0.0
    for name, N, K in (("qkv", 3 * d, d), ("out_proj", d, d), ("c_fc", ff, d), ("c_proj", d, ff)):
        x = torch.randn(M, K, device=dev, dtype=torch.bfloat16)
        w = torch.randn(N, K, device=dev, dtype=torch.bfloat16) * 0.05
        b = torch.randn(N, device=dev, dtype=torch.bfloat16)
        for _ in range(3):
            torch.nn.functional.linear(x, w, b)
        torch.cuda.synchronize()
        n = max(20, int(0.3 / (2.0 * M * N * K / 1.2e15)))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            torch.nn.functional.linear(x, w, b)
        e1.record()
        torch.cuda.synchronize()
        sec = e0.elapsed_time(e1) / 1e3 / n
        out[name] = {"us": 1e6 * sec, "tflops": 2.0 * M * N * K / sec / 1e12}
        tot_flops += 2.0 * M * N * K
        tot_s += sec
        del x, w, b
    out["block_tflops"] = tot_flops / tot_s / 1e12
    out["note"] = "torch F.linear (cuBLASLt) bf16 + bias, linear only; calibration of the denominator, never on the product path"
    return out


def fp32_overlap_leg(dev):
    """Top-k overlap of the bf16-storage search with the reference's pure-fp32 scoring (SURVEY.md §7 hard part 4, §8c):
    the reference scores fp32 embeddings with cos_sim (sentence_transformers/util.py:24-43) and torch.topk (XS:102-108);
    torch on the GPU evaluates exactly that here, as the checker, on a planted 200k x 768 corpus."""
    from sgpt_b200 import CorpusShard

    n, D, nq = 200_000, 768, 128
    g = torch.Generator(device=dev).manual_seed(2024)
    q = torch.randn(nq, D, generator=g, device=dev)
    c = torch.randn(n, D, generator=g, device=dev)
    idx = torch.arange(0, n, 100, device=dev)
    c[idx] = q[(idx // 100) % nq] + 0.5 * c[idx]
    sh = CorpusShard.from_embeddings(c, device=dev)
    s, i = sh.search(q, TOPK + 1, "cos_sim")
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    ref = torch.nn.functional.normalize(q, dim=1) @ torch.nn.functional.normalize(c, dim=1).T
    torch.backends.cuda.matmul.allow_tf32 = prev
    rs, ri = torch.topk(ref, TOPK + 1, dim=1)
    out = {"docs": n, "dim": D, "queries": nq, "reference": "fp32 cos_sim + torch.topk(1001) of the un-rounded embeddings"}
    for kk in (10, 100, 1001):
        inter = sum(len(set(a[:kk]) & set(b[:kk])) for a, b in zip(i.tolist(), ri.tolist()))
        out[f"overlap_at_{kk}"] = inter / (nq * kk)
    # disagreements can only be documents whose fp32 scores sit within the bf16 storage error of the cut
    cut = rs[:, -1:]
    miss = [(ref[qi, list(set(ri[qi].tolist()) - set(i[qi].tolist()))] - cut[qi]).abs().max().item()
            if set(ri[qi].tolist()) - set(i[qi].tolist()) else 0.0 for qi in range(nq)]
    out["max_fp32_score_gap_of_a_missed_doc_to_the_cut"] = max(miss)
    out["score_max_abs_err_vs_fp32"] = (ref.gather(1, i) - s).abs().max().item()
    return out


# ----------------------------------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist

    from sgpt_b200 import CorpusShard, Encoder, PeerGather, _lib, preset, sharded_search
    from sgpt_b200.dist import all_gather_packed, shard_range
    from sgpt_b200.encoder import pack_ragged
    from sgpt_b200.index import merge_topk_packed

    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    lib = _lib.lib()
    weights = synthetic_weights(0)
    enc = Encoder(preset("sgpt-125m"), weights, device=dev, max_tokens=B * S, max_batch=B)
    batches = token_batches(4, seed=1234 + 1 + rank)
    mask = np.ones((B, S), dtype=np.int8)
    # HBM-resident ragged inputs for the device-timed loop
    resident = []
    for ids in batches:
        p, pos, cu, mx = pack_ragged(ids.numpy(), mask)
        resident.append((torch.from_numpy(p).to(dev), torch.from_numpy(pos).to(dev), torch.from_numpy(cu).to(dev)))
    # corpus shard: generated on the device in slabs (1% planted near-duplicates of the queries)
    D = CFG["d_model"]
    gq = torch.Generator(device=dev).manual_seed(4321)  # the SAME queries on every rank (a sharded search is collective)
    queries = torch.randn(NQ, D, generator=gq, device=dev)
    g = torch.Generator(device=dev).manual_seed(4321 + 17 * (rank + 1))
    shard = CorpusShard(D, NDOCS, device=dev, id_base=rank * NDOCS)
    fill_shard(shard, NDOCS, D, g, dev, queries=queries)
    q_host = queries.cpu().pin_memory()
    kk = TOPK + 1

    # ---- exchange of the per-shard top-k (N > 1) -------------------------------------------------------------------
    gather, transport = None, "none (single GPU)"
    if world > 1:
        transport = "nccl: one all-gather of packed 8-byte (score, id) entries + merge kernel"
        if os.environ.get("SGPT_BENCH_TRANSPORT", "p2p") == "p2p":
            ok = torch.zeros(1, device=dev)
            try:
                gather = PeerGather(NQ, kk, dev)
                ok += 1
            except Exception as e:  # noqa: BLE001 - e.g. CUDA IPC not permitted: every rank falls back together
                print(f"[bench] rank {rank}: peer gather unavailable ({e!r}); using the NCCL all-gather", file=sys.stderr)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if ok.item() < 1:
                gather = None
            else:
                transport = ("p2p: the final selection kernel stores its list into every rank's gather buffer over NVLink "
                             "peer mappings and signals per query; the merge kernel waits on the signals (no collective)")

    def search_step(q_dev, sh=None):
        sh = sh or shard
        if world == 1:
            return sh.search(q_dev, kk, "cos_sim")
        return sharded_search(q_dev, sh, kk, "cos_sim", gather=gather)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxr(x):  # max over ranks (device-timed numbers are reported as the slowest rank's)
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # ---- N > 1: verify the merged result (VERDICT r01 item 1b) -------------------------------------------------------
    # A small planted corpus is split over the ranks exactly like the big one; every rank also holds the WHOLE corpus
    # and searches it alone.  exchange + merge across ranks must reproduce the single-rank result: same scores, same ids
    # except inside groups of tied scores at equal rank.
    merge_verified = None
    if world > 1:
        nv = 64_000 * world
        gv = torch.Generator(device=dev).manual_seed(99)
        cv = torch.randn(nv, D, generator=gv, device=dev)
        idx = torch.arange(0, nv, 100, device=dev)
        cv[idx] = queries[(idx // 100) % NQ] + 0.5 * cv[idx]
        whole = CorpusShard.from_embeddings(cv, device=dev)
        lo, hi = shard_range(nv, rank, world)
        part = CorpusShard.from_embeddings(cv[lo:hi], device=dev, id_base=lo)
        ws_, wi_ = whole.search(queries, kk, "cos_sim")
        good = True
        for rep in range(3):  # both buffer parities of the peer exchange
            ms_, mi_ = search_step(queries, part)
            same_scores = bool((ms_ - ws_).abs().max().item() <= 1e-6)
            agree = (mi_ == wi_).float().mean().item()
            good = good and same_scores and agree > 0.999
        # the NCCL transport as well (it stays the fallback)
        ms2, mi2 = merge_topk_packed(all_gather_packed(part.search_packed(queries, kk, "cos_sim")))
        good = good and bool((ms2 - ws_).abs().max().item() <= 1e-6) and (mi2 == wi_).float().mean().item() > 0.999
        t = torch.tensor([1.0 if good else 0.0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        merge_verified = bool(t.item() > 0)
        del cv, whole, part
        torch.cuda.empty_cache()

    # ---- warm-up -----------------------------------------------------------------------------------------------
    # nvidia-smi needs ~0.5 s to produce its first sample: start it before the warm-up; samples cover warm-up + both
    # timed loops (all of them run the same kernels back to back)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    for w_ in range(max(args.warmup, 1)):
        r = resident[w_ % len(resident)]
        enc.encode_packed(r[0], r[1], r[2], B, B * S, S)
        search_step(queries)
        enc.encode_tokens(batches[w_ % 4].numpy(), mask).cpu()
    barrier()

    # ---- device-timed loop (inputs resident in HBM) -------------------------------------------------------------
    # The timed region is the K = --steps steps back to back; every number below is divided by K (at ~7 ms a step, 30
    # steps are a 0.2 s region: pass a larger --steps for a longer one).  Two passes over the SAME steps:
    # pass 1 is the timed region of `value` (three CUDA events per step); pass 2 repeats K steps with the library's
    # per-launch CUDA events switched on (two event records around each of the ~140 launches of a step cost ~7 % of the
    # step, so they stay out of pass 1) and feeds `roofline` / `kernel_ms_per_step`.
    prof_ms = (ctypes.c_double * 8)()
    prof_n = (ctypes.c_int64 * 8)()
    tot_n0 = (ctypes.c_int64 * 8)()
    tot_n1 = (ctypes.c_int64 * 8)()
    gclk_c, gclk_ns = ctypes.c_double(), ctypes.c_double()

    def timed_pass(n_steps):
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(n_steps)]
        barrier()
        t_w0 = time.perf_counter()
        for k in range(n_steps):
            r = resident[k % len(resident)]
            ev[k][0].record()
            emb = enc.encode_packed(r[0], r[1], r[2], B, B * S, S)
            ev[k][1].record()
            s, i = search_step(queries)
            ev[k][2].record()
        barrier()
        t_w = time.perf_counter() - t_w0
        e_ms = sum(ev[k][0].elapsed_time(ev[k][1]) for k in range(n_steps))
        s_ms = sum(ev[k][1].elapsed_time(ev[k][2]) for k in range(n_steps))
        return e_ms, s_ms, ev[0][0].elapsed_time(ev[-1][2]), t_w, (emb, s, i)

    K = args.steps
    lib.sgpt_profile_read(None, None, tot_n0)
    lib.sgpt_profile_gemm_clock(ctypes.byref(gclk_c), ctypes.byref(gclk_ns))  # reset
    enc_ms, sea_ms, tot_ms, t_wall, (emb, s, i) = timed_pass(K)
    lib.sgpt_profile_read(None, None, tot_n1)
    lib.sgpt_profile_gemm_clock(ctypes.byref(gclk_c), ctypes.byref(gclk_ns))
    launches = sum(int(tot_n1[c] - tot_n0[c]) for c in range(8))
    if args.dump_outputs and rank == 0:
        # what a caller of the timed path receives from its last step: the pooled embeddings and the search result
        dump_outputs(args.dump_outputs, {"embeddings": emb.cpu().numpy(), "search_scores": s.cpu().numpy(),
                                         "search_ids": i.cpu().double().numpy()})
    del emb, s, i
    lib.sgpt_profile_enable(1)
    _, _, prof_tot_ms, _, _ = timed_pass(K)
    lib.sgpt_profile_enable(0)
    lib.sgpt_profile_read(prof_ms, prof_n, tot_n1)

    # ---- phases of the sharded search (N > 1): local search vs exchange + merge --------------------------------------
    phases = None
    if world > 1:
        t_full = time_search(lambda: search_step(queries), 20)
        t_local = time_search(lambda: shard.search_packed(queries, kk, "cos_sim"), 20)
        pk_ = shard.search_packed(queries, kk, "cos_sim")
        t_gather = time_search(lambda: all_gather_packed(pk_), 20)
        gp_ = all_gather_packed(pk_)
        t_merge = time_search(lambda: merge_topk_packed(gp_), 20)
        phases = {"full_search_ms": maxr(t_full), "local_scan_and_selects_ms": maxr(t_local),
                  "exchange_plus_merge_ms": maxr(t_full) - maxr(t_local),
                  "nccl_all_gather_packed_alone_ms": maxr(t_gather), "merge_kernel_alone_ms": maxr(t_merge)}

    # ---- end-to-end loop: public API, HOST buffers in, HOST results out -------------------------------------------
    # Every step copies its inputs host->device (pinned, inside encode_tokens / .to) and its results device->host into
    # pinned buffers.  The D2H copies are asynchronous on the compute stream and double-buffered, exactly like
    # SentenceEncoder.encode, which only synchronises when it hands the embeddings back — so the host can prepare step
    # k+1 while step k runs; all copies complete inside the timed region (barrier at its end).
    emb_host = [torch.empty((B, D), dtype=torch.float32).pin_memory() for _ in range(2)]
    s_host = [torch.empty((NQ, kk), dtype=torch.float32).pin_memory() for _ in range(2)]
    i_host = [torch.empty((NQ, kk), dtype=torch.int64).pin_memory() for _ in range(2)]
    slot_evt = [torch.cuda.Event() for _ in range(2)]

    def e2e_pass(with_search, steps):
        h2d = d2h = 0
        gc_was_on = gc.isenabled()
        if os.environ.get("SGPT_BENCH_GC", "off") == "off":
            gc.collect()
            gc.disable()  # keep the collector's pauses out of the timed loop (DESIGN.md §5.3)
        barrier()
        t0 = time.perf_counter()
        for k in range(steps):
            slot = k % 2
            slot_evt[slot].synchronize()  # the consumer of this slot's previous results is done with them
            emb = enc.encode_tokens(batches[k % 4].numpy(), mask)
            h2d += enc.h2d_bytes_last
            emb_host[slot].copy_(emb, non_blocking=True)
            d2h += emb_host[slot].numel() * 4
            if with_search:
                qd = q_host.to(dev, non_blocking=True)
                h2d += q_host.numel() * 4
                s, i = search_step(qd)
                s_host[slot].copy_(s, non_blocking=True)
                i_host[slot].copy_(i, non_blocking=True)
                d2h += s_host[slot].numel() * 4 + i_host[slot].numel() * 8
            slot_evt[slot].record()
        barrier()
        t_total = time.perf_counter() - t0
        if gc_was_on:
            gc.enable()
        return t_total, h2d, d2h

    # W untimed warm-up steps of exactly this loop first (host->device query copy, copies into the pinned result buffers)
    e2e_pass(True, max(args.warmup, 3))
    e2e_s, h2d, d2h = e2e_pass(True, K)
    e2e_enc_s, _, _ = e2e_pass(False, K)  # encode-only variant (extra key)

    # the same search issued back to back (no encode in between): inside a step it starts in the clock / power state the
    # encoder leaves behind (SM and L2 clocks ~1.6 of 1.96 GHz under the power cap), which slows an HBM-streaming kernel
    # through the L2's per-clock throughput cap (profiles/r02_search_phases_clock_state_and_query_count.jsonl)
    iso_ms = maxr(time_search(lambda: search_step(queries), 50))
    # a DRES-sized query batch (XS:54-60 encodes ALL queries before it scores): 1024 queries per call are scanned 256 at a
    # time by CTA pairs (cta_group::2, M = 256), i.e. 4 passes over the shard instead of 8
    large = None
    if world == 1:
        try:
            q_large = torch.randn(1024, D, generator=gq, device=dev)
            lg_ms = time_search(lambda: shard.search(q_large, kk, "cos_sim"), 10)
            large = {"queries": 1024, "ms_per_search": lg_ms, "queries_per_s": 1024 / (lg_ms / 1e3),
                     "similarity_tflops": 2.0 * 1024 * NDOCS * D / (lg_ms / 1e3) / 1e12,
                     "passes_over_the_shard": 4, "corpus_GBps": 4 * (NDOCS * D * 2 + NDOCS * 4) / (lg_ms / 1e3) / 1e9}
            del q_large
        except Exception as e:  # noqa: BLE001 - reported, never fatal for the main line
            large = {"error": repr(e)[:300]}

    # ---- strong scaling of the exact search over ONE 10 M-doc corpus split across the ranks -----------------------------
    # (north_star: "linear top-k scaling to 8 GPUs on a 10M-doc synthetic corpus"; the main line above is weak scaling at
    # 1 M docs per GPU.)  Two legs: D = 768 (the 125M model's embedding size) and D = 4096 (config 5: sgpt-bloom-7b1).  A
    # failure is reported as an error string and cannot cost the main numbers.
    big = None
    if args.corpus_10m:
        big = {}
        for Dbig in (768, 4096):
            try:
                total = 10_000_000
                lo, hi = shard_range(total, rank, world)
                gb = torch.Generator(device=dev).manual_seed(555 + rank)
                qb_ = torch.randn(NQ, Dbig, generator=gq, device=dev)
                big_shard = CorpusShard(Dbig, hi - lo, device=dev, id_base=lo)
                fill_shard(big_shard, hi - lo, Dbig, gb, dev, queries=qb_, slab=125_000)
                barrier()
                n_it = max(5, min(K, 20))
                big_ms = maxr(time_search(lambda: search_step(qb_, big_shard), n_it))
                loc_ms = maxr(time_search(lambda: big_shard.search_packed(qb_, kk, "cos_sim"), n_it)) if world > 1 else big_ms
                byts = (hi - lo) * (Dbig * 2 + 4)
                big[f"dim_{Dbig}"] = {"corpus_docs": total, "docs_per_gpu": hi - lo, "dim": Dbig, "queries": NQ, "top_k": TOPK,
                                      "ms_per_search": big_ms, "queries_per_s": NQ / (big_ms / 1e3), "scaling": "strong",
                                      "local_scan_and_selects_ms": loc_ms, "exchange_plus_merge_ms": big_ms - loc_ms,
                                      "frac_of_hbm_roofline": (byts / (big_ms / 1e3) / 1e9) / peaks()["hbm"]}
                del big_shard
                torch.cuda.empty_cache()
            except Exception as e:  # noqa: BLE001 - reported, never fatal for the main line
                big[f"dim_{Dbig}"] = {"error": repr(e)[:300]}
    clocks = sampler.stop() if sampler else None

    enc_ms, sea_ms, tot_ms, e2e_s, e2e_enc_s = maxr(enc_ms), maxr(sea_ms), maxr(tot_ms), maxr(e2e_s), maxr(e2e_enc_s)
    extra_legs, overlap, cublas_cal = None, None, None
    if world == 1 and args.other_configs:
        shard_keep = shard
        try:
            cublas_cal = cublas_same_shapes(dev)
        except Exception as e:  # noqa: BLE001
            cublas_cal = {"error": repr(e)[:300]}
        try:
            overlap = fp32_overlap_leg(dev)
        except Exception as e:  # noqa: BLE001
            overlap = {"error": repr(e)[:300]}
        extra_legs = other_config_legs(dev, peaks(), lib, steps=5)
        del shard_keep
    if gather is not None:
        gather.close()
    if rank != 0:
        return
    pk = peaks()
    lin_flops, att_flops = encoder_flops_per_seq(S)
    emb_per_s = world * B * K / (enc_ms / 1e3)
    qps = NQ * K / (sea_ms / 1e3)
    gemm_ms, gemm_n = prof_ms[2], int(prof_n[2])
    gemm_tflops = (lin_flops * B * K) / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else None
    att_ms = prof_ms[3]
    att_tflops = (att_flops * B * K) / (att_ms / 1e3) / 1e12 if att_ms > 0 else None
    sim_ms, sim_n = prof_ms[5], int(prof_n[5])
    sim_bytes = NDOCS * D * 2 + NDOCS * 4 + NQ * D * 2  # corpus shard + inv norms + queries (SURVEY §8d)
    # algorithmic bytes = the shard ONCE per query batch; the two launches of the kernel read it 1 + 1/stride times (the
    # sampled tiles are scanned again by the filtered pass: <= 1/8, 3.7 % at this shape) — that re-read is overhead, not
    # credit: bytes per search / summed device time of both launches
    sim_gbs = sim_bytes * K / (sim_ms / 1e3) / 1e9 if sim_ms > 0 else None
    whole_search_gbs = sim_bytes * K / (sea_ms / 1e3) / 1e9
    traffic, traffic_src = measured_traffic()
    gemm_traffic = traffic.get("linear_gemm", {}).get("dram_bytes_per_launch")
    sim_traffic = traffic.get("similarity_gemm", {}).get("dram_bytes_per_launch")
    sim_launches = max(1, sim_n // max(1, K))
    # algorithmic HBM bytes of the four linear layers of one block (bf16 in, bf16 out / fp32 residual read+write), / 4
    Tt, dm, ffd = B * S, CFG["d_model"], CFG["d_ff"]
    gemm_alg_bytes = (Tt * dm * 2 + 3 * dm * dm * 2 + Tt * 3 * dm * 2        # qkv
                      + Tt * dm * 2 + dm * dm * 2 + 2 * Tt * dm * 4            # out-proj + residual
                      + Tt * dm * 2 + dm * ffd * 2 + Tt * ffd * 2              # c_fc + gelu
                      + Tt * ffd * 2 + dm * ffd * 2 + 2 * Tt * dm * 4) / 4     # c_proj + residual
    gemm_launches_per_step = max(1, gemm_n // max(1, K))
    line = {
        "metric": METRIC, "value": emb_per_s, "unit": "embeddings/s", "n_gpus": world, "steps": K, "warmup": args.warmup,
        "ms_per_step": tot_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic", "config": workload_config(world),
        "timed_region": {"steps_timed": K, "device_seconds": tot_ms / 1e3,
                         "note": "every per-step figure is the region's total divided by steps_timed"},
        "encode_ms_per_step": enc_ms / K, "search_ms_per_step": sea_ms / K,
        "search": {"value": qps, "unit": "queries/s", "corpus_docs": NDOCS * world, "top_k": TOPK,
                   "pairs_per_s": qps * NDOCS * world, "exchange": transport,
                   "whole_search_frac_of_hbm": whole_search_gbs / pk["hbm"],
                   "back_to_back": {"ms_per_search": iso_ms, "queries_per_s": NQ / (iso_ms / 1e3),
                                    "whole_search_frac_of_hbm": sim_bytes / (iso_ms / 1e3) / 1e9 / pk["hbm"],
                                    "note": "50 searches in a row, nothing else on the GPU; the step figure above is "
                                            "measured right after the encoder (power-capped clocks)"},
                   "large_query_batch": large},
        "encoder_model_tflops": (lin_flops + att_flops) * B * world * K / (enc_ms / 1e3) / 1e12,
        "roofline": {"kernel": "gemm_bf16_tn_kernel (tcgen05 linear layers)", "bound": "tensor", "achieved": gemm_tflops,
                     "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                     "frac": (gemm_tflops / pk["tf_sustained"]) if gemm_tflops else None, "traffic": gemm_traffic,
                     "traffic_unit": "DRAM bytes per launch (ncu, read+write, mean over the layer shapes)",
                     "traffic_source": traffic_src, "algorithmic_bytes_per_launch": gemm_alg_bytes,
                     "peak_source": pk["src"] + " (sustained: kernel timed inside a long step)",
                     "timed_in": "pass 2: K steps repeated with per-launch CUDA events on the launching stream",
                     "launches_timed": gemm_n, "avg_launch_ms": gemm_ms / max(1, gemm_n),
                     "algorithmic_flops_per_launch": lin_flops * B / gemm_launches_per_step},
        "roofline_attention": {"kernel": "attention kernel", "bound": "tensor", "achieved": att_tflops,
                               "peak": pk["tf_sustained"], "unit": "TFLOP/s (causal FLOPs 2*S*(S+1)*d per layer per sequence)",
                               "frac": (att_tflops / pk["tf_sustained"]) if att_tflops else None,
                               "device_ms_per_step": att_ms / K, "traffic": traffic.get("attention", {}).get("dram_bytes_per_launch")},
        "roofline_similarity": {"kernel": "gemm_bf16_tn_kernel<EpiFilterRows> (query x corpus, threshold filter)",
                                "bound": "hbm", "achieved": sim_gbs, "peak": pk["hbm"], "unit": "GB/s",
                                "frac": (sim_gbs / pk["hbm"]) if sim_gbs else None,
                                "traffic": sim_traffic * sim_launches if sim_traffic else None,
                                "traffic_unit": "DRAM bytes per search (ncu, read+write, summed over its launches)",
                                "traffic_source": traffic_src,
                                "algorithmic_bytes_per_search": sim_bytes, "launches_per_search": sim_n // max(1, K),
                                "device_ms_per_search": sim_ms / K},
        "kernel_ms_per_step": {c: prof_ms[i] / K for i, c in enumerate(CATS)},
        "profiled_pass_ms_per_step": prof_tot_ms / K,
        "gemm_sm_clock_mhz": (1e3 * gclk_c.value / gclk_ns.value) if gclk_ns.value > 0 else None,
        "gpu_launches": launches,
        "e2e": {"value": world * B * K / e2e_s, "unit": "embeddings/s", "h2d_bytes_per_step": h2d // K,
                "d2h_bytes_per_step": d2h // K, "full_step_ms": 1000 * e2e_s / K,
                "encode_only_embeddings_per_s": world * B * K / e2e_enc_s,
                "search_queries_per_s": None,
                "note": "FULL step through the public API: Encoder.encode_tokens(host ids) -> embeddings copied into pinned "
                        "host memory, host->device queries, exact top-1001 search (+ cross-GPU exchange/merge at N>1), "
                        "device->host scores and ids; double-buffered, all copies inside the timed region; value = "
                        "embeddings of the encode half of every step per second of the whole step"},
        "clocks": clocks, "wall_s_timed_loop": t_wall,
    }
    if merge_verified is not None:
        line["merge_verified"] = merge_verified
        line["search_phases_ms"] = phases
    if big is not None:
        line["search_10m_strong_scaling"] = big
    e2e_search_ms = 1000 * e2e_s / K - 1000 * e2e_enc_s / K
    line["e2e"]["search_queries_per_s"] = NQ / (e2e_search_ms / 1e3) if e2e_search_ms > 0 else None
    if cublas_cal is not None:
        line["roofline"]["cublas_same_shapes"] = cublas_cal
        if gemm_tflops and cublas_cal.get("block_tflops"):
            line["roofline"]["frac_of_cublas_same_shapes"] = gemm_tflops / cublas_cal["block_tflops"]
    if overlap is not None:
        line["topk_overlap_vs_fp32_reference"] = overlap
    if extra_legs is not None:
        line["other_configs"] = extra_legs
    if world == 1 and not args.no_cpu_baseline:
        # batch 256 at least once (VERDICT r01 item 8) when this host can do it in bounded time, else a smaller sample
        probe = cpu_reference_times(weights, enc_batch=8, n_enc=1, search_docs=10_000, warm=True)
        eb = 256 if 256 / max(probe["emb_s"], 1e-6) < 45 else int(min(64, max(4, round(probe["emb_s"] * 5.0))))
        docs = int(min(200_000, max(10_000, round(10_000 * 2.0 / max(probe["t_search"], 1e-3) / 10_000) * 10_000)))
        r = cpu_reference_times(weights, enc_batch=eb, n_enc=1 if eb == 256 else 2, search_docs=docs, warm=False)
        line["cpu_baseline"] = {"value": r["emb_s"], "unit": "embeddings/s", "cores": usable_cores(),
                                "cpu_model": cpu_model_name(),
                                "kind": "port", "sample": r["sample"], "how": r["how"], "search_qps_1m": r["qps_1m"]}
    print(json.dumps(line), flush=True)
    enc.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them returned to DIR/<name>.npy: embeddings "
                         "(float32 [256, 768], rank 0's batch), search_scores (float32 [128, 1001]) and search_ids "
                         "(float64 [128, 1001]); the inputs are seeded, so two builds can be compared output for output")
    ap.add_argument("--no-corpus-10m", dest="corpus_10m", action="store_false",
                    help="skip the extra legs that time the exact search over one 10M-doc corpus (D = 768 and 4096) split "
                         "across the ranks (strong scaling; reported as search_10m_strong_scaling)")
    ap.add_argument("--no-other-configs", dest="other_configs", action="store_false",
                    help="skip the N=1 legs for BASELINE configs 3-5 (1.3B / 5.8B / bloom-7b1 encoders, their shard shapes) "
                         "and the fp32 top-k overlap leg")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
        run_reference(args, rank)
        return
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
