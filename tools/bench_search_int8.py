"""A/B of the exact search over the same corpus stored as bf16 and as int8 (one GPU, one process).

Per shape: the seeded corpus is generated on the GPU in chunks and added to a bf16 shard and to an int8 shard; the
queries are noisy copies of corpus rows.  bf16 and int8 searches then alternate (CUDA events around `--iters`
back-to-back searches, `--reps` rounds each) and one JSON line per shape reports ms per search for both, their ratio,
the corpus bytes each search reads and that rate as a fraction of the measured HBM copy rate (a 4 GiB device-to-device
copy), the quantizer's GB/s (bytes in + out over kernel time), the top-k overlap of int8 against bf16, and the GPU's
name and power limit read in the same run.  Every shard is far larger than the 126 MB L2, so each search streams it
from HBM.  Output: profiles/r03_search_int8_ab.jsonl (appended).

    python tools/bench_search_int8.py [--shapes 1000000x768x128,...] [--k 1001] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DEFAULT_SHAPES = ("1000000x768x1,1000000x768x128,1000000x768x1024,1000000x2048x128,1250000x4096x128,"
                  "10000000x768x128,10000000x4096x128")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                          "-i", "0"], capture_output=True, text=True).stdout.strip()
    name, power, clock = [x.strip() for x in out.split(",")] if out.count(",") == 2 else (out, "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def copy_rate(dev):
    a = torch.empty(1 << 32, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    rate = 2 * a.numel() * 10 / (e0.elapsed_time(e1) * 1e-3)  # read + write bytes per second
    del a, b
    torch.cuda.empty_cache()
    return rate


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def run_shape(n, D, nq, k, iters, reps, fn, dev, hbm):
    from sgpt_b200 import CorpusShard
    from sgpt_b200.index import quantize_rows_i8

    g = torch.Generator(device=dev).manual_seed(1234 + D)
    b16 = CorpusShard(D, n, device=dev, dtype="bf16")
    i8 = CorpusShard(D, n, device=dev, dtype="int8")
    chunk = max(1, min(n, (1 << 31) // (4 * D)))  # <= 2 GiB of fp32 per chunk
    quant_ms, quant_bytes, q = 0.0, 0, None
    for s0 in range(0, n, chunk):
        c = torch.randn(min(chunk, n - s0), D, generator=g, device=dev)
        if q is None:
            q = c[torch.arange(nq, device=dev) % c.shape[0]] + 0.3 * torch.randn(nq, D, generator=g, device=dev)
        b16.add(c)
        i8.add(c)
        quant_ms += timed(lambda: quantize_rows_i8(c), 3)
        quant_bytes += c.numel() * (4 + 1) + c.shape[0] * 8
        del c
    torch.cuda.synchronize()
    for sh in (b16, i8):  # warm-up: modules, workspace, both paths
        for _ in range(3):
            sh.search(q, k, fn)
    t = {"bf16": [], "int8": []}
    for _ in range(reps):  # alternate the two formats
        t["bf16"].append(timed(lambda: b16.search(q, k, fn), iters))
        t["int8"].append(timed(lambda: i8.search(q, k, fn), iters))
    _, ib = b16.search(q, k, fn)
    _, ii = i8.search(q, k, fn)
    overlap = {}
    for kk in (10, 100, k):
        if kk <= k:
            overlap[str(kk)] = sum(len(set(a[:kk]) & set(b[:kk])) for a, b in zip(ii.tolist(), ib.tolist())) / (nq * kk)
    ms = {f: min(v) for f, v in t.items()}
    read = {"bf16": n * D * 2 + n * 4, "int8": n * D + n * 4}
    del b16, i8
    torch.cuda.empty_cache()
    return {"n": n, "D": D, "queries": nq, "k": k, "score_function": fn,
            "ms_bf16": ms["bf16"], "ms_int8": ms["int8"], "ms_all_bf16": t["bf16"], "ms_all_int8": t["int8"],
            "speedup_int8": ms["bf16"] / ms["int8"],
            "bytes_per_search_bf16": read["bf16"], "bytes_per_search_int8": read["int8"],
            "hbm_frac_bf16": read["bf16"] / (ms["bf16"] * 1e-3) / hbm, "hbm_frac_int8": read["int8"] / (ms["int8"] * 1e-3) / hbm,
            "quantizer_GBps": quant_bytes / (quant_ms * 1e-3) / 1e9, "overlap_int8_vs_bf16": overlap}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default=DEFAULT_SHAPES, help="comma-separated n x D x queries")
    ap.add_argument("--k", type=int, default=1001)
    ap.add_argument("--score", default="cos_sim", choices=["cos_sim", "dot"])
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_search_int8_ab.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_search_int8.py needs a GPU")
    dev = torch.device("cuda:0")
    info = gpu_info()
    hbm = copy_rate(dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    for shape in args.shapes.split(","):
        n, D, nq = (int(x) for x in shape.split("x"))
        t0 = time.time()
        row = run_shape(n, D, nq, args.k, args.iters, args.reps, args.score, dev, hbm)
        row.update(info, hbm_copy_GBps=hbm / 1e9, wall_s=time.time() - t0)
        line = json.dumps(row)
        print(line, flush=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
