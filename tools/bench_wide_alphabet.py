"""Step and sampler time at wide alphabets (DESIGN.md section 11, "wide alphabets").

    python tools/bench_wide_alphabet.py [--steps 100] [--rounds 3] [--out profiles/wide_alphabet_bench.json]
    python tools/bench_wide_alphabet.py --profile [--out profiles/wide_alphabet_kernels.json]

Step time: B=64, T=500, K=16, L=100, random and peaky logits, V in {64, 65, 128, 256}.  V = 64 runs the
single-launch kernel, V > 64 the chain of stand-alone kernels.  One functional.StepQueue call (one
pgasr_pg_ctc_step_multi call) per region of --steps steps over a pool of distinct batches whose logits exceed the
126 MB L2 (>= 5 batches at V = 256, 32.8 MB each); CUDA events around the region, warm-up first; the V values take
turns, --rounds times, and the median round is reported.
Sampler time: pgasr_softmax_sample at the same B, T, K (Philox draws, probs written, as the step's chain path calls
it), V = 64 (softmax_sample_kernel<64>) against V = 256 (softmax_sample_wide_kernel), CUDA events around 200 calls
rotating over the same pool.
--profile: a separate run under torch.profiler (CUDA activity), 10 steps per V, the mean time of every kernel.
Prints one JSON line (and writes it to --out); the card's name and power limit are part of it.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

B, T, K, L = 64, 500, 16, 100
VS = (64, 65, 128, 256)
L2_BYTES = 126 * 2**20


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 else torch.cuda.get_device_name(0)
    except Exception:                                      # (no nvidia-smi: the torch name only)
        return torch.cuda.get_device_name(0)


def pool_of(V, dev, regime):
    from tests.synth import make_batch
    n = max(3, -(-int(1.25 * L2_BYTES) // (B * T * V * 4)))
    out = []
    for i in range(n):
        lg, tg, il, tl, _ = make_batch(B, T, V, K, L, seed=1000 + 10 * V + i, regime=regime)
        out.append({"logits": torch.from_numpy(lg).to(dev), "targets": torch.from_numpy(tg).to(dev),
                    "in_len": torch.from_numpy(il).to(dev), "tgt_len": torch.from_numpy(tl).to(dev)})
    return out


def run_steps(q, first, n):
    pool = len(q.batches)
    done = 0
    while done < n:
        c = min(pool, n - done)
        q.run(first=first + done, n=c, seed=0x5EED + first + done)
        done += c


def time_region(fn, warm_s=0.05):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < warm_s:
        fn()
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3


def sampler_us(F, pool, calls=200):
    def fn():
        for i in range(calls):
            p = pool[i % len(pool)]
            F.softmax_sample(p["logits"], p["in_len"], K=K, seed=i, return_probs=True)
    return time_region(fn) / calls


def bench(args, F, dev):
    result = {"shape": dict(B=B, T=T, K=K, L=L), "steps": args.steps, "rounds": args.rounds, "gpu": gpu_info(),
              "regimes": {}}
    for regime in ("random", "peaky"):
        pools = {V: pool_of(V, dev, regime) for V in VS}
        queues = {V: F.StepQueue(pools[V], K=K, want=("rewards", "nll")) for V in VS}
        times = {V: [] for V in VS}
        for _ in range(args.rounds):
            for V in VS:
                times[V].append(time_region(lambda: run_steps(queues[V], 0, args.steps)) / args.steps)
        rows = {}
        for V in VS:
            us = statistics.median(times[V])
            rows[str(V)] = {"us_per_step": round(us, 2), "pool": len(pools[V]), "rounds_us": [round(x, 2) for x in times[V]],
                            "path": "single launch" if V <= 64 else "chain"}
        if regime == "random":
            s64 = [sampler_us(F, pools[64]) for _ in range(args.rounds)]
            s256 = [sampler_us(F, pools[256]) for _ in range(args.rounds)]
            a, b = statistics.median(s64), statistics.median(s256)
            result["sampler"] = {"V64_us": round(a, 2), "V256_us": round(b, 2), "ratio": round(b / a, 3), "target_ratio": 4.0,
                                 "V64_rounds": [round(x, 2) for x in s64], "V256_rounds": [round(x, 2) for x in s256]}
        result["regimes"][regime] = rows
        del queues, pools
        torch.cuda.empty_cache()
    return result


def profile(args, F, dev):
    from torch.profiler import ProfilerActivity, profile as tprof
    result = {"shape": dict(B=B, T=T, K=K, L=L), "gpu": gpu_info(), "kernels": {}}
    for V in VS:
        pool = pool_of(V, dev, "random")
        q = F.StepQueue(pool, K=K, want=("rewards", "nll"))
        run_steps(q, 0, 5)
        torch.cuda.synchronize()
        with tprof(activities=[ProfilerActivity.CUDA]) as prof:
            run_steps(q, 0, 10)
            torch.cuda.synchronize()
        rows = {}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            if e.count and t > 0:
                rows[e.key[:120]] = {"count": e.count, "mean_us": round(t / e.count, 2)}
        result["kernels"][str(V)] = rows
        del q, pool
        torch.cuda.empty_cache()
    return result


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_wide_alphabet needs a CUDA device")
    from pgasr_b200 import functional as F
    dev = torch.device("cuda:0")
    result = profile(args, F, dev) if args.profile else bench(args, F, dev)
    line = json.dumps(result)
    print(line)
    out = args.out or os.path.join(ROOT, "profiles",
                                   "wide_alphabet_kernels.json" if args.profile else "wide_alphabet_bench.json")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
