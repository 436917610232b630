"""Step time of the word-level rewards beside the character ones, in one process (DESIGN.md "word reward spec").

    python tools/bench_word_reward.py [--steps 200] [--warmup 20] [--rounds 5] [--out profiles/x.json]

Shape: bench.py's configs[1] (B=64, T=500, V=30, K=16, L=100), text-like transcripts (words of 2-8 random letters
joined by the separator id), random-logit and peaky regimes.  Driver as bench.py's: functional.StepQueue over a pool
of >= 44 distinct batches (more logits than the 126 MB L2), warm-up max(--warmup, 3) steps plus ~30 ms, CUDA events
around --steps steps.  The modes ed, cer, wed, wer take turns, --rounds times; the median round is reported.
Prints one JSON line (and writes it to --out).
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

B, T, V, K, L = 64, 500, 30, 16, 100
BLANK, SPACE = 0, 1
MODES = ("ed", "cer", "wed", "wer")
L2_BYTES = 126 * 2**20


def text_batch(seed, regime):
    from tests.synth import make_batch
    logits, _, in_len, tgt_len, _ = make_batch(B, T, V, K, L, seed=seed)
    rng = np.random.default_rng(seed + 1)
    letters = np.arange(2, V, dtype=np.int32)
    targets = np.zeros((B, L), np.int32)
    for b in range(B):
        row = []
        while len(row) < L:
            row += list(rng.choice(letters, size=int(rng.integers(2, 9)))) + [SPACE]
        targets[b] = row[:L]
    if regime == "peaky":                                  # blank-dominant, the transcript spread over the utterance
        logits[:, :, BLANK] += 10.0
        pos = np.linspace(0, T - 1, L + 2)[1:-1].astype(int)
        for b in range(B):
            logits[b, pos, targets[b]] += 14.0
    return logits, targets, in_len, tgt_len


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown"
    except Exception:                                      # (no nvidia-smi: the torch name only)
        return torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_word_reward needs a CUDA device")
    from pgasr_b200 import functional as F
    dev = torch.device("cuda:0")
    pool = max(44, -(-int(1.25 * L2_BYTES) // (B * T * V * 4)))
    result = {"shape": dict(B=B, T=T, V=V, K=K, L=L), "pool": pool, "steps": args.steps, "rounds": args.rounds,
              "warmup": max(args.warmup, 3), "gpu": gpu_info(), "regimes": {}}
    for regime in ("random", "peaky"):
        devb = []
        for i in range(pool):
            lg, tg, il, tl = text_batch(100 + i, regime)
            devb.append({"logits": torch.from_numpy(lg).to(dev), "targets": torch.from_numpy(tg).to(dev),
                         "in_len": torch.from_numpy(il).to(dev), "tgt_len": torch.from_numpy(tl).to(dev)})
        queues = {m: F.StepQueue(devb, K=K, blank=BLANK, reward=m, want=("rewards", "nll"),
                                 space_id=SPACE if m in F.WORD_REWARDS else None) for m in MODES}

        def run_steps(q, first, n):
            done = 0
            while done < n:
                c = min(pool, n - done)
                q.run(first=first + done, n=c, seed=0x5EED + first + done)
                done += c

        times = {m: [] for m in MODES}
        first = max(args.warmup, 3)
        for r in range(args.rounds):
            for m in MODES:
                q = queues[m]
                run_steps(q, 0, first)
                torch.cuda.synchronize()
                t_w = time.perf_counter()
                while time.perf_counter() - t_w < 0.03:
                    run_steps(q, first, pool)
                    torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run_steps(q, first, args.steps)
                e1.record()
                torch.cuda.synchronize()
                times[m].append(e0.elapsed_time(e1) * 1e3 / args.steps)
        rows = {}
        for m in MODES:
            us = statistics.median(times[m])
            rows[m] = {"us_per_step": round(us, 2), "utt_per_s": round(B / (us * 1e-6), 1),
                       "rounds_us": [round(x, 2) for x in times[m]]}
        for m in ("wed", "wer"):
            rows[m]["vs_ed"] = round(rows[m]["us_per_step"] / rows["ed"]["us_per_step"], 4)
        result["regimes"][regime] = rows
        del queues, devb
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
