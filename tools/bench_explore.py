"""Step time of the exploration controls (temperature, entropy bonus) beside the default step, in one process, and how
often the K draws of an utterance all earn the same reward (DESIGN.md "exploration spec").

    python tools/bench_explore.py [--steps 200] [--warmup 20] [--rounds 5] [--out profiles/x.json]

Shape: bench.py's configs[1] (B=64, T=500, V=30, K=16, L=100), text-like transcripts (tools/bench_word_reward.py),
random-logit and peaky regimes.  Driver as bench.py's: functional.StepQueue over a pool of >= 44 distinct batches
(more logits than the 126 MB L2), warm-up max(--warmup, 3) steps plus ~30 ms, CUDA events around --steps steps.  The
lanes take turns, --rounds times; the median round is reported:
  ed                   defaults (the kernels bench.py times)
  ed_tau1.5            temperature 1.5
  ed_beta0.01          entropy_weight 0.01 (the dense softmax pass under the mean baseline)
  wer_tau1.5_beta0.01  word error rate reward with both
all_equal: per reward mode (ed, wer) and temperature (1, 1.5, 2), the fraction of utterances whose K rewards are all
equal -- under the mean baseline their advantages are all 0 and the PG term contributes nothing -- over 16 batches
(1024 utterances) of each regime.  Prints one JSON line (and writes it to --out).
"""
import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_word_reward import B, BLANK, K, L, L2_BYTES, SPACE, T, V, gpu_info, text_batch  # noqa: E402

LANES = {"ed": dict(reward="ed"),
         "ed_tau1.5": dict(reward="ed", temperature=1.5),
         "ed_beta0.01": dict(reward="ed", entropy_weight=0.01),
         "wer_tau1.5_beta0.01": dict(reward="wer", space_id=SPACE, temperature=1.5, entropy_weight=0.01)}
TAUS = (1.0, 1.5, 2.0)


def all_equal_fraction(F, devb, reward, tau, n_batches=16):
    eq = tot = 0
    for i, b in enumerate(devb[:n_batches]):
        out = F.pg_ctc_step(b["logits"], b["targets"], b["in_len"], b["tgt_len"], K=K, blank=BLANK, reward=reward,
                            seed=0xA11 + i, want=("rewards",), temperature=tau,
                            space_id=SPACE if reward in F.WORD_REWARDS else None)
        R = out["rewards"]
        eq += int((R == R[:, :1]).all(dim=1).sum())
        tot += R.shape[0]
    return round(eq / tot, 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_explore needs a CUDA device")
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
        queues = {n: F.StepQueue(devb, K=K, blank=BLANK, want=("rewards", "nll"), **kw) for n, kw in LANES.items()}

        def run_steps(q, first, n):
            done = 0
            while done < n:
                c = min(pool, n - done)
                q.run(first=first + done, n=c, seed=0x5EED + first + done)
                done += c

        times = {n: [] for n in LANES}
        first = max(args.warmup, 3)
        for r in range(args.rounds):
            for n in LANES:
                q = queues[n]
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
                times[n].append(e0.elapsed_time(e1) * 1e3 / args.steps)
        rows = {}
        for n in LANES:
            us = statistics.median(times[n])
            rows[n] = {"us_per_step": round(us, 2), "utt_per_s": round(B / (us * 1e-6), 1),
                       "rounds_us": [round(x, 2) for x in times[n]]}
        for n in LANES:
            rows[n]["vs_ed"] = round(rows[n]["us_per_step"] / rows["ed"]["us_per_step"], 4)
        result["regimes"][regime] = {"lanes": rows,
                                     "all_equal": {rw: {str(tau): all_equal_fraction(F, devb, rw, tau) for tau in TAUS}
                                                   for rw in ("ed", "wer")}}
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
