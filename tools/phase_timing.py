"""Phase timing of the fused kernel (CTA of utterance 0) from the -DPGASR_TIMING build:
    python policy-gradient-asr_b200/build.py --timing
    PGASR_LIB=policy-gradient-asr_b200/lib/libpgasr_b200_timing.so python tools/phase_timing.py
PROF_REWARD=wed|wer: the word-level rewards on tools/bench_word_reward.py's text-like transcripts (space id 1;
PROF_REGIME=random|peaky); the "collapse" phase then includes the word phase, split as W1 (transcripts) / W2.
"""
import ctypes
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from pgasr_b200 import _native, functional as F  # noqa: E402
from tests.synth import make_batch  # noqa: E402

B = int(os.environ.get("PROF_B", "64"))
dev = torch.device("cuda:0")
REWARD = os.environ.get("PROF_REWARD", "ed")
WORD = REWARD in F.WORD_REWARDS
KW = dict(reward=REWARD, space_id=1) if WORD else {}
if WORD:
    from tools.bench_word_reward import text_batch  # noqa: E402
    make_batch = lambda B_, T_, V_, K_, L_, seed: (*text_batch(seed, os.environ.get("PROF_REGIME", "random")), None)  # noqa: E731
lg, tg, il, tl, _ = make_batch(B, 500, 30, 16, 100, seed=1)
t = lambda a: torch.from_numpy(a).to(dev)
lg, tg, il, tl = t(lg), t(tg), t(il), t(tl)
lib = _native.lib()
buf = (ctypes.c_longlong * 64)()
ws = None
for mode, (wp, wc) in {"both": (1.0, 1.0), "ctc": (0.0, 1.0), "pg": (1.0, 0.0)}.items():
    for i in range(3):
        out = F.pg_ctc_step(lg, tg, il, tl, K=16, seed=i, workspace=ws, pg_weight=wp, ctc_weight=wc, **KW)
        ws = out["workspace"]
    lib.pgasr_debug_read(buf, 1)
    out = F.pg_ctc_step(lg, tg, il, tl, K=16, seed=7, workspace=ws, pg_weight=wp, ctc_weight=wc, **KW)
    lib.pgasr_debug_read(buf, 1)
    d = list(buf)
    print(f"== {mode} (cycles)")
    if wc:
        print(f" ctc: zero-rows {d[1]-d[0]}  softmax-tile {d[2]-d[1]}  lattice+grad {d[3]-d[2]}  total {d[3]-d[0]}")
        print(f" ctc CTA outside the role's stamps: start->grid-dependency wait passed {d[5]-d[4]}  ->role entry {d[6]-d[5]}  ->transcript and lengths in {d[0]-d[6]}"
              f"  | flag {d[9]-d[3]}  done ticket {d[7]-d[9]}  ->exit {d[8]-d[7]}  | CTA total {d[8]-d[4]}")
        print(f" walker start after the tile barrier: alpha +{d[10]-d[2]}  beta +{d[14]-d[2]}   mid barrier passed at: alpha +{d[12]-d[2]}  beta +{d[16]-d[2]}")
        print(f" alpha walker: first-half {d[11]-d[10]}  mid-wait {d[12]-d[11]}  second-half {d[13]-d[12]}")
        print(f" beta  walker: first-half {d[15]-d[14]}  mid-wait {d[16]-d[15]}  second-half {d[17]-d[16]}")
        print(f" alpha worker0: waiting {d[20]}  busy {d[21]}   beta worker0: waiting {d[22]}  busy {d[23]}")
        print(f" alpha worker0: phaseA {d[25]}  phaseB {d[26]}")
        print(f" block workers: alpha A0 ring-wait {d[40]} buffer-wait {d[41]} busy {d[42]} | beta A0 {d[44]} {d[45]} {d[46]}")
        print(f"                alpha B0 block-wait {d[48]} rows {d[49]} copy-out {d[50]} | beta B0 {d[52]} {d[53]} {d[54]}")
        print(f"                alpha B0 rows split: pre {d[56]} loop {d[57]} blocks {d[58]} trips/block {d[59]}")
    if wp:
        names = ["tile-load", "sample", "collapse", "myers", "advantages", "grad-tile", "flag-wait", "rmw-out"]
        print(f" pg sampling split (thread 0): cdf build {d[60]-d[31]}  draws {d[32]-d[60]}")
        print(" pg:  " + "  ".join(f"{n} {d[31+i]-d[30+i]}" for i, n in enumerate(names)) + f"  total {d[38]-d[30]}")
        if WORD:
            print(f" pg word phase: collapse {d[61]-d[32]}  W1 transcripts {d[62]-d[61]}  W2 hypotheses {d[33]-d[62]}")

if WORD:       # (the per-CTA wall times below are recorded by the character-mode kernel only)
    sys.exit(0)

# per-CTA wall times of the last fused launch (globaltimer ns): role start/end spread over the grid
import numpy as np  # noqa: E402
out = F.pg_ctc_step(lg, tg, il, tl, K=16, seed=9, workspace=ws, **KW)
n = 2 * B
arr = (ctypes.c_ulonglong * (3 * n))()
assert lib.pgasr_debug_cta_times(arr, n) == 0
t = np.array(list(arr), dtype=np.float64).reshape(n, 3)
t0 = t[:, 0].min()
t = (t - t0) / 1e3
for name, sl in (("CTC role CTAs", slice(0, B)), ("PG role CTAs", slice(B, n))):
    x = t[sl]
    print(f" {name}: start {x[:,0].min():6.1f}..{x[:,0].max():6.1f} us   role end {x[:,1].min():6.1f}..{x[:,1].max():6.1f} "
          f"(median {np.median(x[:,1]):6.1f})   exit {x[:,2].min():6.1f}..{x[:,2].max():6.1f}   "
          f"role duration median {np.median(x[:,1]-x[:,0]):6.1f} max {np.max(x[:,1]-x[:,0]):6.1f}")

# does a CTC CTA's duration follow the largest class count of its transcript (the gather's tail loop)?
tgn = tg.cpu().numpy()
cmax = np.array([np.bincount(tgn[b], minlength=30)[1:].max() for b in range(B)])
dur = t[:B, 1] - t[:B, 0]
order = np.argsort(dur)
print(" CTC role duration by utterance (us) / max labels of one class:")
print("   fastest: " + "  ".join(f"{dur[i]:.1f}/{cmax[i]}" for i in order[:8]))
print("   slowest: " + "  ".join(f"{dur[i]:.1f}/{cmax[i]}" for i in order[-8:]))
print(f"   corr(duration, cmax) = {np.corrcoef(dur, cmax)[0, 1]:.2f}")

# the same per-CTA times with consecutive steps overlapping (pgasr_pg_ctc_step_multi, two lanes): how long a CTA lives
# when the SMs are shared with the neighbouring steps (entries are overwritten by whichever step finishes last)
batches = []
for i in range(8):
    a, b, c, d, _ = make_batch(B, 500, 30, 16, 100, seed=100 + i)
    batches.append({"logits": torch.from_numpy(a).to(dev), "targets": torch.from_numpy(b).to(dev),
                    "in_len": torch.from_numpy(c).to(dev), "tgt_len": torch.from_numpy(d).to(dev)})
q = F.StepQueue(batches, K=16, **KW)
for rep in range(3):
    q.run(first=0, n=8, seed=rep)
torch.cuda.synchronize()
arr = (ctypes.c_ulonglong * (3 * n))()
assert lib.pgasr_debug_cta_times(arr, n) == 0
t = np.array(list(arr), dtype=np.float64).reshape(n, 3) / 1e3
for name, sl in (("CTC role CTAs", slice(0, B)), ("PG role CTAs", slice(B, n))):
    x = t[sl]
    dur = x[:, 1] - x[:, 0]
    print(f" overlapped steps, {name}: role duration median {np.median(dur):6.1f} us  min {dur.min():6.1f}  max {dur.max():6.1f}")

# SM time per CTA in the steady state of overlapped steps (timing build: per-role sums over every CTA of a long run)
if hasattr(lib, "pgasr_debug_role_times"):
    r8 = (ctypes.c_ulonglong * 8)()
    NS = 32                                                # steps per call: fill and drain are ~3 % of a call
    q = F.StepQueue([batches[i % 8] for i in range(NS)], K=16, **KW)
    for rep in range(6):
        q.run(first=0, n=NS, seed=10 + rep)
    lib.pgasr_debug_role_times(r8, 1)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    nrep = 12
    for rep in range(nrep):
        q.run(first=0, n=NS, seed=20 + rep)
    ev1.record()
    torch.cuda.synchronize()
    lib.pgasr_debug_role_times(r8, 0)
    r = list(r8)
    us_step = ev0.elapsed_time(ev1) * 1e3 / (NS * nrep)
    print(f" steady state, {NS * nrep} overlapped steps: {us_step:.2f} us per step")
    tot = 0.0
    for i, name in enumerate(("CTC", "PG")):
        n_, w_, a_, f_ = r[4 * i:4 * i + 4]
        if n_:
            print(f"   {name} CTAs: {n_ / (NS * nrep):.0f} per step, at the grid-dependency wait {w_ / n_ / 1e3:6.2f} us, "
                  f"active {a_ / n_ / 1e3:6.2f} us" + (f" (of which waiting for CTC flags {f_ / n_ / 1e3:6.2f} us)" if i else ""))
            tot += (w_ + a_) / (NS * nrep) / 1e3
    print(f"   SM time per step {tot:.0f} us = {tot / 148:.2f} us x 148 SMs")
