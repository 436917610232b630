"""TEST INFRASTRUCTURE -- the reference CPU leg of bench.py (BASELINE.md section 3, SURVEY.md 8d).

The hot path as an upstream maintainer would have had to run it with upstream's own code: the REAL
`CTCdecoder.collapse_fn` (CTCdecoder.py:119-131) and `metrics.edit_dist` (metrics.py:4-21), imported from
oracle/_ref/ (verbatim copies made by oracle/make_ref.py), around torch-CPU for the parts upstream has no code for
(softmax + multinomial sampling, the REINFORCE surrogate and its autograd, `F.ctc_loss` forward + backward --
the arithmetic upstream's requirements.txt:1 would have supplied).  Only bench.py's CPU legs and tests call this.
"""
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")


def available():
    return all(os.path.exists(os.path.join(REF_DIR, f)) for f in ("metrics.py", "CTCdecoder.py"))


def _upstream():
    import importlib.util
    mods = {}
    for name in ("metrics", "CTCdecoder"):
        spec = importlib.util.spec_from_file_location(f"_pgasr_upstream_{name}", os.path.join(REF_DIR, name + ".py"))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        mods[name] = m
    return mods["metrics"].edit_dist, mods["CTCdecoder"].collapse_fn


def step(logits, targets, in_len, tgt_len, K, w_pg=1.0, w_ctc=1.0, seed=0, upstream=None):
    """One PG + CTC loss step on the CPU.  Returns (loss, rewards [B,K], dlogits [B,T,V]) as numpy arrays.
    `upstream`: the (edit_dist, collapse_fn) pair to run instead of the copies in oracle/_ref."""
    import numpy as np
    import torch
    edit_dist, collapse_fn = upstream or _upstream()
    z = torch.tensor(logits, dtype=torch.float32, requires_grad=True)
    B, T, V = z.shape
    logp_all = torch.log_softmax(z, dim=-1)
    loss = torch.zeros((), dtype=torch.float32)
    rewards = np.zeros((B, K), np.float32)
    if w_pg:
        g = torch.Generator().manual_seed(int(seed))
        terms = []
        for b in range(B):
            Tb, Lb = int(in_len[b]), int(tgt_len[b])
            ref = "".join(chr(48 + int(c)) for c in targets[b, :Lb])
            smp = torch.multinomial(logp_all[b, :Tb].detach().exp(), K, replacement=True, generator=g)   # [Tb, K]
            R = []
            for k in range(K):
                path = "".join(chr(48 + int(c)) for c in smp[:, k])
                hyp = collapse_fn(path).replace(chr(48), "")            # merge repeats (upstream), then drop the blank
                R.append(-float(edit_dist(ref, hyp)[0]))
            R = torch.tensor(R)
            rewards[b] = R.numpy()
            A = R - R.mean()
            lp = logp_all[b, :Tb].gather(1, smp).sum(0)                 # [K] sequence log-probs
            terms.append(-(A * lp).sum())
        loss = loss + w_pg * torch.stack(terms).sum() / (B * K)
    if w_ctc:
        nll = torch.nn.functional.ctc_loss(logp_all.transpose(0, 1), torch.tensor(targets, dtype=torch.long),
                                           torch.tensor(in_len, dtype=torch.long), torch.tensor(tgt_len, dtype=torch.long),
                                           blank=0, reduction="none", zero_infinity=False)
        loss = loss + w_ctc * nll.mean()
    loss.backward()
    return float(loss.detach()), rewards, z.grad.numpy()


def time_step(B, T, V, K, L, regime="random", w_pg=1.0, w_ctc=1.0):
    import torch
    sys.path.insert(0, os.path.dirname(HERE))
    from tests.synth import make_batch
    logits, targets, in_len, tgt_len, _ = make_batch(B, T, V, K, L, seed=4321, regime=regime)
    t0 = time.perf_counter()
    step(logits, targets, in_len, tgt_len, K, w_pg, w_ctc)
    dt = time.perf_counter() - t0
    return {"value": B / dt, "unit": "utt/s", "cores": 1, "kind": "reference",
            "torch_threads": torch.get_num_threads(),
            "sample": f"1 step x {B} utterances (T={T},V={V},K={K},L={L}, {regime}): upstream collapse_fn + edit_dist "
                      "(pure Python, one core) around torch-CPU multinomial / autograd / F.ctc_loss"}
