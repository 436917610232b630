"""Every output of a fixed list of steps, for comparing the library's A/B switches (PGASR_NO_BULK_TILE, PGASR_NO_PAIR,
PGASR_NO_CDF_SMEM, PGASR_NO_BW, PGASR_NO_OVERLAP, PGASR_LANES, PGASR_NO_PDL, PGASR_PDL_THROUGHPUT).

    PGASR_NO_PAIR=1 python tools/variant_matrix.py out.npz

The library reads each switch once per process, so one run covers one setting; tests/test_buffer_placement.py runs
this once with default settings and once per switch and compares the files.  The cases cover single steps and
multi-step calls, character, word and exploration modes, and aligned as well as offset buffers.  Keys of the .npz:
"<case>/<step>/<output>".
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from pgasr_b200 import functional as F  # noqa: E402
from tests.placement import at_offset, multi_step, offset_outputs  # noqa: E402
from tests.synth import make_batch, make_word_batch  # noqa: E402

WANT = ("rewards", "nll", "logp", "dist", "hyp_len", "samples")
SHAPE = (5, 200, 30, 8, 40)        # B, T, V, K, L: block workers, CDF rows in shared memory, paired PG CTAs in a queue

# name, single step or queue, offset of each step's buffers (elements; 0 = fresh tensors), step keywords, outputs
CASES = [
    ("char_single", "single", [0], dict(reward="ed", baseline="loo"), WANT),
    ("char_single_offset", "single", [3], dict(reward="cer", baseline="mean"), WANT),
    ("togo_single_offset", "single", [1], dict(reward="ed_to_go", baseline="mean"),
     ("rewards", "samples", "to_go", "r_pos", "nll", "dist", "hyp_len")),
    ("char_queue", "queue", [0, 1, 0, 2, 0], dict(reward="ed", baseline="loo"), WANT),
    ("word_queue", "queue", [0, 0, 3, 0, 1], dict(reward="wer", baseline="loo", space_id=1), WANT),
    ("explore_single_offset", "single", [2], dict(temperature=1.5, entropy_weight=0.01), WANT + ("entropy",)),
    ("explore_queue", "queue", [2, 0, 0, 1, 0], dict(reward="wed", baseline="mean", space_id=1, temperature=1.5,
                                                       entropy_weight=0.01), WANT + ("entropy",)),
]


def batch(dev, host, off):
    put = (lambda a: at_offset(a, off, dev)) if off else (lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev))
    lg, tg, il, tl, uni = host
    return dict(logits=put(lg), targets=put(tg), in_len=put(il), tgt_len=put(tl), uniforms=put(uni))


def run(path):
    dev = torch.device("cuda:0")
    B, T, V, K, L = SHAPE
    res = {}
    for ci, (name, kind, offs, kw, want) in enumerate(CASES):
        words = kw.get("space_id") is not None
        mk = make_word_batch if words else (lambda *a: make_batch(*a[:5], seed=a[5], ragged=True))
        hosts = [mk(B, T, V, K, L, 100 * ci + i) for i in range(len(offs))]
        batches = [batch(dev, h, off) for h, off in zip(hosts, offs)]
        outs = [offset_outputs(F, (B, T, V, K, L), dev, want, off) if off else
                F._alloc_outputs((B, T, V, K, L), dev, want) for off in offs]
        if kind == "single":
            b = batches[0]
            F.pg_ctc_step(b["logits"], b["targets"], b["in_len"], b["tgt_len"], K=K, uniforms=b["uniforms"], seed=7,
                          want=want, out=outs[0], **kw)
        else:
            multi_step(F, batches, outs, K, seed=7, **kw)
        torch.cuda.synchronize()
        for i, o in enumerate(outs):
            for k, t in o.items():
                res[f"{name}/{i}/{k}"] = t.cpu().numpy()
    np.savez(path, **res)
    print(f"{len(res)} arrays from {len(CASES)} cases -> {path}")


if __name__ == "__main__":
    if len(sys.argv) != 2 or not sys.argv[1].endswith(".npz"):
        sys.exit("usage: python tools/variant_matrix.py OUT.npz")
    run(sys.argv[1])
