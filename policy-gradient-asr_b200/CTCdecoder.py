"""Drop-in for upstream CTCdecoder.py: collapse_fn (GPU) and CTCDecoder (prefix beam search).

collapse_fn(preds: str) -> str keeps a character iff it differs from its predecessor
(upstream CTCdecoder.py:119-131); it does not remove blanks, exactly like upstream.
CTCDecoder.decode is the eval-time prefix beam search (upstream CTCdecoder.py:41-116; SURVEY.md section 8f.2),
one CTA per utterance on the GPU; decode_batch decodes a whole dev set in one launch.
"""

import numpy as np
import torch

from . import functional as F

NEG_INF = -float("inf")


def collapse_batch(strings):
    """collapse_fn over a list of strings in one launch."""
    if not strings:
        return []
    for s in strings:
        if not isinstance(s, str):
            raise TypeError("can only concatenate str (not \"%s\") to str" % type(s).__name__)
    alphabet = sorted(set("".join(strings)))
    if len(alphabet) > 256:
        raise ValueError("collapse_fn: more than 256 distinct characters in one batch")
    if not torch.cuda.is_available():
        raise RuntimeError("pgasr_b200.CTCdecoder.collapse_fn needs a CUDA device (no CPU fallback)")
    to_id = {c: i for i, c in enumerate(alphabet)}
    T = max(1, max(len(s) for s in strings))
    rows = np.zeros((len(strings), T), np.uint8)
    for i, s in enumerate(strings):
        rows[i, :len(s)] = [to_id[c] for c in s]
    dev = torch.device("cuda", torch.cuda.current_device())
    lens = torch.tensor([len(s) for s in strings], dtype=torch.int32, device=dev)
    out, out_len = F.collapse(torch.from_numpy(rows).to(dev), lens, rows_per_len=1, blank=None)
    out, out_len = out.cpu().numpy(), out_len.cpu().numpy()
    return ["".join(alphabet[x] for x in out[i, :out_len[i]]) for i in range(len(strings))]


def collapse_fn(preds):
    """Upstream CTCdecoder.py:119-131."""
    return collapse_batch([preds])[0]


class CTCDecoder:
    """Prefix beam search with the upstream constructor and decode() signature
    (CTCdecoder.py:23-25, 41-116): decode(probs[T,V] post-softmax, beam_size=100, blank=0)
    -> (labels tuple, negative log-likelihood), computed by the batched GPU kernel (csrc/beam.cu).
    Alphabets of up to 256 classes, beams of up to 128 (up to 104 at 256 classes: the candidate table lives in
    shared memory); larger requests raise PgasrError (status -2)."""

    def __init__(self, alphabet):
        self.alphabet = alphabet
        self.NEG_INF = NEG_INF

    def decode_batch(self, probs_list, beam_size=100, blank=0):
        """decode() for a list of [T_i, V] arrays in one launch (one CTA per utterance)."""
        if not torch.cuda.is_available():
            raise RuntimeError("pgasr_b200.CTCdecoder.CTCDecoder.decode needs a CUDA device (no CPU fallback)")
        if not probs_list:
            return []
        arrs = [np.asarray(p, dtype=np.float64) for p in probs_list]
        V = arrs[0].shape[1]
        T = max(1, max(a.shape[0] for a in arrs))
        batch = np.zeros((len(arrs), T, V), np.float64)
        for i, a in enumerate(arrs):
            if a.ndim != 2 or a.shape[1] != V:
                raise ValueError("every probs array must be [T, V] with the same V")
            batch[i, :a.shape[0]] = a
        dev = torch.device("cuda", torch.cuda.current_device())
        lens = torch.tensor([a.shape[0] for a in arrs], dtype=torch.int32, device=dev)
        labels, label_len, nll = F.ctc_beam_search(torch.from_numpy(batch).to(dev), lens, beam_size=beam_size, blank=blank)
        labels, label_len, nll = labels.cpu().numpy(), label_len.cpu().numpy(), nll.cpu().numpy()
        return [(tuple(int(x) for x in labels[i, :label_len[i]]), float(nll[i])) for i in range(len(arrs))]

    def decode(self, probs, beam_size=100, blank=0):
        return self.decode_batch([probs], beam_size=beam_size, blank=blank)[0]
