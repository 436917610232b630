"""Seeded synthetic inputs shared by the CPU and GPU tests, by bench.py and by the tools (SURVEY.md section 8d): batches
with character transcripts (make_batch) and with word-level ones (make_word_batch)."""
import numpy as np


def make_batch(B, T, V, K, L, seed=0, regime="random", ragged=False):
    """logits [B,T,V] fp32, targets [B,L] int32 (no blanks), in_len [B], tgt_len [B], uniforms [B,K,T]."""
    rng = np.random.default_rng(seed)
    targets = rng.integers(1, V, size=(B, L)).astype(np.int32)
    if ragged:
        in_len = rng.integers(max(T // 2, 1), T + 1, size=B).astype(np.int32)
        tgt_len = rng.integers(max(L // 2, 1), L + 1, size=B).astype(np.int32)
        tgt_len = np.minimum(tgt_len, np.maximum(in_len // 3, 1)).astype(np.int32)
    else:
        in_len = np.full(B, T, np.int32)
        tgt_len = np.full(B, L, np.int32)
    logits = (2.0 * rng.standard_normal((B, T, V))).astype(np.float32)
    if regime == "peaky":
        # blank-dominant posteriors with the transcript spread over the utterance
        for b in range(B):
            Tb, Lb = int(in_len[b]), int(tgt_len[b])
            pos = np.linspace(0, Tb - 1, Lb + 2)[1:-1].astype(int)
            boost = np.zeros((T,), np.int64)
            boost[pos] = targets[b, :Lb]
            logits[b, np.arange(T), boost] += 6.0
    for b in range(B):
        targets[b, tgt_len[b]:] = 0
    uniforms = rng.random((B, K, T), dtype=np.float32)
    uniforms = np.minimum(uniforms, np.float32(1.0 - 2.0 ** -24))
    return logits, targets, in_len, tgt_len, uniforms


def text_targets(rng, B, L, V, blank, sep, tgt_len, style="text"):
    """Transcripts: words of 2-8 random letters joined by the separator ('text'), only separators ('allsep'), or
    separators at random, doubled ones included ('random')."""
    letters = np.array([c for c in range(V) if c not in (blank, sep)], np.int32)
    tg = np.zeros((B, L), np.int32)
    for b in range(B):
        m = int(tgt_len[b])
        if style == "allsep":
            row = [sep] * m
        elif style == "random":
            row = list(rng.choice(letters, size=m))
            for i in range(m):
                if rng.random() < 0.25:
                    row[i] = sep
        else:
            row = []
            while len(row) < m:
                row += list(rng.choice(letters, size=int(rng.integers(2, 9)))) + [sep]
            row = row[:m]
        tg[b, :m] = row
    return tg


def make_word_batch(B, T, V, K, L, seed, regime="random", ragged=False, blank=0, sep=1, style="text"):
    logits, _, in_len, tgt_len, uni = make_batch(B, T, V, K, L, seed=seed, ragged=ragged)
    rng = np.random.default_rng(seed + 7)
    targets = text_targets(rng, B, L, V, blank, sep, tgt_len, style)
    if regime == "peaky":                                           # the transcript spread over the utterance
        logits[:, :, blank] += 10.0
        for b in range(B):
            Tb, Lb = int(in_len[b]), int(tgt_len[b])
            if Lb == 0:
                continue
            pos = np.linspace(0, Tb - 1, Lb + 2)[1:-1].astype(int)
            logits[b, pos, targets[b, :Lb]] += 14.0
    return logits, targets, in_len, tgt_len, uni
