"""Oracle of the word-level rewards (DESIGN.md "word reward spec").  TEST INFRASTRUCTURE ONLY.

Built from the C oracle's pieces (oracle/cport.py) without changing them: the sampler, the collapse, the Levenshtein
DP and the policy-gradient / CTC terms are the pinned ones.  What is new is the split into words:
  word_edit_distance  split both id sequences at `sep`, map the words to ids by exact comparison, orc_edit_distance
  pyref_word_distance the same spec restated on strings with str.split(" ") and oracle/pyref's edit_dist
  pg_ctc_step_words   orc_pg_ctc_step with ED_w in place of ED: R = -ED_w, or -ED_w / n_w (orc_pg_loss_grad's one fp32
                      division, with n_w where it divides by len(ref))
"""
import numpy as np

from oracle import cport, pyref


def split_ids(x, sep):
    """str.split(" ") on an id sequence: count(sep) + 1 words, empty words kept."""
    words, cur = [], []
    for c in x:
        if int(c) == sep:
            words.append(tuple(cur))
            cur = []
        else:
            cur.append(int(c))
    words.append(tuple(cur))
    return words


def word_edit_distance(ref, hyp, sep):
    """(ED_w, n_w): the Levenshtein distance between the word sequences (orc_edit_distance on word ids)."""
    table = {}
    wr = [table.setdefault(w, len(table)) for w in split_ids(ref, sep)]
    wh = [table.setdefault(w, len(table)) for w in split_ids(hyp, sep)]
    return int(cport.edit_distance(np.array(wr, np.int32), np.array(wh, np.int32))), len(wr)


def ids_to_str(x, sep):
    """An id sequence as a string: sep -> ' ', every other id -> a character of its own (never a space)."""
    return "".join(" " if int(c) == sep else chr(0x100 + int(c)) for c in x)


def pyref_word_distance(ref, hyp, sep):
    """The spec restated: str.split(" ") on strings, then upstream's edit_dist on the word lists."""
    return pyref.edit_dist(ids_to_str(ref, sep).split(" "), ids_to_str(hyp, sep).split(" "))


def collapse_score_words(samples, targets, in_len, tgt_len, sep, blank=0):
    """hyp_len [B,K] (collapsed, in ids), dist [B,K] = ED_w, n_w [B]."""
    _, hyp_len, _ = cport.collapse_score(samples, targets, in_len, tgt_len, blank)
    B, K, T = samples.shape
    dist = np.zeros((B, K), np.int32)
    n_w = np.zeros(B, np.int32)
    for b in range(B):
        Tb = T if in_len is None else int(in_len[b])
        m = targets.shape[1] if tgt_len is None else int(tgt_len[b])
        ref = targets[b, :m]
        for k in range(K):
            hyp = cport.collapse(samples[b, k, :Tb], blank)
            dist[b, k], n_w[b] = word_edit_distance(ref, hyp, sep)
    return hyp_len, dist, n_w


def pg_ctc_step_words(logits, targets, in_len=None, tgt_len=None, uniforms=None, seed=0, K=16, blank=0, sep=1,
                      reward="wer", baseline_mode=1, baseline_value=0.0, w_pg=1.0, w_ctc=1.0):
    """The whole step with the word rewards, composed as orc_pg_ctc_step composes it.
    -> dict(loss, rewards [B,K] fp32, nll [B], dlogits [B,T,V] fp32, samples, hyp_len, dist)."""
    logits = np.ascontiguousarray(logits, np.float32)
    B, T, V = logits.shape
    if uniforms is not None:
        K = uniforms.shape[1]
    samples, logp = cport.softmax_sample(logits, in_len, uniforms, seed=seed, K=K)
    hyp_len, dist, n_w = collapse_score_words(samples, targets, in_len, tgt_len, sep, blank)
    lpg, rewards, _, gpg = cport.pg_loss_grad(logits, samples, logp, dist, in_len, n_w, targets.shape[1],
                                              reward_mode=1 if reward == "wer" else 0, baseline_mode=baseline_mode,
                                              baseline_value=baseline_value)
    nll, gctc = cport.ctc_loss_grad(logits, targets, in_len, tgt_len, blank)
    loss, dl = w_pg * lpg, w_pg * gpg
    if w_ctc:                                            # (the step has no CTC term then: no 0 * inf for an infeasible alignment)
        loss, dl = loss + w_ctc * (nll.sum() / B), dl + (w_ctc / B) * gctc
    dlogits = dl.astype(np.float32)
    return dict(loss=loss, rewards=rewards, nll=nll, dlogits=dlogits, samples=samples, hyp_len=hyp_len, dist=dist,
                n_w=n_w)
