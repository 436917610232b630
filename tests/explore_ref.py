"""Oracle of the exploration controls (DESIGN.md "exploration spec").  TEST INFRASTRUCTURE ONLY.

Built from the C oracle's pieces (oracle/cport.py) and tests/word_ref.py without changing them:
  z' = fl32(z * theta), theta = fl32(1 / tau)   numpy's fp32 product rounds exactly like __fmul_rn
  sampler, collapse, rewards, PG loss / grad    the pinned ones, run on z' (the policy that was sampled); the PG
                                                gradient then times theta (the chain factor of z' = theta z)
  entropy_and_grad                              H_bt, H_b and d H / d z' in fp64 numpy
  CTC                                           orc_ctc_loss_grad on the UNTEMPERED z
"""
import numpy as np

from oracle import cport
from tests import word_ref

CHAR_REWARD = {"ed": 0, "cer": 1}


def theta_of(temperature):
    return np.float32(1.0) / np.float32(temperature)


def tempered(logits, temperature):
    return (np.ascontiguousarray(logits, np.float32) * theta_of(temperature)).astype(np.float32)


def entropy_and_grad(zp, in_len=None):
    """H [B] (sum over t < in_len[b] of H(softmax(z'_bt))) and dH_b/dz' [B,T,V], both fp64."""
    z = np.asarray(zp, np.float64)
    B, T, V = z.shape
    m = z.max(axis=2, keepdims=True)
    lp = z - m - np.log(np.exp(z - m).sum(axis=2, keepdims=True))
    p = np.exp(lp)
    plogp = np.where(p > 0, p * np.where(p > 0, lp, 0.0), 0.0)   # 0 log 0 = 0 (a logit of -inf: log p = -inf)
    Ht = -plogp.sum(axis=2)                                       # [B,T]
    live = np.arange(T)[None, :] < (np.full(B, T) if in_len is None else np.asarray(in_len))[:, None]
    Ht = np.where(live, Ht, 0.0)
    dH = np.where(p > 0, -p * (np.where(p > 0, lp, 0.0) + Ht[:, :, None]), 0.0)
    dH = np.where(live[:, :, None], dH, 0.0)
    return Ht.sum(axis=1), dH


def pg_ctc_step_explore(logits, targets, in_len=None, tgt_len=None, uniforms=None, seed=0, K=16, blank=0, reward="ed",
                        baseline_mode=1, baseline_value=0.0, w_pg=1.0, w_ctc=1.0, temperature=1.0, w_ent=0.0, sep=None):
    """The whole step with temperature and entropy bonus:
    loss = w_pg L_pg(z') + w_ctc mean_b nll_b(z) - w_ent mean_b H_b(z').
    -> dict(loss, loss_scale (sum of the terms' magnitudes), rewards, nll, dlogits fp32, samples, hyp_len, dist, logp,
    entropy)."""
    logits = np.ascontiguousarray(logits, np.float32)
    targets = np.ascontiguousarray(targets, np.int32)
    B, T, V = logits.shape
    Lmax = targets.shape[1]
    if uniforms is not None:
        K = uniforms.shape[1]
    theta = theta_of(temperature)
    zp = tempered(logits, temperature)
    samples, logp = cport.softmax_sample(zp, in_len, uniforms, seed=seed, K=K)
    if reward in ("wed", "wer"):
        hyp_len, dist, n_w = word_ref.collapse_score_words(samples, targets, in_len, tgt_len, sep, blank)
        lpg, rewards, _, gpg = cport.pg_loss_grad(zp, samples, logp, dist, in_len, n_w, Lmax,
                                                  reward_mode=1 if reward == "wer" else 0,
                                                  baseline_mode=baseline_mode, baseline_value=baseline_value)
    elif reward == "ed_to_go":
        _, hyp_len, dist = cport.collapse_score(samples, targets, in_len, tgt_len, blank)
        lpg, rewards, _, _, gpg = cport.pg_togo_loss_grad(zp, samples, targets, in_len, tgt_len, blank,
                                                          baseline_mode=baseline_mode, baseline_value=baseline_value)
    else:
        _, hyp_len, dist = cport.collapse_score(samples, targets, in_len, tgt_len, blank)
        lpg, rewards, _, gpg = cport.pg_loss_grad(zp, samples, logp, dist, in_len, tgt_len, Lmax,
                                                  reward_mode=CHAR_REWARD[reward], baseline_mode=baseline_mode,
                                                  baseline_value=baseline_value)
    H, dH = entropy_and_grad(zp, in_len)
    loss = w_pg * lpg - w_ent * H.sum() / B
    # magnitude of the summed terms: the scale the loss's fp32 rounding follows when the terms cancel
    loss_scale = abs(w_pg * lpg) + abs(w_ent * H.sum() / B)
    dl = float(theta) * (w_pg * gpg - (w_ent / B) * dH)
    nll = None
    if w_ctc:                                            # (no CTC term: no 0 * inf for an infeasible alignment)
        nll, gctc = cport.ctc_loss_grad(logits, targets, in_len, tgt_len, blank)
        loss, dl = loss + w_ctc * (nll.sum() / B), dl + (w_ctc / B) * gctc
        loss_scale += abs(w_ctc * nll.sum() / B)
    return dict(loss=loss, loss_scale=loss_scale, rewards=rewards, nll=nll, dlogits=dl.astype(np.float32), dlogits64=dl, samples=samples,
                hyp_len=hyp_len, dist=dist, logp=logp, entropy=H)
