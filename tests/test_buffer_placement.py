"""Buffers at any element offset, and the multi-step calls of the character modes against the oracle.

include/pgasr.h: an array argument needs only its element's natural alignment.  A view with a storage offset (the
criterion on model_out[:, 1:], an out= tensor carved from a larger buffer, a C caller's pointer) is therefore a valid
logits / dlogits / output pointer, while torch's allocator only ever hands out 512-byte aligned storage.  The kernels
take 16-byte accesses where the pointer allows them and 4-byte ones where it does not; the arithmetic is the same, so
every result of a call on offset buffers must equal the call on freshly allocated ones bit for bit.

The multi-step entry point runs its steps on several streams with paired PG CTAs (two utterances per CTA) and without
programmatic dependent launch; every step of such a call is checked here against the C oracle directly.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import cport
from tests import explore_ref, word_ref
from tests.placement import at_offset, multi_step, offset_outputs
from tests.synth import make_batch, make_word_batch
from tests.test_explore import check as check_explore
from tests.test_word_reward import check_against_oracle as check_words

gpu = pytest.mark.gpu
RTOL = 1e-4
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dev_t(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def rel_err(got, want):
    want = np.asarray(want, np.float64)
    got = np.asarray(got, np.float64)
    return np.abs(got - want).max() / max(np.abs(want).max(), 1e-30)


def grad_close(got, want):
    """tests/test_gpu_parity.py's element-wise bar."""
    want = np.asarray(want, np.float64)
    got = np.asarray(got, np.float64)
    atol = max(1e-7, 1e-5 * float(np.abs(want).max()))
    return not (np.abs(got - want) > RTOL * np.abs(want) + atol).any()


def char_oracle(host, K, reward="ed", baseline="mean", baseline_value=-0.5, w_pg=1.0, w_ctc=1.0, seed=0,
                uniforms=True, blank=0):
    from pgasr_b200 import functional as F
    lg, tg, il, tl, uni = host
    uni = uni if uniforms else None
    loss, R, nll, dl = cport.pg_ctc_step(lg, tg, il, tl, uni, seed=seed, K=K, blank=blank,
                                         reward_mode=F.REWARD_MODES[reward], baseline_mode=F.BASELINE_MODES[baseline],
                                         baseline_value=baseline_value, w_pg=w_pg, w_ctc=w_ctc)
    s, logp = cport.softmax_sample(lg, il, uni, seed=seed, K=K)
    _, hl, d = cport.collapse_score(s, tg, il, tl, blank=blank)
    if w_ctc == 0.0:
        # the step's loss is then the PG term alone; the oracle's sum would be 0 * inf = nan for an utterance without
        # an alignment
        loss = w_pg * cport.pg_loss_grad(lg, s, logp, d, il, tl, tg.shape[1], F.REWARD_MODES[reward],
                                         F.BASELINE_MODES[baseline], baseline_value, want_grad=False)[0]
    return dict(loss=loss, rewards=R, nll=nll, dlogits=dl, samples=s, hyp_len=hl, dist=d)


def check_char(out, ref, w_pg=1.0, w_ctc=1.0):
    """step_case's bars (tests/test_gpu_parity.py), with utterances that have no alignment (nll = +inf) allowed."""
    if w_pg:
        for name in ("samples", "hyp_len", "dist"):
            assert np.array_equal(out[name].cpu().numpy(), ref[name]), name
        assert np.array_equal(out["rewards"].cpu().numpy(), ref["rewards"])
    if w_ctc:
        nll, want = out["nll"].cpu().numpy().astype(np.float64), ref["nll"]
        assert np.array_equal(np.isinf(nll), np.isinf(want))
        ok = np.isfinite(want)
        assert (np.abs(nll[ok] - want[ok]) <= RTOL * np.abs(want[ok])).all()
    loss, want = float(out["loss"].reshape(-1)[0]), ref["loss"]
    if np.isfinite(want):
        assert abs(loss - want) <= RTOL * abs(want) + 1e-5
    else:
        assert loss == want
    dl = out["dlogits"].cpu().numpy()
    assert rel_err(dl, ref["dlogits"]) < RTOL
    assert grad_close(dl, ref["dlogits"])


def togo_oracle_check(out, host, baseline="mean", baseline_value=-0.5, w_ctc=1.0):
    """tests/test_gpu_parity.py::test_step_reward_to_go's bars."""
    from pgasr_b200 import functional as F
    lg, tg, il, tl, uni = host
    B = lg.shape[0]
    samples = out["samples"].cpu().numpy()
    s_ref, _ = cport.softmax_sample(lg, il, uni)
    assert np.array_equal(samples, s_ref)
    loss_pg, R, to_go, r_pos, g_pg = cport.pg_togo_loss_grad(lg, samples, tg, il, tl,
                                                             baseline_mode=F.BASELINE_MODES[baseline],
                                                             baseline_value=baseline_value)
    assert np.array_equal(out["to_go"].cpu().numpy(), to_go)
    assert np.array_equal(out["r_pos"].cpu().numpy(), r_pos)
    assert np.array_equal(out["rewards"].cpu().numpy(), R)
    want_g = g_pg
    if w_ctc:
        _, g_ctc = cport.ctc_loss_grad(lg, tg, il, tl)
        want_g = g_pg + (w_ctc / B) * g_ctc
    got = out["dlogits"].cpu().numpy()
    assert rel_err(got, want_g) < RTOL and grad_close(got, want_g)


# ---------------------------------------------------------------- A. single steps at offsets
CHAR_WANT = ("rewards", "nll", "logp", "dist", "hyp_len", "samples")
# name: (B, T, V, K, L), step keywords, outputs; every shape has T*V % 4 == 0, so the 16-byte paths are the ones meant
PATHS = {
    "tile_block_workers": ((3, 200, 30, 8, 40), dict(reward="cer", baseline="loo"), CHAR_WANT),
    "tile_round1_workers": ((2, 260, 40, 8, 50), dict(), CHAR_WANT),
    "ctc_role_streams": ((1, 1300, 64, 4, 150), dict(), CHAR_WANT),
    "both_roles_stream": ((2, 2000, 30, 16, 100), dict(reward="cer", baseline="loo"), CHAR_WANT),
    "spl32": ((2, 2000, 30, 4, 400), dict(), CHAR_WANT),
    # (without a CTC term nll is not computed, and not written)
    "no_ctc_term": ((4, 120, 30, 8, 24), dict(ctc_weight=0.0, baseline="none"), ("rewards", "logp", "dist", "hyp_len",
                                                                                  "samples")),
    "no_pg_term": ((4, 120, 30, 8, 24), dict(pg_weight=0.0), ("nll",)),
    "ed_to_go": ((3, 120, 30, 8, 20), dict(reward="ed_to_go"),
                 ("rewards", "samples", "to_go", "r_pos", "nll", "dist", "hyp_len")),
    "wer": ((5, 120, 30, 8, 24), dict(reward="wer", space_id=1), CHAR_WANT),
    "explore": ((5, 150, 30, 8, 30), dict(temperature=1.5, entropy_weight=0.01), CHAR_WANT + ("entropy",)),
    "chain": ((2, 1800, 30, 64, 50), dict(reward="cer", baseline="loo"), CHAR_WANT),
}


def path_batch(name, shape):
    B, T, V, K, L = shape
    if name == "wer":
        return make_word_batch(B, T, V, K, L, seed=T + K, ragged=True, regime="peaky")
    return make_batch(B, T, V, K, L, seed=T + K + len(name), ragged=True)


def step_at(cuda, host, K, kw, want, where, off):
    """The step with logits (and uniforms, targets, lengths) and / or every output `off` elements into a buffer."""
    from pgasr_b200 import functional as F
    lg, tg, il, tl, uni = host
    ins = where in ("logits", "both")
    put = (lambda a: at_offset(a, off, cuda)) if ins else (lambda a: dev_t(a, cuda))
    out = None
    if where in ("dlogits", "both"):
        B, T, V = lg.shape
        out = offset_outputs(F, (B, T, V, K, tg.shape[1]), cuda, want, off)
    res = F.pg_ctc_step(put(lg), put(tg), put(il), put(tl), K=K, uniforms=put(uni), seed=5, baseline_value=-0.5,
                        want=want, out=out, **kw)
    if out is not None:
        for name in out:                                  # written in place: no copy was made on the way
            assert res[name].data_ptr() == out[name].data_ptr()
    return {k: res[k].reshape(-1).clone() for k in ("loss", "dlogits") + tuple(want)}


@gpu
@pytest.mark.parametrize("name", list(PATHS))
def test_step_at_unaligned_offsets(cuda, name):
    """Logits only, outputs only, and both at float offsets 1, 2, 3 (uint8 samples and int16 reward-to-go then sit at
    odd byte offsets): every output equals the call on fresh tensors bit for bit; the call with both misaligned also
    meets the oracle's bars."""
    shape, kw, want = PATHS[name]
    B, T, V, K, L = shape
    assert T * V % 4 == 0
    host = path_batch(name, shape)
    fresh = step_at(cuda, host, K, kw, want, None, 0)
    got = None
    for where in ("logits", "dlogits", "both"):
        for off in (1, 2, 3):
            got = step_at(cuda, host, K, kw, want, where, off)
            for k in fresh:
                assert torch.equal(got[k], fresh[k]), (where, off, k)
    res = {k: got[k].reshape(s) for k, s in _out_shapes(shape, want).items()}
    lg, tg, il, tl, uni = host
    w_pg, w_ctc = kw.get("pg_weight", 1.0), kw.get("ctc_weight", 1.0)
    if name == "wer":
        ref = word_ref.pg_ctc_step_words(lg, tg, il, tl, uni, seed=5, K=K, sep=1, reward="wer", baseline_mode=1,
                                         baseline_value=-0.5)
        check_words(res, ref)
    elif name == "explore":
        ref = explore_ref.pg_ctc_step_explore(lg, tg, il, tl, uni, seed=5, K=K, reward="ed", baseline_mode=1,
                                              baseline_value=-0.5, temperature=1.5, w_ent=0.01)
        check_explore(res, ref)
    elif name == "ed_to_go":
        togo_oracle_check(res, host)
    else:
        check_char(res, char_oracle(host, K, kw.get("reward", "ed"), kw.get("baseline", "mean"), w_pg=w_pg,
                                    w_ctc=w_ctc, seed=5), w_pg, w_ctc)


def _out_shapes(shape, want):
    B, T, V, K, L = shape
    s = {"loss": (1,), "dlogits": (B, T, V)}
    for name in want:
        s[name] = (B,) if name in ("nll", "entropy") else (B, K, T) if name in ("samples", "to_go", "r_pos") else (B, K)
    return s


# ---------------------------------------------------------------- B. stand-alone entry points at offsets
def _ctc_c(cuda, logits, probs, targets, il, tl, dlogits, accumulate):
    """pgasr_ctc_loss_grad with the caller's dlogits (functional.ctc_loss_grad only accepts one to accumulate into)."""
    from pgasr_b200 import _native
    src = logits if logits is not None else probs
    B, T, V = src.shape
    Lmax = targets.shape[1]
    nbytes = _native.lib().pgasr_ctc_workspace_bytes(B, T, V, Lmax)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=cuda)
    nll = torch.empty((B,), dtype=torch.float32, device=cuda)
    p = lambda t: None if t is None else t.data_ptr()
    _native.call("pgasr_ctc_loss_grad", p(logits), p(probs), p(targets), p(il), p(tl), B, T, V, Lmax, 0, 0.5,
                 accumulate, p(nll), p(dlogits), p(ws), nbytes, torch.cuda.current_stream().cuda_stream)
    return nll, dlogits


@gpu
@pytest.mark.parametrize("V", [30, 40])
def test_ctc_loss_grad_at_offsets(cuda, V):
    """The CTC-only single-launch kernel, and the classic kernel (accumulate; probabilities only)."""
    B, T, L = 3, 160, 30
    lg, tg, il, tl, _ = make_batch(B, T, V, 1, L, seed=V, ragged=True)
    assert T * V % 4 == 0
    probs = torch.softmax(dev_t(lg, cuda), -1)
    d = lambda a: dev_t(a, cuda)
    base = [_ctc_c(cuda, d(lg), None, d(tg), d(il), d(tl), torch.empty((B, T, V), device=cuda), 0),
            _ctc_c(cuda, d(lg), None, d(tg), d(il), d(tl), torch.full((B, T, V), 0.25, device=cuda), 1),
            _ctc_c(cuda, None, probs, d(tg), d(il), d(tl), torch.empty((B, T, V), device=cuda), 0)]
    nll_ref, g_ref = cport.ctc_loss_grad(lg, tg, il, tl)
    assert np.abs(base[0][0].cpu().numpy() / nll_ref - 1).max() < RTOL
    assert rel_err(base[0][1].cpu().numpy() / 0.5, g_ref) < RTOL        # (grad_scale 0.5)
    for off in (1, 2, 3):
        o = lambda a: at_offset(a, off, cuda)
        got = [_ctc_c(cuda, o(lg), None, o(tg), o(il), o(tl), at_offset(((B, T, V), torch.float32), off, cuda), 0),
               _ctc_c(cuda, o(lg), None, o(tg), o(il), o(tl), at_offset(torch.full((B, T, V), 0.25, device=cuda),
                                                                         off, cuda), 1),
               _ctc_c(cuda, None, at_offset(probs, off, cuda), o(tg), o(il), o(tl),
                      at_offset(((B, T, V), torch.float32), off, cuda), 0)]
        for i, ((n0, g0), (n1, g1)) in enumerate(zip(base, got)):
            assert torch.equal(n0, n1) and torch.equal(g0, g1), (off, i)


@gpu
def test_sampler_pg_grad_and_distances_at_offsets(cuda):
    """softmax_sample (logits, uniforms, samples, logp, probs), pg_grad (probs, out), collapse, edit_distance,
    word_edit_distance and edit_distance_tokens with uint8 rows at byte offsets 1-3 and int32 rows at offsets."""
    from pgasr_b200 import _native, functional as F
    B, T, V, K, L = 3, 120, 30, 8, 24
    lg, tg, il, tl, uni = make_batch(B, T, V, K, L, seed=4, ragged=True)
    stream = lambda: torch.cuda.current_stream().cuda_stream

    def sample(logits, il_, uniforms, off):
        samples = at_offset(((B, K, T), torch.uint8), off, cuda) if off else torch.empty((B, K, T), dtype=torch.uint8,
                                                                                            device=cuda)
        logp = at_offset(((B, K), torch.float32), off, cuda) if off else torch.empty((B, K), device=cuda)
        probs = at_offset(((B, T, V), torch.float32), off, cuda) if off else torch.empty((B, T, V), device=cuda)
        _native.call("pgasr_softmax_sample", logits.data_ptr(), il_.data_ptr(), uniforms.data_ptr(), 0, B, T, V, K,
                     samples.data_ptr(), logp.data_ptr(), probs.data_ptr(), stream())
        return samples, logp, probs

    s0, lp0, p0 = sample(dev_t(lg, cuda), dev_t(il, cuda), dev_t(uni, cuda), 0)
    s_ref, _ = cport.softmax_sample(lg, il, uni)
    assert np.array_equal(s0.cpu().numpy(), s_ref)
    adv = torch.randn(B, K, device=cuda)
    g0 = F.pg_grad(s0, adv, dev_t(il, cuda), probs=p0, scale=0.1, out=torch.full((B, T, V), 0.5, device=cuda))
    c0, n0 = F.collapse(s0, dev_t(il, cuda))
    d0 = F.edit_distance(c0, n0.reshape(-1), dev_t(tg, cuda), dev_t(tl, cuda), rows_per_ref=K, vocab=V)
    w0 = F.word_edit_distance(c0, n0.reshape(-1), dev_t(tg, cuda), 1, dev_t(tl, cuda), rows_per_ref=K)
    t0 = F.edit_distance_tokens(c0.reshape(B * K, T).to(torch.int32), n0.reshape(-1), dev_t(tg, cuda),
                                dev_t(tl, cuda), rows_per_ref=K)
    for off in (1, 2, 3):
        o = lambda a: at_offset(a, off, cuda)
        s1, lp1, p1 = sample(o(lg), o(il), o(uni), off)
        assert torch.equal(s1, s0) and torch.equal(lp1, lp0) and torch.equal(p1, p0), off
        out = at_offset(torch.full((B, T, V), 0.5, device=cuda), off, cuda)
        g1 = F.pg_grad(s1, o(adv), o(il), probs=p1, scale=0.1, out=out)
        assert g1.data_ptr() == out.data_ptr() and torch.equal(g1, g0), off
        c1, n1 = F.collapse(o(s0), o(il))
        assert torch.equal(c1, c0) and torch.equal(n1, n0), off
        hy, hl, rf, rl = o(c0), o(n0.reshape(-1)), o(tg), o(tl)
        assert torch.equal(F.edit_distance(hy, hl, rf, rl, rows_per_ref=K, vocab=V), d0), off
        w1 = F.word_edit_distance(hy, hl, rf, 1, rl, rows_per_ref=K)
        assert torch.equal(w1[0], w0[0]) and torch.equal(w1[1], w0[1]), off
        t1 = F.edit_distance_tokens(o(c0.reshape(B * K, T).to(torch.int32)), hl, rf, rl, rows_per_ref=K)
        assert torch.equal(t1, t0), off


# ---------------------------------------------------------------- C. multi-step call, mixed placement
@gpu
@pytest.mark.parametrize("mode", ["char", "wer", "explore"])
def test_multi_step_mixed_placement_equals_single_steps(cuda, mode):
    """Records of one pgasr_pg_ctc_step_multi* call alternate aligned and offset buffers (offset dlogits in the
    records, which StepQueue cannot build); five steps, so every lane takes more than one.  Each step equals its
    single step on fresh tensors bit for bit."""
    from pgasr_b200 import functional as F
    B, T, V, K, L = 5, 200, 30, 8, 40
    kw = dict(K=K, reward="ed", baseline="loo")
    want = CHAR_WANT
    if mode == "wer":
        kw.update(reward="wer", space_id=1)
    if mode == "explore":
        kw.update(temperature=1.5, entropy_weight=0.01)
        want = CHAR_WANT + ("entropy",)
    mk = (lambda s: make_word_batch(B, T, V, K, L, seed=s, ragged=True)) if mode == "wer" else \
        (lambda s: make_batch(B, T, V, K, L, seed=s, ragged=True))
    hosts = [mk(60 + i) for i in range(5)]
    offs = [0, 1, 0, 3, 2]
    batches, outs = [], []
    for (lg, tg, il, tl, uni), off in zip(hosts, offs):
        put = (lambda a: at_offset(a, off, cuda)) if off else (lambda a: dev_t(a, cuda))
        batches.append(dict(logits=put(lg), targets=put(tg), in_len=put(il), tgt_len=put(tl), uniforms=put(uni)))
        outs.append(offset_outputs(F, (B, T, V, K, L), cuda, want, off) if off else
                    F._alloc_outputs((B, T, V, K, L), cuda, want))
    multi_step(F, batches, outs, seed=21, **kw)
    torch.cuda.synchronize()
    for i, (lg, tg, il, tl, uni) in enumerate(hosts):
        o = F.pg_ctc_step(dev_t(lg, cuda), dev_t(tg, cuda), dev_t(il, cuda), dev_t(tl, cuda),
                          uniforms=dev_t(uni, cuda), seed=21 + i, want=want, **kw)
        for name in ("loss", "dlogits") + want:
            assert torch.equal(outs[i][name].reshape(-1), o[name].reshape(-1)), (i, offs[i], name)


# ---------------------------------------------------------------- D. the criterion slot
@gpu
def test_criterion_on_a_view_with_an_offset(cuda):
    """criterion(model_out[:, 1:], t) for a model that emits one extra leading frame: at B = 1 the slice is contiguous
    and starts 120 bytes (8 mod 16) into the storage.  The gradient equals the one of a cloned input."""
    import pgasr_b200
    B, T, V, K, L = 1, 500, 30, 16, 80
    lg, tg, il, tl, uni = make_batch(B, T + 1, V, K, L, seed=13)
    grads = []
    for clone in (False, True):
        model_out = dev_t(lg, cuda).requires_grad_(True)
        x = model_out[:, 1:]
        if clone:
            x = x.clone()
        else:
            assert x.is_contiguous() and x.data_ptr() % 16 == 8
        crit = pgasr_b200.PolicyGradCTCLoss(K=K, seed=3)
        loss = crit(x, dev_t(tg, cuda), torch.full((B,), T, dtype=torch.int32, device=cuda), dev_t(tl, cuda))
        loss.backward()
        grads.append((loss.detach().clone(), model_out.grad.clone()))
    assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1])
    assert (grads[0][1][:, 0] == 0).all() and float(grads[0][1].abs().sum()) > 0


# ---------------------------------------------------------------- 3. character-mode multi-step calls vs the oracle
def _pair_smem(T, V, K, L):
    """Shared memory of a PG CTA that serves two utterances, CDF rows included: fused.cu's pairing test
    (pg_role_smem(..., cdf = true, nutt = 2) <= kFusedSmemLimit), mirrored from fused.cu / fused_args.cuh."""
    S = 2 * L + 1
    spl = next(s for s in (4, 8, 16, 32) if S <= 32 * s)
    threads, W = (256 if spl >= 32 else 512), spl // 2
    Tp, Tp2 = (T + 15) & ~15, (T // 2 + 16) & ~15
    ub = 2 * K * Tp + K * Tp2 + 2 * (V + 1) * W * 4 + ((K + 7) & ~7) * (W * 32 + 2) * 2
    ub = ((ub + 15) & ~15) + (threads // 32) * 64 * 8 + 3 * 64 * 4 + 16
    ub = (ub + 15) & ~15
    return ((T * V * 4 + 15) & ~15) + 2 * ub + 16 + threads * 33 * 4 + 16


SMEM_LIMIT = 220 * 1024       # fused.cu: kFusedSmemLimit
# T = 671 is the last length at V = 30, K = 16, L = 40 whose PG pair fits (225072 bytes), T = 672 the first whose pair
# does not (225696); the single-utterance PG role fits at both.  The values follow fused.cu's pairing test
# (pg_role_smem(..., cdf = true, nutt = 2) <= kFusedSmemLimit) and fused_args.cuh's pg_u_bytes.  The library does not
# report whether it pairs, so _pair_smem restates that arithmetic, and a change to either C function has to be carried
# into it and into the two byte counts test_pair_threshold pins.
T_PAIR_FITS = 671

QUEUE_CASES = [
    # (B, T, V, K, L, reward, baseline, w_pg, w_ctc, n_steps)
    (2, 120, 30, 8, 24, "ed", "mean", 1.0, 1.0, 2),
    (3, 120, 30, 8, 24, "cer", "loo", 1.0, 1.0, 4),
    (5, 120, 30, 8, 24, "ed", "none", 1.0, 1.0, 7),
    (5, 120, 30, 8, 24, "cer", "value", 1.0, 1.0, 4),
    (3, 150, 2, 5, 12, "ed", "loo", 1.0, 1.0, 4),
    (5, 150, 31, 8, 24, "cer", "mean", 1.0, 1.0, 4),
    (3, 150, 32, 16, 30, "ed", "value", 1.0, 1.0, 7),
    (3, 150, 33, 8, 24, "ed", "loo", 1.0, 1.0, 4),
    (5, 120, 30, 8, 24, "ed", "loo", 1.0, 0.0, 4),
    (3, 120, 30, 8, 24, "cer", "mean", 0.0, 1.0, 4),
    (3, T_PAIR_FITS, 30, 16, 40, "ed", "loo", 1.0, 1.0, 4),
    (3, T_PAIR_FITS + 1, 30, 16, 40, "ed", "loo", 1.0, 1.0, 4),
]


def test_pair_threshold():
    assert _pair_smem(T_PAIR_FITS, 30, 16, 40) == 225072 <= SMEM_LIMIT
    assert _pair_smem(T_PAIR_FITS + 1, 30, 16, 40) == 225696 > SMEM_LIMIT


@gpu
@pytest.mark.parametrize("B,T,V,K,L,reward,baseline,w_pg,w_ctc,n", QUEUE_CASES)
def test_step_queue_against_the_oracle(cuda, B, T, V, K, L, reward, baseline, w_pg, w_ctc, n):
    """StepQueue steps (several streams, paired PG CTAs -- the last CTA of an odd B serves one utterance) checked
    against the C oracle, with an utterance without frames and (under 'ed') an empty transcript in every batch."""
    from pgasr_b200 import functional as F
    hosts = []
    for i in range(n):
        lg, tg, il, tl, uni = make_batch(B, T, V, K, L, seed=1000 * B + T + V + i, ragged=True,
                                         regime="peaky" if i % 2 else "random")
        il[i % B] = 0
        if reward == "ed":                               # (an empty transcript has no CER)
            j = (i + 1) % B
            tl[j] = 0
            tg[j] = 0
        hosts.append((lg, tg, il, tl, uni))
    batches = [dict(logits=dev_t(lg, cuda), targets=dev_t(tg, cuda), in_len=dev_t(il, cuda), tgt_len=dev_t(tl, cuda),
                    uniforms=dev_t(uni, cuda)) for lg, tg, il, tl, uni in hosts]
    want = CHAR_WANT if w_pg else ("nll",)
    q = F.StepQueue(batches, K=K, reward=reward, baseline=baseline, baseline_value=-0.5, pg_weight=w_pg,
                    ctc_weight=w_ctc, want=want)
    q.run(first=0, n=n, seed=0)
    torch.cuda.synchronize()
    for i, host in enumerate(hosts):
        check_char(q.outputs[i], char_oracle(host, K, reward, baseline, w_pg=w_pg, w_ctc=w_ctc), w_pg, w_ctc)


# ---------------------------------------------------------------- 4. the A/B switches
SWITCHES = ["PGASR_NO_BULK_TILE", "PGASR_NO_PAIR", "PGASR_NO_CDF_SMEM", "PGASR_NO_BW", "PGASR_NO_OVERLAP",
            "PGASR_LANES=1", "PGASR_LANES=4", "PGASR_NO_PDL", "PGASR_PDL_THROUGHPUT"]
# switches that change only how data is copied or scheduled (or, NO_PAIR, which CTA serves an utterance): bit for bit
BIT_IDENTICAL = {"PGASR_NO_BULK_TILE", "PGASR_NO_PAIR", "PGASR_NO_OVERLAP", "PGASR_LANES=1", "PGASR_LANES=4",
                 "PGASR_NO_PDL", "PGASR_PDL_THROUGHPUT"}
EXACT_OUTPUTS = ("samples", "dist", "hyp_len", "rewards", "to_go", "r_pos")


def _run_matrix(path, switch=None):
    env = {k: v for k, v in os.environ.items() if not k.startswith("PGASR_")}
    if switch:
        name, _, value = switch.partition("=")
        env[name] = value or "1"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "variant_matrix.py"), str(path)], env=env,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (switch, r.stdout[-2000:], r.stderr[-3000:])
    with np.load(path) as z:
        return {k: z[k] for k in z.files}


@gpu
def test_switch_matrix(cuda, tmp_path):
    """tools/variant_matrix.py once with default settings and once per A/B switch (each reads its switch once per
    process, hence a subprocess each).  Copy and scheduling switches and NO_PAIR: every output bit for bit.
    NO_CDF_SMEM: samples, distances and rewards bit for bit, the rest at the oracle's bars.  NO_BW: the oracle's bars."""
    base = _run_matrix(tmp_path / "default.npz")
    assert any(k.endswith("/dlogits") for k in base)
    for switch in SWITCHES:
        got = _run_matrix(tmp_path / (switch.replace("=", "_") + ".npz"), switch)
        assert sorted(got) == sorted(base), switch
        for key, want in base.items():
            g = got[key]
            name = key.rsplit("/", 1)[1]
            if switch in BIT_IDENTICAL or name in EXACT_OUTPUTS:
                assert np.array_equal(g.view(np.uint8), want.view(np.uint8)), (switch, key)
            elif name == "dlogits":
                assert rel_err(g, want) < RTOL and grad_close(g, want), (switch, key)
            else:                                         # loss, nll, logp, entropy
                w = want.astype(np.float64)
                assert np.array_equal(np.isinf(g), np.isinf(w)), (switch, key)
                ok = np.isfinite(w)
                assert (np.abs(g[ok] - w[ok]) <= RTOL * np.maximum(np.abs(w[ok]), 1.0)).all(), (switch, key)
