"""Word-level rewards (DESIGN.md "word reward spec"): reward='wed' (-ED_w) and 'wer' (-ED_w / n_w).

CPU: the word oracle (tests/word_ref.py) against upstream's golden evaluate / edit_dist vectors and against a
str.split restatement; argument validation of the C ABI; the Python-level checks.
GPU (-m gpu): the fused word phase, the chain path and the stand-alone kernel against the oracle -- samples,
hyp_len, dist and rewards bit-exact, loss and dlogits within 1e-4.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import cport, pyref
from tests import word_ref
from tests.synth import make_batch

RTOL = 1e-4


def str_ids(s, alphabet):
    return np.array([alphabet.index(c) for c in s], np.int32)


def alphabet_of(*strs):
    return ["<pad>", " "] + sorted(set("".join(strs)) - {" "})


# ---------------------------------------------------------------- CPU: the oracle
def test_word_oracle_reproduces_evaluate_wer(golden):
    for e in golden["evaluate"]:
        al = alphabet_of(e["ref"], e["hyp"])
        d, n = word_ref.word_edit_distance(str_ids(e["ref"], al), str_ids(e["hyp"], al), al.index(" "))
        assert d / n == e["out"][1], e
    al = alphabet_of("ab cd")
    assert word_ref.word_edit_distance(str_ids("ab cd", al), str_ids("ab  cd", al), 1) == (1, 2)   # empty word kept


def test_word_oracle_reproduces_word_edit_dist_golden(golden):
    cases = [e for e in golden["edit_dist"] if e["kind"] == "words"]
    assert cases
    for e in cases:
        al = alphabet_of(e["ref"], e["hyp"])
        got = word_ref.word_edit_distance(str_ids(e["ref"], al), str_ids(e["hyp"], al), al.index(" "))
        assert list(got) == e["out"], e


def test_word_oracle_edge_cases():
    sep = 1
    assert word_ref.split_ids([], sep) == [()]
    assert word_ref.split_ids([1, 1], sep) == [(), (), ()]
    assert word_ref.word_edit_distance([], [], sep) == (0, 1)          # len("".split(" ")) == 1: never a division by 0
    assert word_ref.word_edit_distance([], [2, 1, 3], sep) == (2, 1)
    assert word_ref.word_edit_distance([1, 1, 1], [], sep) == (3, 4)
    assert word_ref.word_edit_distance([2, 3, 1, 2, 3], [2, 3, 1, 2, 3], sep) == (0, 2)


def random_id_seq(rng, sep, n_max=24):
    kind = rng.integers(6)
    n = int(rng.integers(0, n_max + 1))
    if kind == 0:
        return np.array([], np.int32)
    if kind == 1:
        return np.full(n, sep, np.int32)                            # all separators
    x = rng.integers(2, 2 + int(rng.integers(1, 4)), size=n).astype(np.int32)   # small alphabets: many equal words
    x[rng.random(n) < 0.3] = sep
    if kind == 2 and n:
        x[0] = sep                                                  # leading
    if kind == 3 and n:
        x[-1] = sep                                                 # trailing
    if kind == 4 and n >= 3:
        i = int(rng.integers(0, n - 1))
        x[i:i + 2] = sep                                            # doubled
    return x


def test_c_oracle_equals_str_split_restatement():
    rng = np.random.default_rng(1234)
    sep = 1
    for _ in range(600):
        ref, hyp = random_id_seq(rng, sep), random_id_seq(rng, sep)
        assert word_ref.word_edit_distance(ref, hyp, sep) == word_ref.pyref_word_distance(ref, hyp, sep), (ref, hyp)


# ---------------------------------------------------------------- CPU: validation
def _multi_args(reward_mode, blank=0, V=30):
    from pgasr_b200 import _native
    io = _native.StepIO()
    dummy = C.c_void_p(1 << 20)                                     # 256-byte aligned, never dereferenced
    return io, (C.byref(io), 1, 0, 4, 50, V, 4, 10, blank, reward_mode, 1, 0.0, 1.0, 1.0), dummy


def test_step_rejects_bad_separator_and_word_modes_elsewhere():
    from pgasr_b200 import _native
    L = _native.lib()
    nbytes = 1 << 30
    _, head, ws = _multi_args(4)
    assert L.pgasr_pg_ctc_step_multi_ws(*head, 0, ws, nbytes, None) == -1          # separator == blank
    assert L.pgasr_pg_ctc_step_multi_ws(*head, 30, ws, nbytes, None) == -1         # separator >= V
    assert L.pgasr_pg_ctc_step_multi_ws(*head, -1, ws, nbytes, None) == -1         # separator < 0
    _, head3, _ = _multi_args(3, blank=2)
    assert L.pgasr_pg_ctc_step_multi_ws(*head3, 2, ws, nbytes, None) == -1
    _, head5, _ = _multi_args(5)
    assert L.pgasr_pg_ctc_step_multi_ws(*head5, 1, ws, nbytes, None) == -1         # no such reward mode
    for mode in (3, 4):                                                            # word modes only through _ws
        _, h, _ = _multi_args(mode)
        assert L.pgasr_pg_ctc_step_multi(*h, ws, nbytes, None) == -1
        assert L.pgasr_pg_ctc_step(ws, ws, None, None, None, 0, 4, 50, 30, 4, 10, 0, mode, 1, 0.0, 1.0, 1.0,
                                   ws, ws, None, None, None, None, None, None, ws, nbytes, None) == -1
    assert L.pgasr_word_edit_distance_u8(ws, ws, 4, 10, ws, None, 2, 10, -1, ws, None, None) == -1
    assert L.pgasr_word_edit_distance_u8(ws, ws, 4, 10, ws, None, 2, 512, 1, ws, None, None) == -2   # ref_len <= 511


def test_python_level_word_mode_checks():
    import pgasr_b200
    from pgasr_b200 import functional as F
    assert F.REWARD_MODES["wed"] == 3 and F.REWARD_MODES["wer"] == 4
    with pytest.raises(ValueError):
        pgasr_b200.PolicyGradCTCLoss(reward="wer")                  # no space_id
    with pytest.raises(ValueError):
        pgasr_b200.PolicyGradCTCLoss(reward="wed", blank=0, space_id=0)
    crit = pgasr_b200.PolicyGradCTCLoss(reward="wer", space_id=1)
    assert crit.space_id == 1
    with pytest.raises(ValueError):
        F._step_entry("wer", 0, None)
    with pytest.raises(ValueError):
        pgasr_b200.HostPipeline(2, 20, 30, 4, 5, reward="wer")      # host-buffer API: character modes only
    assert F._step_entry("ed", 0, None) == ("pgasr_pg_ctc_step_multi", ())
    assert F._step_entry("wed", 0, 3) == ("pgasr_pg_ctc_step_multi_ws", (3,))


# ---------------------------------------------------------------- GPU
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


def dev_t(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def rel_err(got, want):
    want = np.asarray(want, np.float64)
    got = np.asarray(got, np.float64)
    return np.abs(got - want).max() / max(np.abs(want).max(), 1e-30)


def grad_close(got, want, rtol=RTOL):
    want = np.asarray(want, np.float64)
    got = np.asarray(got, np.float64)
    atol = max(1e-7, 1e-5 * float(np.abs(want).max()))
    return not (np.abs(got - want) > rtol * np.abs(want) + atol).any()


def check_against_oracle(out, ref, w_pg=1.0, w_ctc=1.0):
    if w_pg:
        assert np.array_equal(out["samples"].cpu().numpy(), ref["samples"])
        assert np.array_equal(out["hyp_len"].cpu().numpy(), ref["hyp_len"])
        assert np.array_equal(out["dist"].cpu().numpy(), ref["dist"])
        assert np.array_equal(out["rewards"].cpu().numpy().view(np.uint32), ref["rewards"].view(np.uint32))
    if w_ctc:                                            # (+inf where no alignment exists, on both sides)
        nll, want = out["nll"].cpu().numpy().astype(np.float64), ref["nll"]
        assert np.array_equal(np.isinf(nll), np.isinf(want))
        ok = np.isfinite(want)
        assert not ok.any() or np.abs(nll[ok] / want[ok] - 1).max() < RTOL
    if np.isfinite(ref["loss"]):
        assert abs(float(out["loss"]) - ref["loss"]) <= RTOL * abs(ref["loss"]) + 1e-5
    else:
        assert float(out["loss"]) == ref["loss"]
    dl = out["dlogits"].cpu().numpy()
    assert rel_err(dl, ref["dlogits"]) < RTOL
    assert grad_close(dl, ref["dlogits"])


WANT = ("rewards", "nll", "logp", "dist", "hyp_len", "samples")


def word_case(cuda, B, T, V, K, L, seed, ragged=False, regime="random", reward="wer", baseline="mean", w_pg=1.0,
              w_ctc=1.0, philox=False, blank=0, sep=1, style="text"):
    from pgasr_b200 import functional as F
    logits, targets, in_len, tgt_len, uni = make_word_batch(B, T, V, K, L, seed, regime, ragged, blank, sep, style)
    uni = None if philox else uni
    ref = word_ref.pg_ctc_step_words(logits, targets, in_len, tgt_len, uni, seed=77, K=K, blank=blank, sep=sep,
                                     reward=reward, baseline_mode=F.BASELINE_MODES[baseline], baseline_value=-0.5,
                                     w_pg=w_pg, w_ctc=w_ctc)
    out = F.pg_ctc_step(dev_t(logits, cuda), dev_t(targets, cuda), dev_t(in_len, cuda), dev_t(tgt_len, cuda), K=K,
                        blank=blank, reward=reward, baseline=baseline, baseline_value=-0.5, pg_weight=w_pg,
                        ctc_weight=w_ctc, uniforms=None if uni is None else dev_t(uni, cuda), seed=77, want=WANT,
                        space_id=sep)
    check_against_oracle(out, ref, w_pg, w_ctc)
    return out, ref


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,V,K,L,ragged,regime,reward", [
    (64, 500, 30, 16, 100, False, "random", "wer"),                 # the headline shape
    (64, 500, 30, 16, 100, False, "peaky", "wed"),
    (16, 500, 30, 16, 100, True, "peaky", "wer"),
    (7, 300, 30, 16, 60, True, "random", "wed"),
])
def test_word_step_matches_oracle(cuda, B, T, V, K, L, ragged, regime, reward):
    out, ref = word_case(cuda, B, T, V, K, L, seed=B + K, ragged=ragged, regime=regime, reward=reward)
    if regime == "peaky":
        assert (ref["dist"] < ref["n_w"][:, None]).any()           # words do match: the class lookup is exercised


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 5, 7, 33, 64])
def test_word_step_k(cuda, K):
    word_case(cuda, 3, 160, 30, K, 30, seed=K, ragged=True, regime="peaky")


@pytest.mark.gpu
@pytest.mark.parametrize("L", [63, 127, 255, 511])
def test_word_step_all_separator_transcripts(cuda, L):
    # n_w = L + 1 words: the bit vectors' last word is in use (W * 32 >= Lmax + 1)
    word_case(cuda, 2, 300, 30, 4, L, seed=L, regime="peaky", style="allsep", w_ctc=0.0)
    word_case(cuda, 2, 300, 30, 4, L, seed=L + 1, ragged=True, style="random", reward="wed", w_ctc=0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("V", [30, 32, 33, 64])
def test_word_step_alphabets(cuda, V):
    word_case(cuda, 4, 200, V, 8, 40, seed=V, ragged=True, regime="peaky")
    word_case(cuda, 4, 200, V, 8, 40, seed=V + 1, style="random", reward="wed", philox=True)


@pytest.mark.gpu
def test_word_step_nonzero_blank_modes_and_baselines(cuda):
    word_case(cuda, 4, 150, 30, 8, 30, seed=1, ragged=True, regime="peaky", blank=3, sep=0)
    word_case(cuda, 4, 150, 30, 8, 30, seed=2, blank=5, sep=7, philox=True, reward="wed")
    for i, bl in enumerate(("none", "mean", "loo", "value")):
        word_case(cuda, 5, 120, 30, 8, 24, seed=10 + i, ragged=True, regime="peaky", baseline=bl)
        word_case(cuda, 5, 120, 30, 8, 24, seed=20 + i, baseline=bl, philox=True, reward="wed")
    word_case(cuda, 4, 120, 30, 8, 24, seed=30, w_pg=1.0, w_ctc=0.0)
    word_case(cuda, 4, 120, 30, 8, 24, seed=31, w_pg=0.3, w_ctc=1.0, regime="peaky", baseline="loo")


@pytest.mark.gpu
def test_word_step_randomised(cuda):
    """150 randomised word-mode cases: shapes, alphabets, separators, blanks, regimes, modes, baselines."""
    rng = np.random.default_rng(2026)
    for i in range(150):
        V = int(rng.choice([3, 5, 30, 32, 33, 64]))
        blank = int(rng.integers(V))
        sep = int((blank + 1 + rng.integers(V - 1)) % V)
        B, K = int(rng.integers(1, 6)), int(rng.integers(1, 17))
        T = int(rng.integers(1, 160))
        L = int(rng.integers(1, 60))
        word_case(cuda, B, T, V, K, L, seed=1000 + i, ragged=bool(rng.integers(2)),
                  regime=str(rng.choice(["random", "peaky"])), reward=str(rng.choice(["wed", "wer"])),
                  baseline=str(rng.choice(["none", "mean", "loo", "value"])), philox=bool(rng.integers(2)),
                  blank=blank, sep=sep, style=str(rng.choice(["text", "random", "allsep"])),
                  w_ctc=float(rng.choice([0.0, 1.0])))


@pytest.mark.gpu
def test_word_step_queue_equals_single_steps(cuda):
    """StepQueue (pgasr_pg_ctc_step_multi_ws, steps on three streams, PG CTAs in pairs, odd B): bit for bit the
    single steps, and the oracle."""
    from pgasr_b200 import functional as F
    B, T, V, K, L = 5, 300, 30, 16, 60
    host = [make_word_batch(B, T, V, K, L, seed=50 + i, regime="peaky" if i % 2 else "random", ragged=True)
            for i in range(6)]
    batches = [dict(logits=dev_t(lg, cuda), targets=dev_t(tg, cuda), in_len=dev_t(il, cuda), tgt_len=dev_t(tl, cuda))
               for lg, tg, il, tl, _ in host]
    q = F.StepQueue(batches, K=K, reward="wer", baseline="loo", want=WANT, space_id=1)
    q.run(first=0, n=len(batches), seed=11)
    torch.cuda.synchronize()
    for i, (b, (lg, tg, il, tl, _)) in enumerate(zip(batches, host)):
        o = F.pg_ctc_step(b["logits"], b["targets"], b["in_len"], b["tgt_len"], K=K, reward="wer", baseline="loo",
                          seed=11 + i, want=WANT, space_id=1)
        for name in WANT + ("loss", "dlogits"):
            assert torch.equal(q.outputs[i][name].reshape(-1), o[name].reshape(-1)), (i, name)
        ref = word_ref.pg_ctc_step_words(lg, tg, il, tl, None, seed=11 + i, K=K, sep=1, reward="wer", baseline_mode=2)
        res = dict(q.outputs[i])
        res["loss"] = res["loss"][0]
        check_against_oracle(res, ref)


@pytest.mark.gpu
def test_word_step_chain_path(cuda):
    """K = 64, T = 1400: the samples do not fit an SM, the PG part chains the stand-alone kernels."""
    word_case(cuda, 2, 1400, 30, 64, 100, seed=3, regime="peaky", reward="wer")
    word_case(cuda, 2, 1400, 30, 64, 100, seed=4, ragged=True, reward="wed", baseline="none", philox=True)


@pytest.mark.gpu
def test_word_edit_distance_kernel(cuda):
    from pgasr_b200 import functional as F
    rng = np.random.default_rng(7)
    sep = 1

    def run(refs, ref_len, hyps, hyp_len, rows):
        d, nw = F.word_edit_distance(dev_t(hyps, cuda), dev_t(hyp_len, cuda), dev_t(refs, cuda), sep,
                                     ref_len=dev_t(ref_len, cuda), rows_per_ref=rows)
        d, nw = d.cpu().numpy(), nw.cpu().numpy()
        for r in range(hyps.shape[0]):
            g = r // rows
            want = word_ref.word_edit_distance(refs[g, :ref_len[g]], hyps[r, :hyp_len[r]], sep)
            assert (d[r], nw[g]) == want, (r, d[r], nw[g], want)

    # rows_per_ref > 1, hypotheses made of the transcript's words with edits
    G, rows, Lr, Th = 4, 6, 120, 200
    refs = np.zeros((G, Lr), np.int32)
    ref_len = rng.integers(0, Lr + 1, size=G).astype(np.int32)
    hyps = np.zeros((G * rows, Th), np.uint8)
    hyp_len = np.zeros(G * rows, np.int32)
    for g in range(G):
        refs[g] = text_targets(rng, 1, Lr, 12, 0, sep, [ref_len[g]], "text")[0]
        for k in range(rows):
            h = list(refs[g, :ref_len[g]])
            for _ in range(int(rng.integers(0, 6))):
                i = int(rng.integers(0, len(h) + 1))
                h.insert(i, int(rng.integers(1, 12)))
            h = h[:Th]
            hyps[g * rows + k, :len(h)] = h
            hyp_len[g * rows + k] = len(h)
    run(refs, ref_len, hyps, hyp_len, rows)
    # words longer than 32 ids
    w1, w2 = list(rng.integers(2, 5, size=40)), list(rng.integers(2, 5, size=70))
    ref = np.array(w1 + [sep] + w2 + [sep] + w1, np.int32)[None]
    hyp = np.zeros((3, 200), np.uint8)
    hl = np.zeros(3, np.int32)
    for r, h in enumerate([w1 + [sep] + w2, w2 + [sep] + w1 + [sep] + w1, w1[:-1] + [sep] + w2 + [sep] + w1]):
        hyp[r, :len(h)] = h
        hl[r] = len(h)
    run(ref, np.array([ref.shape[1]], np.int32), hyp, hl, 3)
    # 190 distinct transcript words at L = 511 (V = 64: 62 one-id words, then two-id words)
    letters = [c for c in range(64) if c not in (0, sep)]
    words = [[c] for c in letters] + [[a, b] for a in letters[:12] for b in letters[:11]][:128]
    ref = []
    for w in words:
        ref += w + [sep]
    ref = np.array(ref[:511], np.int32)
    n_distinct = len(set(tuple(w) for w in word_ref.split_ids(ref, sep)))
    assert n_distinct >= 190
    perm = [words[i] for i in rng.permutation(len(words))]
    hyp = np.zeros((4, 600), np.uint8)
    hl = np.zeros(4, np.int32)
    for r in range(4):
        h = []
        for w in perm[r * 20:r * 20 + 120]:
            h += w + [sep]
        hyp[r, :len(h)] = h
        hl[r] = len(h)
    run(ref[None], np.array([len(ref)], np.int32), hyp, hl, 4)


def forced_logits(paths, T, V, margin=40.0):
    lg = np.zeros((len(paths), T, V), np.float32)
    for b, p in enumerate(paths):
        for t in range(T):
            lg[b, t, p[t] if t < len(p) else 0] += margin
    return lg


@pytest.mark.gpu
def test_word_step_forced_paths(cuda):
    from pgasr_b200 import functional as F
    al = alphabet_of("ab cd")
    V, T, K = 8, 24, 4
    ab_cd, ab__cd = list(str_ids("ab cd", al)), list(str_ids("ab  cd", al))
    spread = lambda ids: sum(([c, 0] for c in ids), [])              # a blank after every id: repeats survive
    targets = np.zeros((2, 6), np.int32)
    targets[0, :5] = ab_cd
    targets[1, :5] = ab_cd
    tl = np.array([5, 5], np.int32)
    lg = forced_logits([spread(ab_cd), spread(ab__cd)], T, V)
    for reward, want_r in (("wed", [-0.0, -1.0]), ("wer", [-0.0, -0.5])):
        out = F.pg_ctc_step(dev_t(lg, cuda), dev_t(targets, cuda), None, dev_t(tl, cuda), K=K, reward=reward,
                            space_id=1, want=WANT)
        assert (out["dist"].cpu().numpy() == np.array([[0], [1]])).all()
        assert (out["hyp_len"].cpu().numpy() == np.array([[5], [6]])).all()
        r = out["rewards"].cpu().numpy()
        assert (r == np.array(want_r, np.float32)[:, None]).all(), r


@pytest.mark.gpu
def test_word_module_in_criterion_slot(cuda):
    """loss = criterion(model_out, t); loss.backward() with reward='wer': the gradient is the fused step's dlogits."""
    import pgasr_b200
    from pgasr_b200 import functional as F
    B, T, V, K, L = 4, 120, 30, 8, 24
    logits, targets, _, _, _ = make_word_batch(B, T, V, K, L, seed=5, regime="peaky")
    model_out = dev_t(logits, cuda).requires_grad_(True)
    crit = pgasr_b200.PolicyGradCTCLoss(K=K, reward="wer", space_id=1, pg_weight=0.5)
    loss = crit(model_out, dev_t(targets, cuda))
    loss.backward()
    tl = (targets != 0).astype(np.int32).cumprod(axis=1).sum(axis=1).astype(np.int32)
    ref = F.pg_ctc_step(dev_t(logits, cuda), dev_t(targets, cuda), None, dev_t(tl, cuda), K=K, reward="wer", space_id=1,
                        pg_weight=0.5, seed=0, want=("dist",))
    assert torch.equal(model_out.grad, ref["dlogits"])
    assert torch.equal(crit.last["dist"], ref["dist"])
    want = word_ref.pg_ctc_step_words(logits, targets, None, tl, None, seed=0, K=K, sep=1, reward="wer", w_pg=0.5)
    assert np.array_equal(crit.last["dist"].cpu().numpy(), want["dist"])
    assert rel_err(model_out.grad.cpu().numpy(), want["dlogits"]) < RTOL


@pytest.mark.gpu
def test_word_step_soak_bit_reproducible(cuda):
    from pgasr_b200 import functional as F
    lg, tg, il, tl, _ = make_word_batch(64, 500, 30, 16, 100, seed=9)
    lg, tg, il, tl = dev_t(lg, cuda), dev_t(tg, cuda), dev_t(il, cuda), dev_t(tl, cuda)
    first = F.pg_ctc_step(lg, tg, il, tl, K=16, reward="wer", space_id=1, seed=5, want=("rewards", "dist", "nll"))
    ws = first["workspace"]
    for _ in range(50):
        out = F.pg_ctc_step(lg, tg, il, tl, K=16, reward="wer", space_id=1, seed=5, workspace=ws,
                            want=("rewards", "dist", "nll"))
        for name in ("loss", "dlogits", "rewards", "dist", "nll"):
            assert torch.equal(out[name], first[name]), name
