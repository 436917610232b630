"""CPU: the oracle against the upstream-generated golden vectors and against independent references."""
import math

import numpy as np
import pytest
import torch

from oracle import cport, pyref
from tests.synth import make_batch


def enc(s):
    return [ord(c) for c in s]


def test_edit_dist_golden(golden):
    for e in golden["edit_dist"]:
        a, b = e["ref"], e["hyp"]
        if e["kind"] == "words":
            a, b = a.split(" "), b.split(" ")
        assert list(pyref.edit_dist(a, b)) == e["out"]
        if e["kind"] == "ids":
            assert cport.edit_distance(a, b) == e["out"][0]
        elif e["kind"] == "str":
            assert cport.edit_distance(enc(a), enc(b)) == e["out"][0]


def test_survey_known_answers():
    # SURVEY.md 8(c), produced by the upstream functions
    assert pyref.edit_dist("kitten", "sitting") == (3, 6)
    assert pyref.edit_dist("", "abc") == (3, 0)
    assert pyref.edit_dist("abc", "") == (3, 3)
    assert pyref.edit_dist("a b c".split(" "), "a x c d".split(" ")) == (2, 3)
    assert pyref.evaluate("the cat sat", "the bat sat on") == (0.36363636363636365, 0.6666666666666666)
    with pytest.raises(ZeroDivisionError):
        pyref.evaluate("", "abc")


def test_evaluate_and_collapse_golden(golden):
    for e in golden["evaluate"]:
        assert list(pyref.evaluate(e["ref"], e["hyp"])) == e["out"]
    for e in golden["collapse_fn"]:
        assert pyref.collapse_fn(e["in"]) == e["out"]
        assert "".join(map(chr, cport.collapse(enc(e["in"]), blank=-1))) == e["out"]
    for e in golden["collapse_paths"]:
        assert cport.collapse(e["path"], blank=-1).tolist() == e["collapsed"]
        assert cport.collapse(e["path"], blank=0).tolist() == e["collapsed_no_blank"]
        assert pyref.collapse_ids(e["path"], blank=0) == e["collapsed_no_blank"]
    # SURVEY 8(c): lengths 15 / 490, 11 / 476 after the blank drop
    assert [len(e["collapsed"]) for e in golden["collapse_paths"]] == [15, 490]
    assert [len(e["collapsed_no_blank"]) for e in golden["collapse_paths"]] == [11, 476]


def test_ctc_order_repeats_then_blanks():
    # a, blank, a -> a, a   (merge on the raw path first, then drop blanks)
    assert cport.collapse([1, 0, 1], blank=0).tolist() == [1, 1]
    assert cport.collapse([1, 1, 0, 0, 1, 2, 2], blank=0).tolist() == [1, 1, 2]
    assert cport.collapse([0, 0, 0], blank=0).tolist() == []


def test_reward_positions_golden(golden):
    for e in golden["reward_positions"]:
        y, h = e["true_y"], e["hyp"]
        r = cport.reward_positions(enc(y), enc(h), len(h) + 2)
        assert r[1:].tolist() == e["r"]
        assert [pyref.reward_from_hyp(y, h, t) for t in range(1, len(h) + 3)] == e["r"]
    # telescoping identity (SURVEY row a4): sum_t r_t = |y*| - ED(y*, yhat)
    y, h = "hello world", "helo wurld!"
    r = cport.reward_positions(enc(y), enc(h), len(h) - 1)
    assert r[1:].tolist() == [2, 1, 1, 1, 1, 0, 1, 1, 1, -1]
    assert int(r[1:].sum()) == len(y) - pyref.edit_dist(y, h)[0] == 8
    with pytest.raises(UnboundLocalError):
        pyref.reward_from_hyp(y, h, 0)


def test_nll_golden(golden):
    g = golden["nll"]
    inp = np.array(g["inp"], np.float32)
    tgt = np.array(g["target"], np.int64)
    for c in g["cases"]:
        ign = c["ignore_index"]
        assert abs(pyref.nll_sum(inp, tgt, ign) - c["out"]) < 1e-5
        val, grad = cport.nll_sum(inp, tgt, ign if ign else -1, want_grad=True)
        assert abs(val - c["out"]) < 1e-5
        t_inp = torch.tensor(inp, dtype=torch.float64, requires_grad=True)
        loss = sum(torch.nn.functional.nll_loss(t_inp[i], torch.tensor(tgt[:, i]),
                                                ignore_index=ign if ign else -100) for i in range(inp.shape[0]))
        loss.backward()
        np.testing.assert_allclose(grad, t_inp.grad.numpy(), atol=1e-12)
    # upstream quirk: ignore_index=0 is falsy and ignores nothing (loss.py:9)
    assert g["cases"][0]["out"] == g["cases"][1]["out"]


def test_beam_search_golden(golden):
    for e in golden["beam_search"]:
        labels, nll = pyref.prefix_beam_search(np.array(e["probs"]), beam_size=e["beam"])
        assert list(labels) == e["labels"]
        assert abs(nll - e["nll"]) < 1e-9


def test_philox_known_answers():
    # Random123 known-answer vectors for philox4x32-10
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, out in kat:
        assert tuple(int(x) for x in cport.philox4x32_10(ctr, key)) == out
    u = [cport.philox_uniform(0x5EED, 3, 7, k) for k in range(8)]
    assert all(0.0 <= x < 1.0 for x in u) and len(set(u)) == 8


def test_exp_spec_accuracy():
    x = -np.abs(np.random.default_rng(0).standard_normal(4000) * 12).astype(np.float32)
    got = cport.exp_spec(x).astype(np.float64)
    want = np.exp(x.astype(np.float64))
    rel = np.abs(got - want) / want
    assert rel.max() < 4e-7
    assert cport.exp_spec(np.float32([0.0]))[0] == 1.0
    assert cport.exp_spec(np.float32([-88.0]))[0] == 0.0


def test_sampler_matches_numpy_restatement():
    # the C sampler against a numpy float32 restatement of the same written spec
    logits, _, in_len, _, uni = make_batch(3, 17, 30, 4, 5, seed=5, ragged=True)
    samples, logp = cport.softmax_sample(logits, in_len, uni)
    f = np.float32
    for b in range(3):
        for t in range(int(in_len[b])):
            z = logits[b, t]
            e = cport.exp_spec(z - z.max())
            c = np.zeros(30, f)
            acc = f(0)
            for v in range(30):
                acc = f(acc + e[v])
                c[v] = acc
            for k in range(4):
                tau = f(uni[b, k, t] * acc)
                assert samples[b, k, t] == min(int((c <= tau).sum()), 29)
        assert (samples[b, :, int(in_len[b]):] == 0).all()
    lsm = torch.log_softmax(torch.tensor(logits, dtype=torch.float64), -1).numpy()
    for b in range(3):
        for k in range(4):
            want = sum(lsm[b, t, samples[b, k, t]] for t in range(int(in_len[b])))
            assert abs(logp[b, k] - want) < 1e-9


def test_sampler_statistics():
    # frequencies follow softmax (chi-square-ish bound), Philox mode
    rng = np.random.default_rng(1)
    z = (rng.standard_normal((1, 1, 8)) * 1.5).astype(np.float32)
    logits = np.repeat(z, 4000, axis=1)                     # one distribution, 4000 frames
    samples, _ = cport.softmax_sample(logits, None, None, seed=123, K=16)
    p = np.exp(z[0, 0] - z[0, 0].max())
    p /= p.sum()
    freq = np.bincount(samples.ravel(), minlength=8) / samples.size
    assert np.abs(freq - p).max() < 4 * np.sqrt(p.max() / samples.size) + 1e-3


@pytest.mark.parametrize("ragged", [False, True])
def test_ctc_oracle_vs_torch(ragged):
    B, T, V, L = 4, 40, 7, 9
    logits, targets, in_len, tgt_len, _ = make_batch(B, T, V, 2, L, seed=2, ragged=ragged)
    targets[0, :3] = [2, 2, 3]                               # a repeated label
    nll, grad = cport.ctc_loss_grad(logits, targets, in_len, tgt_len)
    x = torch.tensor(logits, dtype=torch.float64, requires_grad=True)
    lp = torch.log_softmax(x, -1).transpose(0, 1)
    want = torch.nn.functional.ctc_loss(lp, torch.tensor(targets, dtype=torch.long), torch.tensor(in_len, dtype=torch.long),
                                        torch.tensor(tgt_len, dtype=torch.long), blank=0, reduction="none")
    want.sum().backward()
    np.testing.assert_allclose(nll, want.detach().numpy(), rtol=1e-10)
    np.testing.assert_allclose(grad, x.grad.numpy(), atol=1e-10)


def test_ctc_oracle_infeasible():
    logits, targets, in_len, tgt_len, _ = make_batch(2, 6, 5, 2, 5, seed=3)
    targets[0] = [1, 1, 1, 1, 1]                             # needs 9 frames, has 6
    targets[1] = [1, 2, 3, 4, 1]
    nll, grad = cport.ctc_loss_grad(logits, targets, in_len, tgt_len)
    assert math.isinf(nll[0]) and np.all(grad[0] == 0)
    assert np.isfinite(nll[1])


@pytest.mark.parametrize("baseline,bmode", [("mean", 1), ("loo", 2), ("none", 0), ("value", 3)])
def test_pg_oracle_vs_autograd(baseline, bmode):
    B, T, V, K, L = 3, 12, 6, 5, 4
    logits, targets, in_len, tgt_len, uni = make_batch(B, T, V, K, L, seed=4, ragged=True)
    samples, logp = cport.softmax_sample(logits, in_len, uni)
    _, _, dist = cport.collapse_score(samples, targets, in_len, tgt_len)
    loss, R, A, grad = cport.pg_loss_grad(logits, samples, logp, dist, in_len, tgt_len, L, reward_mode=1,
                                          baseline_mode=bmode, baseline_value=-0.7)
    x = torch.tensor(logits, dtype=torch.float64, requires_grad=True)
    lsm = torch.log_softmax(x, -1)
    total = 0.0
    for b in range(B):
        for k in range(K):
            idx = torch.tensor(samples[b, k, :in_len[b]].astype(np.int64))
            lpk = lsm[b, torch.arange(int(in_len[b])), idx].sum()
            assert abs(float(lpk) - logp[b, k]) < 1e-9
            total = total - float(A[b, k]) * lpk
    total = total / (B * K)
    total.backward()
    assert abs(float(total) - loss) < 1e-10
    np.testing.assert_allclose(grad, x.grad.numpy(), atol=1e-12)
    want_R = -dist / tgt_len[:, None].astype(np.float32)
    np.testing.assert_array_equal(R, want_R.astype(np.float32))


def test_step_composition():
    B, T, V, K, L = 2, 20, 6, 4, 5
    logits, targets, in_len, tgt_len, uni = make_batch(B, T, V, K, L, seed=6)
    loss, R, nll, dl = cport.pg_ctc_step(logits, targets, in_len, tgt_len, uni, w_pg=0.5, w_ctc=2.0)
    samples, logp = cport.softmax_sample(logits, in_len, uni)
    _, _, dist = cport.collapse_score(samples, targets, in_len, tgt_len)
    lpg, R2, _, gpg = cport.pg_loss_grad(logits, samples, logp, dist, in_len, tgt_len, L)
    nll2, gctc = cport.ctc_loss_grad(logits, targets, in_len, tgt_len)
    assert abs(loss - (0.5 * lpg + 2.0 * nll2.mean())) < 1e-9
    np.testing.assert_allclose(dl, 0.5 * gpg + 2.0 / B * gctc, atol=1e-6)
    np.testing.assert_array_equal(R, R2)


# ---------------------------------------------------------------- 8f.1 reward-to-go (DESIGN.md "reward-to-go spec")
def test_togo_r_pos_is_upstream_reward_golden(golden):
    """r_pos of the oracle IS upstream's policy_grad.reward sequence: r_t (t >= 2) equals r_pos[t], upstream's t == 1
    branch equals r_pos[0] + r_pos[1] (policy_grad.py:14-15 subtracts len(y*) = c[0])."""
    for e in golden["reward_positions"]:
        y, h = enc(e["true_y"]), enc(e["hyp"])
        if not h:
            continue
        V = 128
        # a path that collapses to exactly `h`: every symbol once, a blank between equal neighbours
        path = []
        for i, c in enumerate(h):
            if i and h[i - 1] == c:
                path.append(0)
            path.append(c)
        T = len(path) + 2
        samples = np.zeros((1, 1, T), np.uint8)
        samples[0, 0, :len(path)] = path
        logits = np.zeros((1, T, V), np.float32)
        tg = np.array([y], np.int32)
        loss, R, to_go, r_pos, _ = cport.pg_togo_loss_grad(logits, samples, tg, np.array([len(path)], np.int32),
                                                           np.array([len(y)], np.int32), baseline_mode=0)
        rp = r_pos[0, 0, :len(h)].tolist()
        up = e["r"]                                            # upstream r_1, r_2, ...
        assert rp[0] + (rp[1] if len(h) > 1 else 0) == up[0]
        assert rp[2:] == up[1:len(h) - 1]
        assert int(R[0, 0]) == len(y) - cport.edit_distance(y, h) == sum(rp)
        assert int(to_go[0, 0, 0]) == sum(rp) and (to_go[0, 0, len(path):] == 0).all()


@pytest.mark.parametrize("baseline_mode", [0, 1, 2, 3])
def test_togo_oracle_against_autograd(baseline_mode):
    """Credit assignment and gradient of the oracle against an independent numpy restatement + fp64 torch autograd."""
    B, T, V, K, L = 3, 40, 7, 5, 6
    logits, targets, in_len, tgt_len, uni = make_batch(B, T, V, K, L, seed=11 + baseline_mode, ragged=True)
    samples, _ = cport.softmax_sample(logits, in_len, uni)
    loss, R, to_go, r_pos, grad = cport.pg_togo_loss_grad(logits, samples, targets, in_len, tgt_len,
                                                          baseline_mode=baseline_mode, baseline_value=-0.75)
    # independent restatement: collapse with emission frames, last column by the pure-Python edit distance
    G = np.zeros((B, K, T))
    for b in range(B):
        ref = targets[b, :tgt_len[b]].tolist()
        for k in range(K):
            path = samples[b, k, :in_len[b]].tolist()
            emit = [t for t, c in enumerate(path) if c != 0 and (t == 0 or path[t - 1] != c)]
            hyp = [path[t] for t in emit]
            col = [pyref.edit_dist(ref, hyp[:i])[0] for i in range(len(hyp) + 1)]
            r = [-(col[i + 1] - col[i]) for i in range(len(hyp))]
            assert r_pos[b, k, :len(hyp)].tolist() == r and not r_pos[b, k, len(hyp):].any()
            for t in range(in_len[b]):
                G[b, k, t] = sum(r[i] for i, e in enumerate(emit) if e >= t)
            assert R[b, k] == len(ref) - col[-1]
    assert np.array_equal(to_go, G.astype(np.int16))
    z = torch.tensor(logits, dtype=torch.float64, requires_grad=True)
    lp = torch.log_softmax(z, -1)
    Gt = torch.tensor(G)
    if baseline_mode == 1:
        base = Gt.mean(1, keepdim=True)
    elif baseline_mode == 2:
        base = (Gt.sum(1, keepdim=True) - Gt) / (K - 1)
    elif baseline_mode == 3:
        base = torch.full_like(Gt, -0.75)
    else:
        base = torch.zeros_like(Gt)
    A = Gt - base
    tot = 0.0
    for b in range(B):
        for k in range(K):
            idx = torch.tensor(samples[b, k, :in_len[b]].astype(np.int64))
            tot = tot - (A[b, k, :in_len[b]] * lp[b, torch.arange(in_len[b]), idx]).sum()
    tot = tot / (B * K)
    tot.backward()
    assert abs(float(tot) - loss) <= 1e-12 * max(1.0, abs(loss))
    np.testing.assert_allclose(grad, z.grad.numpy(), atol=1e-13)
    # the whole-step entry with reward_mode 2 chains the same function
    l2, R2, nll, dl = cport.pg_ctc_step(logits, targets, in_len, tgt_len, uni, reward_mode=2, baseline_mode=baseline_mode,
                                        baseline_value=-0.75, w_pg=1.0, w_ctc=0.0)
    assert np.array_equal(R2, R) and np.allclose(dl, grad, atol=1e-7)


def test_reference_cpu_leg_runs_on_upstream_code():
    """oracle/refpath.py (the `kind: reference` CPU leg of bench.py) runs upstream's collapse_fn / edit_dist and agrees
    with the oracle on the CTC part (the sampled part differs by construction: torch RNG).  Upstream's source is not
    part of this repository: with no copy in oracle/_ref the leg runs oracle/pyref's restatements of the two
    functions, which the golden vectors (upstream's own outputs) pin in test_edit_dist_golden and
    test_evaluate_and_collapse_golden."""
    from oracle import make_ref, refpath
    make_ref.make()
    upstream = None if refpath.available() else (pyref.edit_dist, pyref.collapse_fn)
    B, T, V, K, L = 2, 30, 6, 3, 4
    logits, targets, in_len, tgt_len, _ = make_batch(B, T, V, K, L, seed=5, ragged=True)
    loss, R, g = refpath.step(logits, targets, in_len, tgt_len, K, w_pg=0.0, w_ctc=1.0, upstream=upstream)
    nll, gref = cport.ctc_loss_grad(logits, targets, in_len, tgt_len)
    assert abs(loss - nll.mean()) < 1e-4 * abs(nll.mean())
    assert np.abs(g - gref / B).max() < 1e-5
    loss, R, g = refpath.step(logits, targets, in_len, tgt_len, K, w_pg=1.0, w_ctc=0.0, upstream=upstream)
    assert R.shape == (B, K) and (R <= 0).all() and np.isfinite(g).all()
