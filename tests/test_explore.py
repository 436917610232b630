"""Sampling temperature and entropy bonus of the policy-gradient step (DESIGN.md "exploration spec").

CPU: argument checks (Python and the C entry point), routing of the default arguments, the oracle's self-checks.
GPU: the single-launch kernel (tile and streaming modes, word modes), the chain path and the multi-step queue against
tests/explore_ref.py, plus checks that do not rest on the oracle: fp64 autograd of the loss with the samples held
fixed, a chi-square test of the tempered sampler, and the default-equivalence of the exploration entry point.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import cport
from tests import explore_ref
from tests.synth import make_batch, make_word_batch

RTOL = 1e-4
REWARDS = ("ed", "cer", "ed_to_go", "wed", "wer")
BASELINES = ("none", "mean", "loo", "value")


# ---------------------------------------------------------------- CPU: validation and routing
def _ex_args(reward_mode=0, blank=0, V=30, w_pg=1.0):
    from pgasr_b200 import _native
    io = _native.StepIO()
    return io, (C.byref(io), 1, 0, 4, 50, V, 4, 10, blank, reward_mode, 1, 0.0, w_pg, 1.0)


def test_c_entry_rejects_bad_arguments_before_any_launch():
    from pgasr_b200 import _native
    L = _native.lib()
    ws, nbytes = C.c_void_p(1 << 20), 1 << 30                      # 256-byte aligned, never dereferenced
    ent = (C.c_void_p * 1)(1 << 21)
    n0 = L.pgasr_launch_count()
    _, head = _ex_args()
    for tau in (0.0, 0.0099, 100.5, -1.0, math.inf, math.nan):
        assert L.pgasr_pg_ctc_step_multi_ex(*head, None, -1, tau, 0.0, ws, nbytes, None) == -1, tau
    for beta in (-0.01, math.inf, math.nan):
        assert L.pgasr_pg_ctc_step_multi_ex(*head, None, -1, 1.5, beta, ws, nbytes, None) == -1, beta
    _, head0 = _ex_args(w_pg=0.0)
    assert L.pgasr_pg_ctc_step_multi_ex(*head0, None, -1, 1.0, 0.01, ws, nbytes, None) == -1   # bonus without PG
    assert L.pgasr_pg_ctc_step_multi_ex(*head0, ent, -1, 1.0, 0.0, ws, nbytes, None) == -1     # H_b without PG
    _, h3 = _ex_args(3)
    assert L.pgasr_pg_ctc_step_multi_ex(*h3, None, -1, 1.5, 0.0, ws, nbytes, None) == -1       # word mode, no separator
    assert L.pgasr_pg_ctc_step_multi_ex(*h3, None, 0, 1.5, 0.0, ws, nbytes, None) == -1        # separator == blank
    assert L.pgasr_pg_ctc_step_multi_ex(*h3, None, 30, 1.5, 0.0, ws, nbytes, None) == -1       # separator >= V
    _, h5 = _ex_args(5)
    assert L.pgasr_pg_ctc_step_multi_ex(*h5, None, 1, 1.5, 0.0, ws, nbytes, None) == -1        # no such reward mode
    assert L.pgasr_launch_count() == n0


EXPLORE_MSG = r"^(temperature must be|entropy_weight must be|the entropy bonus and the entropy output need)"


def test_python_argument_checks():
    import pgasr_b200
    from pgasr_b200 import functional as F
    for kw in (dict(temperature=0.001), dict(temperature=101.0), dict(temperature=float("nan")),
               dict(temperature=float("inf")), dict(entropy_weight=-1.0), dict(entropy_weight=float("nan")),
               dict(entropy_weight=float("inf")), dict(entropy_weight=0.1, pg_weight=0.0)):
        with pytest.raises(ValueError, match=EXPLORE_MSG):
            F.pg_ctc_step(None, None, **kw)
        with pytest.raises(ValueError, match=EXPLORE_MSG):
            pgasr_b200.PolicyGradCTCLoss(**kw)
        with pytest.raises(ValueError, match=EXPLORE_MSG):            # (a batch list StepQueue would accept)
            F.StepQueue([{"logits": None, "targets": None}], **kw)
    with pytest.raises(ValueError, match=EXPLORE_MSG):
        F.pg_ctc_step(None, None, pg_weight=0.0, want=("entropy",))
    with pytest.raises(ValueError, match=EXPLORE_MSG):
        F.StepQueue([{"logits": None, "targets": None}], pg_weight=0.0, want=("entropy",))
    with pytest.raises(ValueError):
        pgasr_b200.HostPipeline(2, 20, 30, 4, 5, temperature=1.5)
    with pytest.raises(ValueError):
        pgasr_b200.HostPipeline(2, 20, 30, 4, 5, entropy_weight=0.01)
    crit = pgasr_b200.PolicyGradCTCLoss(temperature=0.01, entropy_weight=0.0)
    assert crit.temperature == 0.01 and "entropy" in crit._want
    assert "entropy" not in pgasr_b200.PolicyGradCTCLoss()._want


def test_default_arguments_keep_their_entry_points():
    from pgasr_b200 import functional as F
    assert F._step_entry("ed", 0, None) == ("pgasr_pg_ctc_step_multi", ())
    assert F._step_entry("ed_to_go", 0, None, 1.0, 0.0, False) == ("pgasr_pg_ctc_step_multi", ())
    assert F._step_entry("wer", 0, 3, 1.0, 0.0, False) == ("pgasr_pg_ctc_step_multi_ws", (3,))
    assert F._step_entry("ed", 0, None, 1.5, 0.0) == ("pgasr_pg_ctc_step_multi_ex", (-1, 1.5, 0.0))
    assert F._step_entry("cer", 0, None, 1.0, 0.05) == ("pgasr_pg_ctc_step_multi_ex", (-1, 1.0, 0.05))
    assert F._step_entry("ed", 0, None, 1.0, 0.0, True) == ("pgasr_pg_ctc_step_multi_ex", (-1, 1.0, 0.0))
    assert F._step_entry("wed", 2, 5, 2.0, 0.0) == ("pgasr_pg_ctc_step_multi_ex", (5, 2.0, 0.0))


@pytest.mark.parametrize("reward_mode,baseline_mode", [(0, 1), (1, 2), (0, 0), (1, 3)])
def test_oracle_at_theta_one_is_the_step_oracle(reward_mode, baseline_mode):
    lg, tg, il, tl, uni = make_batch(4, 60, 12, 5, 10, seed=reward_mode + 3 * baseline_mode, ragged=True)
    loss, R, nll, dl = cport.pg_ctc_step(lg, tg, il, tl, uni, reward_mode=reward_mode, baseline_mode=baseline_mode,
                                         baseline_value=-0.5)
    ref = explore_ref.pg_ctc_step_explore(lg, tg, il, tl, uni, reward=("ed", "cer")[reward_mode],
                                          baseline_mode=baseline_mode, baseline_value=-0.5)
    assert np.array_equal(ref["rewards"], R)
    assert np.allclose(ref["nll"], nll, rtol=1e-12)
    assert abs(ref["loss"] - loss) <= 1e-6 * abs(loss)
    assert np.abs(ref["dlogits"] - dl).max() <= 1e-6 * np.abs(dl).max()


def test_oracle_entropy_gradient_matches_finite_difference():
    rng = np.random.default_rng(5)
    z = rng.standard_normal((2, 7, 6)) * 3.0
    in_len = np.array([7, 4], np.int32)
    H, dH = explore_ref.entropy_and_grad(z, in_len)
    eps = 1e-6
    for b, t, v in [(0, 0, 0), (0, 3, 5), (1, 2, 1), (1, 3, 4), (1, 5, 2)]:
        zp, zm = z.copy(), z.copy()
        zp[b, t, v] += eps
        zm[b, t, v] -= eps
        fd = (explore_ref.entropy_and_grad(zp, in_len)[0][b] - explore_ref.entropy_and_grad(zm, in_len)[0][b]) / (2 * eps)
        assert abs(fd - dH[b, t, v]) < 1e-7, (b, t, v)
    assert np.all(dH[1, 4:] == 0.0)
    assert abs(explore_ref.entropy_and_grad(np.zeros((1, 3, 5)))[0][0] - 3 * math.log(5)) < 1e-12


def test_oracle_entropy_of_masked_classes():
    """A class with a logit of -inf has p = 0: it contributes 0 to H and gets gradient 0 (0 log 0 = 0, never NaN)."""
    z = np.zeros((1, 2, 4))
    z[0, :, 3] = -np.inf
    with np.errstate(invalid="ignore"):
        H, dH = explore_ref.entropy_and_grad(z)
    assert abs(H[0] - 2 * math.log(3)) < 1e-12
    assert np.all(np.isfinite(dH)) and np.all(dH[0, :, 3] == 0.0)


# ---------------------------------------------------------------- GPU
def dev_t(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def rel_err(got, want):
    want = np.asarray(want, np.float64)
    got = np.asarray(got, np.float64)
    return np.abs(got - want).max() / max(np.abs(want).max(), 1e-30)


def check(out, ref, w_pg=1.0, w_ctc=1.0, entropy=True):
    if w_pg:
        for name in ("samples", "hyp_len", "dist"):
            assert np.array_equal(out[name].cpu().numpy(), ref[name]), name
        assert np.array_equal(out["rewards"].cpu().numpy().view(np.uint32), ref["rewards"].view(np.uint32))
        lp = out["logp"].cpu().numpy().astype(np.float64)
        assert np.abs(lp - ref["logp"]).max() <= RTOL * max(1.0, np.abs(ref["logp"]).max())
        if entropy and "entropy" in out:
            H = out["entropy"].cpu().numpy().astype(np.float64)
            assert np.abs(H - ref["entropy"]).max() <= RTOL * max(1.0, np.abs(ref["entropy"]).max())
    if w_ctc:
        nll, want = out["nll"].cpu().numpy().astype(np.float64), ref["nll"]
        assert np.array_equal(np.isinf(nll), np.isinf(want))
        ok = np.isfinite(want)
        assert not ok.any() or np.abs(nll[ok] / want[ok] - 1).max() < RTOL
    if np.isfinite(ref["loss"]):
        # relative to the terms, not their sum: PG and CTC terms of ~7 can cancel to a loss of ~0.1, and the fp32
        # log-probabilities (ulp 4e-6 at |z'| ~ 60) then move the sum by more than 1e-4 of itself
        assert abs(float(out["loss"]) - ref["loss"]) <= RTOL * max(abs(ref["loss"]), ref["loss_scale"]) + 1e-5
    else:
        assert float(out["loss"]) == ref["loss"]
    dl = out["dlogits"].cpu().numpy().astype(np.float64)
    want = ref["dlogits64"]
    assert rel_err(dl, want) < RTOL
    atol = max(1e-7, 1e-5 * float(np.abs(want).max()))
    assert not (np.abs(dl - want) > RTOL * np.abs(want) + atol).any()


WANT = ("rewards", "nll", "logp", "dist", "hyp_len", "samples", "entropy")


def explore_case(cuda, B, T, V, K, L, seed, tau=1.5, beta=0.05, reward="ed", baseline="mean", ragged=True,
                 regime="random", philox=False, blank=0, w_pg=1.0, w_ctc=1.0, sep=1, want=WANT):
    from pgasr_b200 import functional as F
    words = reward in ("wed", "wer")
    if words:
        lg, tg, il, tl, uni = make_word_batch(B, T, V, K, L, seed, regime, ragged, blank, sep)
    else:
        lg, tg, il, tl, uni = make_batch(B, T, V, K, L, seed=seed, regime=regime, ragged=ragged)
        if blank:
            tg = np.where(tg == blank, 0, tg).astype(np.int32)          # (blank never a label; 0 is then a letter)
            for b in range(B):
                tg[b, :tl[b]] = np.where(tg[b, :tl[b]] == 0, (blank + 1) % V, tg[b, :tl[b]])
    uni = None if philox else uni
    ref = explore_ref.pg_ctc_step_explore(lg, tg, il, tl, uni, seed=77, K=K, blank=blank, reward=reward,
                                          baseline_mode=F.BASELINE_MODES[baseline], baseline_value=-0.5, w_pg=w_pg,
                                          w_ctc=w_ctc, temperature=tau, w_ent=beta, sep=sep if words else None)
    out = F.pg_ctc_step(dev_t(lg, cuda), dev_t(tg, cuda), dev_t(il, cuda), dev_t(tl, cuda), K=K, blank=blank,
                        reward=reward, baseline=baseline, baseline_value=-0.5, pg_weight=w_pg, ctc_weight=w_ctc,
                        uniforms=None if uni is None else dev_t(uni, cuda), seed=77, want=want,
                        space_id=sep if words else None, temperature=tau, entropy_weight=beta)
    check(out, ref, w_pg, w_ctc)
    return out, ref


@pytest.mark.gpu
@pytest.mark.parametrize("reward", REWARDS)
@pytest.mark.parametrize("baseline", BASELINES)
def test_explore_modes_and_baselines(cuda, reward, baseline):
    i = REWARDS.index(reward) * 4 + BASELINES.index(baseline)
    tau = (0.5, 1.5, 4.0)[i % 3]
    explore_case(cuda, 5, 150, 30, 8, 30, seed=100 + i, tau=tau, beta=0.05, reward=reward, baseline=baseline,
                 regime="peaky" if i % 2 else "random", philox=bool(i % 3 == 1), w_ctc=float(i % 4 != 3))
    explore_case(cuda, 4, 120, 30, 8, 24, seed=200 + i, tau=tau, beta=0.0, reward=reward, baseline=baseline,
                 regime="random" if i % 2 else "peaky", philox=bool(i % 3 != 1))


@pytest.mark.gpu
@pytest.mark.parametrize("tau,beta,regime", [(1.5, 0.01, "random"), (0.5, 0.05, "peaky"), (4.0, 0.0, "peaky")])
def test_explore_headline_shape(cuda, tau, beta, regime):
    explore_case(cuda, 64, 500, 30, 16, 100, seed=7, tau=tau, beta=beta, ragged=False, regime=regime)
    explore_case(cuda, 64, 500, 30, 16, 100, seed=8, tau=tau, beta=beta, ragged=False, regime=regime, reward="wer")


@pytest.mark.gpu
@pytest.mark.parametrize("V", [30, 32, 33, 64])
def test_explore_alphabets(cuda, V):
    explore_case(cuda, 4, 200, V, 8, 40, seed=V, tau=1.5, regime="peaky")
    explore_case(cuda, 4, 200, V, 8, 40, seed=V + 1, tau=0.5, beta=0.0, baseline="loo", philox=True, reward="wed")


@pytest.mark.gpu
@pytest.mark.parametrize("L", [63, 127, 255, 511])
def test_explore_label_lengths(cuda, L):
    # one case per states-per-lane variant of the single-launch kernel
    explore_case(cuda, 2, max(300, 2 * L + 10), 30, 4, L, seed=L, tau=4.0, beta=0.05, baseline="none")


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 5, 33, 64])
def test_explore_sample_counts(cuda, K):
    explore_case(cuda, 3, 160, 30, K, 30, seed=K, tau=0.5, beta=0.05, regime="peaky")
    explore_case(cuda, 3, 160, 30, K, 30, seed=K + 1, tau=1.5, beta=0.05, reward="ed_to_go", philox=True)


@pytest.mark.gpu
def test_explore_nonzero_blank(cuda):
    explore_case(cuda, 4, 150, 30, 8, 30, seed=1, tau=1.5, beta=0.05, blank=3, regime="peaky")
    explore_case(cuda, 4, 150, 30, 8, 30, seed=2, tau=0.5, beta=0.05, blank=5, sep=7, reward="wer", philox=True)


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,V,K,L,reward,baseline", [(2, 1000, 30, 64, 120, "ed", "mean"), (2, 2000, 30, 16, 100, "cer", "loo"),
                                                        (3, 1300, 12, 8, 250, "ed", "none"), (2, 2000, 30, 4, 400, "ed", "mean")])
def test_explore_long_utterances_single_launch(cuda, B, T, V, K, L, reward, baseline):
    """The streaming PG role applies theta on read; still one launch."""
    from pgasr_b200 import _native
    n0 = _native.lib().pgasr_launch_count()
    explore_case(cuda, B, T, V, K, L, seed=T + K, tau=1.5, beta=0.05, reward=reward, baseline=baseline)
    assert _native.lib().pgasr_launch_count() - n0 == 1


@pytest.mark.gpu
@pytest.mark.parametrize("reward,baseline", [("ed", "mean"), ("cer", "loo"), ("wer", "mean"), ("wed", "none")])
def test_explore_chain_path(cuda, reward, baseline):
    """K = 64, T = 1400: the samples do not fit an SM, the PG part chains the stand-alone kernels."""
    from pgasr_b200 import _native
    n0 = _native.lib().pgasr_launch_count()
    explore_case(cuda, 2, 1400, 30, 64, 100, seed=3, tau=1.5, beta=0.05, reward=reward, baseline=baseline,
                 regime="peaky")
    assert _native.lib().pgasr_launch_count() - n0 > 1


@pytest.mark.gpu
@pytest.mark.parametrize("reward", ["ed", "wer"])
def test_explore_queue_equals_single_steps(cuda, reward):
    """StepQueue (steps on three streams, PG CTAs in pairs, odd B): bit for bit the single steps, and the oracle."""
    from pgasr_b200 import functional as F
    B, T, V, K, L = 5, 300, 30, 16, 60
    mk = make_word_batch if reward == "wer" else (lambda *a, **k: make_batch(*a[:5], seed=a[5], regime=a[6], ragged=True))
    host = [mk(B, T, V, K, L, 50 + i, "peaky" if i % 2 else "random", True) for i in range(6)]
    batches = [dict(logits=dev_t(lg, cuda), targets=dev_t(tg, cuda), in_len=dev_t(il, cuda), tgt_len=dev_t(tl, cuda))
               for lg, tg, il, tl, _ in host]
    sep = 1 if reward == "wer" else None
    for baseline, beta, want in (("mean", 0.05, WANT), ("loo", 0.05, WANT), ("mean", 0.0, NO_ENT),
                                 ("loo", 0.0, NO_ENT)):
        q = F.StepQueue(batches, K=K, reward=reward, baseline=baseline, want=want, space_id=sep, temperature=1.5,
                        entropy_weight=beta)
        q.run(first=0, n=len(batches), seed=11)
        torch.cuda.synchronize()
        for i, (b, (lg, tg, il, tl, _)) in enumerate(zip(batches, host)):
            o = F.pg_ctc_step(b["logits"], b["targets"], b["in_len"], b["tgt_len"], K=K, reward=reward,
                              baseline=baseline, seed=11 + i, want=want, space_id=sep, temperature=1.5,
                              entropy_weight=beta)
            for name in want + ("loss", "dlogits"):
                assert torch.equal(q.outputs[i][name].reshape(-1), o[name].reshape(-1)), (i, name)
            ref = explore_ref.pg_ctc_step_explore(lg, tg, il, tl, None, seed=11 + i, K=K, reward=reward,
                                                  baseline_mode=F.BASELINE_MODES[baseline], temperature=1.5,
                                                  w_ent=beta, sep=sep)
            res = dict(q.outputs[i])
            res["loss"] = res["loss"][0]
            check(res, ref)


NO_ENT = WANT[:-1]      # temperature alone: the variant runs without the entropy pass (no dense softmax under 'mean')


@pytest.mark.gpu
@pytest.mark.parametrize("reward", REWARDS)
@pytest.mark.parametrize("baseline", BASELINES)
def test_explore_temperature_only(cuda, reward, baseline):
    """beta = 0 and no entropy output: the theta-scaled tile and coefficients, dense rows from the scaled tile."""
    i = REWARDS.index(reward) * 4 + BASELINES.index(baseline)
    explore_case(cuda, 5, 150, 30, 8, 30, seed=500 + i, tau=(0.5, 1.5, 4.0)[i % 3], beta=0.0, reward=reward,
                 baseline=baseline, regime="peaky" if i % 2 else "random", philox=bool(i % 2), want=NO_ENT)


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,V,K,L,reward,baseline", [(2, 1000, 30, 64, 120, "ed", "loo"), (2, 2000, 30, 16, 100, "cer", "mean")])
def test_explore_temperature_only_streaming(cuda, B, T, V, K, L, reward, baseline):
    from pgasr_b200 import _native
    n0 = _native.lib().pgasr_launch_count()
    explore_case(cuda, B, T, V, K, L, seed=T + K + 1, tau=1.5, beta=0.0, reward=reward, baseline=baseline,
                 want=NO_ENT)
    assert _native.lib().pgasr_launch_count() - n0 == 1


@pytest.mark.gpu
def test_explore_masked_classes(cuda):
    """A class whose logit is -inf (a masked output unit): p' = 0, H gets 0 from it and its gradient is 0, no NaN,
    in the tile mode, the streaming mode and the chain path."""
    from pgasr_b200 import functional as F
    for B, T, K in ((4, 150, 8), (2, 1000, 64), (2, 1400, 64)):
        lg, tg, il, tl, uni = make_batch(B, T, 30, K, 30, seed=T, regime="peaky", ragged=True)
        lg[:, :, 29] = -np.inf
        tg = np.where(tg == 29, 1, tg).astype(np.int32)
        for baseline in ("mean", "loo"):
            out = F.pg_ctc_step(dev_t(lg, cuda), dev_t(tg, cuda), dev_t(il, cuda), dev_t(tl, cuda), K=K,
                                baseline=baseline, uniforms=dev_t(uni, cuda), want=WANT, temperature=1.5,
                                entropy_weight=0.05, ctc_weight=0.0)
            dl = out["dlogits"].cpu().numpy()
            assert np.all(np.isfinite(dl)) and np.all(dl[:, :, 29] == 0.0)
            assert np.isfinite(float(out["loss"]))
            with np.errstate(invalid="ignore"):
                H, _ = explore_ref.entropy_and_grad(explore_ref.tempered(lg, 1.5), il)
            assert np.abs(out["entropy"].cpu().numpy() - H).max() <= RTOL * np.abs(H).max()


@pytest.mark.gpu
def test_explore_randomised(cuda):
    """150 randomised cases: shapes, alphabets, blanks, regimes, modes, baselines, weights, temperatures, bonuses."""
    rng = np.random.default_rng(2027)
    for i in range(150):
        V = int(rng.choice([5, 12, 30, 32, 33, 64]))
        reward = str(rng.choice(REWARDS))
        blank = 0 if reward in ("wed", "wer") else int(rng.choice([0, 0, 1]))
        B, K = int(rng.integers(1, 6)), int(rng.integers(1, 17))
        T = int(rng.integers(8, 200))
        L = int(rng.integers(1, 50))
        explore_case(cuda, B, T, V, K, L, seed=3000 + i, tau=float(np.exp(rng.uniform(np.log(0.3), np.log(5.0)))),
                     beta=float(rng.choice([0.0, 0.01, 0.05, 0.3])), reward=reward,
                     baseline=str(rng.choice(BASELINES)), ragged=bool(rng.integers(2)),
                     regime=str(rng.choice(["random", "peaky"])), philox=bool(rng.integers(2)), blank=blank,
                     w_ctc=float(rng.choice([0.0, 1.0])), sep=1)


@pytest.mark.gpu
def test_explore_soak_bit_reproducible(cuda):
    from pgasr_b200 import functional as F
    lg, tg, il, tl, _ = make_batch(64, 500, 30, 16, 100, seed=9, regime="peaky")
    lg, tg, il, tl = dev_t(lg, cuda), dev_t(tg, cuda), dev_t(il, cuda), dev_t(tl, cuda)
    ref = F.pg_ctc_step(lg, tg, il, tl, K=16, seed=3, want=WANT, temperature=1.5, entropy_weight=0.01)
    ws, out = ref["workspace"], ref["workspace"].outputs(WANT)
    for _ in range(50):
        o = F.pg_ctc_step(lg, tg, il, tl, K=16, seed=3, workspace=ws, out=out, temperature=1.5, entropy_weight=0.01)
        for name in WANT + ("dlogits",):
            assert torch.equal(o[name], ref[name]), name
        assert torch.equal(o["loss"], ref["loss"])


@pytest.mark.gpu
@pytest.mark.parametrize("baseline", ["mean", "loo"])
def test_dlogits_equal_fp64_autograd_with_samples_fixed(cuda, baseline):
    """Independent of the oracle: with the kernel's own samples, rewards and advantages held fixed, dlogits is the fp64
    autograd gradient of w_pg L_pg(theta z) - beta / B sum_b H_b(theta z) + w_ctc mean_b ctc_loss(z)."""
    from pgasr_b200 import functional as F
    B, T, V, K, L, tau, beta, w_pg, w_ctc = 4, 120, 30, 8, 20, 1.7, 0.05, 0.8, 1.0
    lg, tg, il, tl, uni = make_batch(B, T, V, K, L, seed=12, regime="peaky", ragged=True)
    out = F.pg_ctc_step(dev_t(lg, cuda), dev_t(tg, cuda), dev_t(il, cuda), dev_t(tl, cuda), K=K, baseline=baseline,
                        uniforms=dev_t(uni, cuda), want=WANT, temperature=tau, entropy_weight=beta, pg_weight=w_pg,
                        ctc_weight=w_ctc)
    smp = out["samples"].cpu().long()
    R = out["rewards"].cpu().double()
    base = R.mean(1, keepdim=True) if baseline == "mean" else (R.sum(1, keepdim=True) - R) / (K - 1)
    A = R - base
    z = torch.from_numpy(lg).double().requires_grad_(True)
    theta = float(np.float32(1.0) / np.float32(tau))
    logq = torch.log_softmax(z * theta, dim=2)
    live = (torch.arange(T)[None, :] < torch.from_numpy(il).long()[:, None]).double()     # [B,T]
    lp = torch.gather(logq[:, None].expand(B, K, T, V), 3, smp[..., None])[..., 0]        # [B,K,T]
    logp = (lp * live[:, None]).sum(2)
    Lpg = -(A * logp).sum() / (B * K)
    H = -((logq.exp() * logq).sum(2) * live).sum(1)
    tgl = [torch.from_numpy(tg[b, :tl[b]]).long() for b in range(B)]
    ctc = torch.nn.functional.ctc_loss(torch.log_softmax(z, 2).transpose(0, 1), torch.cat(tgl),
                                       torch.from_numpy(il).long(), torch.from_numpy(tl).long(), blank=0,
                                       reduction="sum", zero_infinity=False) / B
    loss = w_pg * Lpg - beta / B * H.sum() + w_ctc * ctc
    loss.backward()
    dl = out["dlogits"].cpu().double()
    assert (dl - z.grad).abs().max().item() <= RTOL * z.grad.abs().max().item()
    assert abs(float(out["loss"]) - loss.item()) <= RTOL * abs(loss.item())
    assert torch.allclose(out["entropy"].cpu().double(), H.detach(), rtol=RTOL, atol=0)


@pytest.mark.gpu
def test_tempered_draws_follow_the_tempered_policy(cuda):
    """Chi-square: at tau = 2 the draws of a frame follow softmax(z / 2), and clearly not softmax(z)."""
    from scipy import stats
    from pgasr_b200 import functional as F
    V, T, K, B = 6, 64, 64, 64
    z = np.array([2.0, 1.0, 0.0, -0.5, 1.5, -2.0], np.float32)
    lg = np.broadcast_to(z, (B, T, V)).copy()
    tg = np.ones((B, 4), np.int32)
    out = F.pg_ctc_step(dev_t(lg, cuda), dev_t(tg, cuda), K=K, seed=123, want=("samples",), temperature=2.0,
                        ctc_weight=0.0)
    counts = np.bincount(out["samples"].cpu().numpy().ravel(), minlength=V).astype(np.float64)
    n = counts.sum()
    for zz, should_fit in ((z / 2.0, True), (z, False)):
        p = np.exp(zz - zz.max())
        p /= p.sum()
        chi2 = ((counts - n * p) ** 2 / (n * p)).sum()
        pval = stats.chi2.sf(chi2, V - 1)
        assert (pval > 1e-3) if should_fit else (pval < 1e-12), (should_fit, chi2, pval)


@pytest.mark.gpu
@pytest.mark.parametrize("reward,baseline", [("ed", "mean"), ("cer", "loo"), ("ed_to_go", "mean"), ("wer", "none")])
def test_exploration_entry_at_defaults_equals_default_path(cuda, reward, baseline):
    """tau = 1, beta = 0 with the entropy output requested: the exploration variant runs, and its draws and rewards are
    bit-identical to the default path; loss, dlogits and logp agree to 1e-6."""
    from pgasr_b200 import functional as F
    words = reward == "wer"
    mk = make_word_batch if words else make_batch
    lg, tg, il, tl, _ = mk(8, 300, 30, 16, 60, seed=4, regime="peaky", ragged=True)
    args = [dev_t(a, cuda) for a in (lg, tg, il, tl)]
    kw = dict(K=16, reward=reward, baseline=baseline, seed=9, space_id=1 if words else None)
    base = F.pg_ctc_step(*args, want=WANT[:-1], **kw)
    ex = F.pg_ctc_step(*args, want=WANT, **kw)
    for name in ("samples", "rewards", "dist", "hyp_len", "nll"):
        assert torch.equal(base[name], ex[name]), name
    for name in ("loss", "dlogits", "logp"):
        a, b = base[name].double(), ex[name].double()
        assert (a - b).abs().max().item() <= 1e-6 * max(1.0, a.abs().max().item()), name
    assert bool(torch.isfinite(ex["entropy"]).all()) and bool((ex["entropy"] > 0).all())


@pytest.mark.gpu
def test_explore_module_in_criterion_slot(cuda):
    import pgasr_b200
    from pgasr_b200 import functional as F
    lg, tg, il, tl, _ = make_batch(6, 200, 30, 8, 30, seed=21, regime="peaky", ragged=True)
    crit = pgasr_b200.PolicyGradCTCLoss(K=8, temperature=1.5, entropy_weight=0.02, seed=4)
    model_out = dev_t(lg, cuda).requires_grad_(True)
    t = dev_t(tg, cuda)
    loss = crit(model_out, t)
    loss.backward()
    assert crit.last["entropy"].shape == (6,) and bool((crit.last["entropy"] > 0).all())
    tl_dev = (t != 0).to(torch.int32).cumprod(dim=1).sum(dim=1, dtype=torch.int32)
    ref = F.pg_ctc_step(dev_t(lg, cuda), t, None, tl_dev, K=8, seed=4, temperature=1.5, entropy_weight=0.02,
                        want=("entropy",))
    assert torch.equal(model_out.grad, ref["dlogits"])
    assert torch.equal(crit.last["entropy"], ref["entropy"])
    assert float(loss) == float(ref["loss"])
