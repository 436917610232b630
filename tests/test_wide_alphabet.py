"""Alphabets of 65..256 classes: the wide sampler, the classic CTC kernel with 16 staged frames, the beam search with
four-word symbol masks, and the step's chain of stand-alone kernels above 64 classes.

CPU: a numpy restatement of the sampler spec's exp_spec (the reference the probs output is compared with bit for bit)
against the C oracle, and the size limits the C entry points report without a device.
GPU: every part against the C oracle (oracle/cport.py), tests/explore_ref.py, tests/word_ref.py and
oracle/pyref.prefix_beam_search, with the bars of test_gpu_parity.py.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import cport
from tests import placement
from tests.synth import make_batch, make_word_batch

RTOL = 1e-4
WANT = ("rewards", "nll", "logp", "dist", "hyp_len", "samples")


def dev_t(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def rel_err(got, want):
    want = np.asarray(want, np.float64)
    got = np.asarray(got, np.float64)
    return np.abs(got - want).max() / max(np.abs(want).max(), 1e-30)


def exp_spec_np(x0):
    """DESIGN.md "sampler spec" exp_spec, one fp32 operation per line (numpy rounds every float32 operation to
    nearest even and never fuses them)."""
    f = np.float32
    x0 = np.asarray(x0, np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        x = np.fmax(x0, f(-87.0))
        n = np.rint(x * f(1.44269504088896341))
        r = x - n * f(0.693359375)
        r = r - n * f(-2.12194440e-4)
        p = f(1.9875691500e-4)
        for c in (1.3981999507e-3, 8.3334519073e-3, 4.1665795894e-2, 1.6666665459e-1, 5.0000001201e-1):
            p = p * r + f(c)
        y = p * (r * r)
        y = y + r
        y = y + f(1.0)
        scale = np.ldexp(np.ones_like(y), n.astype(np.int32)).astype(np.float32)
        return (y * scale) * np.where(x0 >= f(-87.0), f(1.0), f(0.0))


def spec_probs(logits, in_len):
    """probs of the sampler spec: e_v * (1 / S), S the sequential fp32 sum in ascending v; zero after in_len."""
    z = np.asarray(logits, np.float32)
    with np.errstate(invalid="ignore"):
        e = exp_spec_np(z - z.max(-1, keepdims=True))
    S = np.cumsum(e, axis=-1, dtype=np.float32)[..., -1:]          # numpy's cumsum is sequential
    p = e * (np.float32(1.0) / S)
    for b in range(z.shape[0]):
        p[b, in_len[b]:] = 0
    return p


# ---------------------------------------------------------------- CPU
def test_exp_spec_restatement_matches_oracle():
    rng = np.random.default_rng(0)
    x = np.concatenate([-rng.random(4000).astype(np.float32) * 100, -rng.random(1000).astype(np.float32) * 2,
                        np.array([0.0, -87.0, -86.99999, -87.00001, -88.0, -np.inf], np.float32)])
    assert np.array_equal(exp_spec_np(x).view(np.uint32), cport.exp_spec(x).view(np.uint32))


def test_size_limits_without_a_device():
    """Workspace queries: non-zero up to 256 classes, zero above; the beam's candidate table caps the beam at 104 for
    256 classes (2188 beam + 2112 bytes of shared memory)."""
    from pgasr_b200 import _native
    L = _native.lib()
    for V in (65, 100, 256):
        assert L.pgasr_pg_ctc_step_workspace_bytes(8, 200, V, 16, 40) > 0
        assert L.pgasr_ctc_workspace_bytes(8, 200, V, 40) > 0
    assert L.pgasr_ctc_beam_search_workspace_bytes(4, 50, 256, 100) > 0
    assert L.pgasr_ctc_beam_search_workspace_bytes(4, 50, 256, 104) > 0
    assert L.pgasr_ctc_beam_search_workspace_bytes(4, 50, 256, 105) == 0
    assert L.pgasr_ctc_beam_search_workspace_bytes(4, 50, 128, 128) > 0
    assert L.pgasr_ctc_beam_search_workspace_bytes(4, 50, 257, 5) == 0
    # V <= 64: the sizes of the one-word kernel, unchanged
    assert L.pgasr_ctc_beam_search_workspace_bytes(4, 50, 64, 128) == L.pgasr_ctc_beam_search_workspace_bytes(4, 50, 30, 128)


def test_c_entry_points_refuse_257_classes_and_reward_to_go_before_any_launch():
    from pgasr_b200 import _native
    L = _native.lib()
    p = C.c_void_p(1 << 20)                                          # 256-byte aligned, never dereferenced
    n0 = L.pgasr_launch_count()
    assert L.pgasr_softmax_sample(p, None, None, 0, 2, 10, 257, 4, p, p, None, None) == -2
    assert L.pgasr_pg_ctc_step(p, p, None, None, None, 0, 2, 10, 257, 4, 3, 0, 0, 1, 0.0, 1.0, 1.0,
                               p, p, None, None, None, None, None, None, p, 1 << 30, None) == -2
    assert L.pgasr_ctc_beam_search(p, None, 2, 10, 257, 5, 0, p, p, p, p, 1 << 30, None) == -2
    assert L.pgasr_launch_count() == n0


# ---------------------------------------------------------------- GPU: sampler
@pytest.mark.gpu
@pytest.mark.parametrize("V", [65, 96, 127, 128, 129, 200, 255, 256])
def test_wide_sampler_bit_exact(cuda, V):
    from pgasr_b200 import functional as F
    for i, (K, T) in enumerate([(1, 37), (16, 300), (64, 1000)]):
        B = 3
        logits, _, in_len, _, uni = make_batch(B, T, V, K, 4, seed=V * 10 + i, ragged=True)
        s_ref, lp_ref = cport.softmax_sample(logits, in_len, uni)
        s, lp, probs = F.softmax_sample(dev_t(logits, cuda), dev_t(in_len, cuda), uniforms=dev_t(uni, cuda),
                                        return_probs=True)
        assert np.array_equal(s.cpu().numpy(), s_ref), (K, T)
        assert np.abs(lp.cpu().numpy() - lp_ref).max() <= RTOL * max(1.0, np.abs(lp_ref).max())
        p_ref = spec_probs(logits, in_len)
        p = probs.cpu().numpy()
        assert (np.abs(p - p_ref) <= 1e-6 * np.abs(p_ref)).all()
        # Philox draws
        s_ref, lp_ref = cport.softmax_sample(logits, in_len, None, seed=0x5EED + i, K=K)
        s2, lp2 = F.softmax_sample(dev_t(logits, cuda), dev_t(in_len, cuda), K=K, seed=0x5EED + i)
        assert np.array_equal(s2.cpu().numpy(), s_ref), (K, T)
        assert np.abs(lp2.cpu().numpy() - lp_ref).max() <= RTOL * max(1.0, np.abs(lp_ref).max())
        # run to run: bit identical
        s3, lp3 = F.softmax_sample(dev_t(logits, cuda), dev_t(in_len, cuda), K=K, seed=0x5EED + i)
        assert torch.equal(s3, s2) and torch.equal(lp3.view(torch.int32), lp2.view(torch.int32))


@pytest.mark.gpu
@pytest.mark.parametrize("V", [65, 256])
def test_wide_sampler_extreme_logits(cuda, V):
    from pgasr_b200 import functional as F
    rng = np.random.default_rng(V)
    T = 64
    logits = (rng.standard_normal((2, T, V)) * 40).astype(np.float32)      # exp underflow below -87
    logits[0, 0, :] = 0.0                                                   # all equal
    logits[0, 1, :] = -1e4
    logits[0, 1, V - 2] = 50.0                                              # one dominant class
    logits[0, 2, :] = -np.inf
    logits[0, 2, 3] = 1.0                                                   # -inf everywhere else
    logits[1, :, ::3] = -np.inf                                             # -inf classes
    uni = np.minimum(rng.random((2, 8, T), dtype=np.float32), np.float32(1 - 2**-24))
    uni[0, 0, :] = 0.0
    uni[0, 1, :] = np.float32(1 - 2**-24)
    s_ref, _ = cport.softmax_sample(logits, None, uni)
    s, _, probs = F.softmax_sample(dev_t(logits, cuda), uniforms=dev_t(uni, cuda), return_probs=True)
    s = s.cpu().numpy()
    assert np.array_equal(s, s_ref)
    assert (s[0, :, 1] == V - 2).all() and (s[0, :, 2] == 3).all()
    assert (s[1] % 3 != 0).all()
    p_ref = spec_probs(logits, np.full(2, T, np.int32))
    assert np.array_equal(probs.cpu().numpy(), p_ref)


@pytest.mark.gpu
def test_wide_sampler_philox_chi_square(cuda):
    """The Philox draws at 256 classes follow the softmax: chi-square over 8 frames x 4096 draws."""
    from scipy import stats
    from pgasr_b200 import functional as F
    V, T, K, B = 256, 8, 64, 64
    rng = np.random.default_rng(7)
    row = (rng.standard_normal((T, V)) * 1.5).astype(np.float32)
    logits = np.broadcast_to(row, (B, T, V)).copy()
    counts = np.zeros((T, V))
    s, _ = F.softmax_sample(dev_t(logits, cuda), K=K, seed=1234)
    s = s.cpu().numpy()                                                     # [B,K,T]
    for t in range(T):
        counts[t] = np.bincount(s[:, :, t].ravel(), minlength=V)
    p = torch.softmax(torch.tensor(row, dtype=torch.float64), -1).numpy()
    n = B * K
    pvals = []
    for t in range(T):
        exp = p[t] * n
        keep = exp >= 5                                                    # pool the rare classes into one bin
        obs = np.append(counts[t, keep], counts[t, ~keep].sum())
        ex = np.append(exp[keep], exp[~keep].sum())
        if ex[-1] == 0:
            obs, ex = obs[:-1], ex[:-1]
        pvals.append(stats.chisquare(obs, ex * obs.sum() / ex.sum()).pvalue)
    assert min(pvals) > 1e-4 and np.median(pvals) > 0.01


# ---------------------------------------------------------------- GPU: classic CTC kernel
@pytest.mark.gpu
@pytest.mark.parametrize("B,T,V,L", [(4, 40, 65, 9), (3, 400, 128, 60), (2, 1500, 196, 200), (3, 700, 197, 120),
                                     (2, 1500, 256, 200), (5, 123, 256, 20)])
def test_classic_ctc_wide(cuda, B, T, V, L):
    """ctc_loss_grad takes the classic kernel above 64 classes (16 staged frames above 196): accumulate into a non-zero
    buffer, and probabilities-only input."""
    from pgasr_b200 import functional as F
    logits, targets, in_len, tgt_len, _ = make_batch(B, T, V, 1, L, seed=T + V, ragged=True)
    targets[0, :min(4, int(tgt_len[0]))] = targets[0, 0]                   # repeats
    nll_ref, g_ref = cport.ctc_loss_grad(logits, targets, in_len, tgt_len)
    fin = np.isfinite(nll_ref)
    nll, g = F.ctc_loss_grad(dev_t(logits, cuda), dev_t(targets, cuda), dev_t(in_len, cuda), dev_t(tgt_len, cuda))
    nll, g = nll.cpu().numpy(), g.cpu().numpy()
    assert np.array_equal(np.isfinite(nll), fin) and np.abs(nll[fin] / nll_ref[fin] - 1).max() < RTOL
    assert rel_err(g, g_ref) < RTOL
    for b in range(B):
        assert (g[b, in_len[b]:] == 0).all()
    base = torch.full((B, T, V), 0.25, dtype=torch.float32, device=cuda)
    nll2, g2 = F.ctc_loss_grad(dev_t(logits, cuda), dev_t(targets, cuda), dev_t(in_len, cuda), dev_t(tgt_len, cuda),
                               grad_scale=0.5, out=base)
    assert g2.data_ptr() == base.data_ptr()
    g2 = (g2.cpu().numpy() - 0.25) / 0.5
    assert np.abs(nll2.cpu().numpy()[fin] / nll_ref[fin] - 1).max() < RTOL
    assert np.abs(g2 - g_ref).max() / np.abs(g_ref).max() < 2 * RTOL      # (the 0.25 offset costs a few fp32 ulps)
    # probabilities only (the C entry point with logits NULL): the same loss and gradient
    probs = torch.softmax(dev_t(logits, cuda), -1).contiguous()
    tg, il, tl = dev_t(targets, cuda), dev_t(in_len, cuda), dev_t(tgt_len, cuda)
    nll3 = torch.empty((B,), dtype=torch.float32, device=cuda)
    g3 = torch.empty((B, T, V), dtype=torch.float32, device=cuda)
    nbytes = F._native.lib().pgasr_ctc_workspace_bytes(B, T, V, L)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=cuda)
    F._launch(probs, "pgasr_ctc_loss_grad", None, probs.data_ptr(), tg.data_ptr(), il.data_ptr(), tl.data_ptr(), B, T, V,
              L, 0, 1.0, 0, nll3.data_ptr(), g3.data_ptr(), ws.data_ptr(), nbytes)
    assert np.abs(nll3.cpu().numpy()[fin] / nll_ref[fin] - 1).max() < RTOL
    assert rel_err(g3.cpu().numpy(), g_ref) < RTOL


@pytest.mark.gpu
def test_classic_ctc_wide_against_torch_cpu_double(cuda):
    from pgasr_b200 import functional as F
    B, T, V, L = 4, 120, 256, 25
    logits, targets, in_len, tgt_len, _ = make_batch(B, T, V, 1, L, seed=78, ragged=True)
    x = torch.tensor(logits, dtype=torch.float64, requires_grad=True)
    want = torch.nn.functional.ctc_loss(torch.log_softmax(x, -1).transpose(0, 1), torch.tensor(targets, dtype=torch.long),
                                        torch.tensor(in_len, dtype=torch.long), torch.tensor(tgt_len, dtype=torch.long),
                                        blank=0, reduction="none")
    want.sum().backward()
    nll, g = F.ctc_loss_grad(dev_t(logits, cuda), dev_t(targets, cuda), dev_t(in_len, cuda), dev_t(tgt_len, cuda))
    assert np.abs(nll.cpu().numpy() / want.detach().numpy() - 1).max() < RTOL
    assert rel_err(g.cpu().numpy(), x.grad.numpy()) < RTOL


# ---------------------------------------------------------------- GPU: the step
def _launches():
    from pgasr_b200 import _native
    return _native.lib().pgasr_launch_count()


@pytest.mark.gpu
@pytest.mark.parametrize("V", [65, 100, 256])
@pytest.mark.parametrize("reward,baseline", [("ed", "mean"), ("cer", "loo"), ("ed", "none"), ("cer", "value")])
def test_wide_step_char_rewards(cuda, V, reward, baseline):
    from tests.test_gpu_parity import step_case
    n0 = _launches()
    step_case(cuda, 6, 200, V, 8, 30, seed=V + len(reward + baseline), ragged=True, regime="random", reward=reward,
              baseline=baseline)
    assert _launches() - n0 == 7          # sampler, collapse, edit distance, advantages, CTC, PG gradient, loss


@pytest.mark.gpu
@pytest.mark.parametrize("V", [65, 100, 256])
def test_wide_step_weights_philox_and_long(cuda, V):
    from tests.test_gpu_parity import step_case
    step_case(cuda, 4, 150, V, 8, 20, seed=1, ragged=True, regime="peaky", w_pg=1.0, w_ctc=0.0)
    step_case(cuda, 4, 150, V, 8, 20, seed=2, ragged=True, regime="random", w_pg=0.0, w_ctc=1.0)
    step_case(cuda, 4, 150, V, 16, 20, seed=3, ragged=True, regime="random", philox=True)
    if V == 256:
        step_case(cuda, 2, 1000, V, 64, 100, seed=4, ragged=True, regime="random")


@pytest.mark.gpu
@pytest.mark.parametrize("V", [65, 256])
def test_wide_step_blank_last_class(cuda, V):
    from pgasr_b200 import functional as F
    blank = V - 1
    B, T, K, L = 4, 120, 8, 15
    logits, targets, in_len, tgt_len, uni = make_batch(B, T, V, K, L, seed=22, ragged=True)
    targets = np.where(targets == blank, 1, targets).astype(np.int32)
    for b in range(B):
        targets[b, tgt_len[b]:] = 0
    loss_ref, R_ref, nll_ref, dl_ref = cport.pg_ctc_step(logits, targets, in_len, tgt_len, uni, blank=blank)
    out = F.pg_ctc_step(dev_t(logits, cuda), dev_t(targets, cuda), dev_t(in_len, cuda), dev_t(tgt_len, cuda),
                        uniforms=dev_t(uni, cuda), blank=blank, want=("rewards", "nll"))
    assert np.array_equal(out["rewards"].cpu().numpy(), R_ref)
    assert np.abs(out["nll"].cpu().numpy() / nll_ref - 1).max() < RTOL
    assert abs(float(out["loss"]) - loss_ref) <= RTOL * abs(loss_ref) + 1e-5
    assert rel_err(out["dlogits"].cpu().numpy(), dl_ref) < RTOL


@pytest.mark.gpu
@pytest.mark.parametrize("V,sep,reward,baseline", [(65, 64, "wer", "mean"), (100, 70, "wed", "loo"),
                                                   (256, 200, "wer", "none"), (256, 255, "wed", "value")])
def test_wide_step_word_rewards(cuda, V, sep, reward, baseline):
    from tests.test_word_reward import word_case
    word_case(cuda, 5, 200, V, 8, 40, seed=V + sep, ragged=True, reward=reward, baseline=baseline, sep=sep)


@pytest.mark.gpu
@pytest.mark.parametrize("V,reward", [(65, "ed"), (100, "wer"), (256, "cer")])
def test_wide_step_temperature_and_entropy(cuda, V, reward):
    from tests.test_explore import explore_case
    out, ref = explore_case(cuda, 4, 160, V, 8, 25, seed=V, tau=1.5, beta=0.01, reward=reward,
                            sep=V - 3 if reward == "wer" else 1)
    assert "entropy" in out


@pytest.mark.gpu
def test_wide_step_at_unaligned_offsets(cuda):
    """logits and every output 1..3 floats into their buffers (4-byte aligned only)."""
    from pgasr_b200 import functional as F
    B, T, V, K, L = 3, 90, 129, 4, 12
    logits, targets, in_len, tgt_len, uni = make_batch(B, T, V, K, L, seed=5, ragged=True)
    _, R_ref, nll_ref, dl_ref = cport.pg_ctc_step(logits, targets, in_len, tgt_len, uni)
    key = (B, T, V, K, L)
    for off in (1, 2, 3):
        out = placement.offset_outputs(F, key, cuda, ("rewards", "nll"), off)
        lg = placement.at_offset(logits, off, cuda)
        res = F.pg_ctc_step(lg, dev_t(targets, cuda), dev_t(in_len, cuda), dev_t(tgt_len, cuda),
                            uniforms=placement.at_offset(uni, off, cuda), out=out)
        assert np.array_equal(res["rewards"].cpu().numpy(), R_ref)
        assert np.abs(res["nll"].cpu().numpy() / nll_ref - 1).max() < RTOL
        assert rel_err(res["dlogits"].cpu().numpy(), dl_ref) < RTOL


@pytest.mark.gpu
def test_wide_step_multi_equals_single_steps(cuda):
    """StepQueue at V = 128 (three overlapped lanes): every step bit for bit what a single call gives."""
    from pgasr_b200 import functional as F
    B, T, V, K, L = 8, 200, 128, 8, 30
    batches = []
    for i in range(5):
        lg, tg, il, tl, _ = make_batch(B, T, V, K, L, seed=40 + i, ragged=True)
        batches.append({"logits": dev_t(lg, cuda), "targets": dev_t(tg, cuda), "in_len": dev_t(il, cuda),
                        "tgt_len": dev_t(tl, cuda)})
    q = F.StepQueue(batches, K=K, reward="cer", baseline="loo", want=("rewards", "nll", "samples"))
    q.run(first=0, n=5, seed=100)
    torch.cuda.synchronize()
    for i, bt in enumerate(batches):
        one = F.pg_ctc_step(bt["logits"], bt["targets"], bt["in_len"], bt["tgt_len"], K=K, reward="cer",
                            baseline="loo", seed=100 + i, want=("rewards", "nll", "samples"))
        for name in ("dlogits", "rewards", "nll", "samples"):
            assert torch.equal(q.outputs[i][name], one[name]), (i, name)
        assert torch.equal(q.outputs[i]["loss"][0], one["loss"])


@pytest.mark.gpu
def test_wide_step_soak_bit_reproducible(cuda):
    from pgasr_b200 import functional as F
    B, T, V, K, L = 16, 300, 256, 16, 60
    lg, tg, il, tl, _ = make_batch(B, T, V, K, L, seed=12, ragged=True)
    lg, tg, il, tl = dev_t(lg, cuda), dev_t(tg, cuda), dev_t(il, cuda), dev_t(tl, cuda)
    first = F.pg_ctc_step(lg, tg, il, tl, K=K, seed=5, want=("nll", "rewards"))
    ws = first["workspace"]
    bad = torch.zeros((), dtype=torch.int64, device=cuda)
    for _ in range(50):
        out = F.pg_ctc_step(lg, tg, il, tl, K=K, seed=5, workspace=ws, want=("nll", "rewards"))
        bad += (out["dlogits"] != first["dlogits"]).sum() + (out["nll"] != first["nll"]).sum() + \
            (out["rewards"] != first["rewards"]).sum() + (out["loss"] != first["loss"]).sum()
    assert int(bad) == 0


@pytest.mark.gpu
def test_module_at_100_classes_trains_and_decodes(cuda):
    """PolicyGradCTCLoss(K=16, reward='cer') on a 100-class alphabet: autograd hands back the step's dlogits, and
    CTCDecoder decodes the posteriors."""
    import pgasr_b200
    from pgasr_b200 import functional as F
    B, T, V, K, L = 4, 120, 100, 16, 20
    lg, tg, il, tl, uni = make_batch(B, T, V, K, L, seed=3, ragged=True)
    x = dev_t(lg, cuda).requires_grad_(True)
    crit = pgasr_b200.PolicyGradCTCLoss(K=K, reward="cer")
    loss = crit(x, dev_t(tg, cuda), dev_t(il, cuda), dev_t(tl, cuda), uniforms=dev_t(uni, cuda))
    loss.backward()
    ref = F.pg_ctc_step(dev_t(lg, cuda), dev_t(tg, cuda), dev_t(il, cuda), dev_t(tl, cuda), K=K, reward="cer",
                        uniforms=dev_t(uni, cuda))
    assert torch.equal(x.grad, ref["dlogits"]) and float(loss) == float(ref["loss"])
    dec = pgasr_b200.CTCdecoder.CTCDecoder(alphabet=[str(i) for i in range(V)])
    p = torch.softmax(x.detach().double(), -1).cpu().numpy()
    outs = dec.decode_batch([p[b, :il[b]] for b in range(B)], beam_size=5)
    assert len(outs) == B and all(np.isfinite(nll) for _, nll in outs)
    assert outs[0] == dec.decode(p[0, :il[0]], beam_size=5)


# ---------------------------------------------------------------- GPU: refusals and unchanged launch counts
@pytest.mark.gpu
def test_wide_refusals(cuda):
    from pgasr_b200 import _native
    from pgasr_b200 import functional as F
    lg, tg, il, tl, _ = make_batch(2, 50, 65, 4, 8, seed=1)
    with pytest.raises(_native.PgasrError) as e:
        F.pg_ctc_step(dev_t(lg, cuda), dev_t(tg, cuda), dev_t(il, cuda), dev_t(tl, cuda), K=4, reward="ed_to_go")
    assert e.value.status == -2
    z = torch.zeros((2, 20, 257), device=cuda)
    with pytest.raises(_native.PgasrError) as e:
        F.softmax_sample(z, K=4)
    assert e.value.status == -2
    with pytest.raises(_native.PgasrError) as e:
        F.pg_ctc_step(z, torch.ones((2, 3), dtype=torch.int32, device=cuda), K=4)
    assert e.value.status == -2
    with pytest.raises(_native.PgasrError) as e:
        F.ctc_beam_search(torch.full((2, 20, 257), 1 / 257, dtype=torch.float64, device=cuda), beam_size=5)
    assert e.value.status == -2
    with pytest.raises(_native.PgasrError) as e:
        F.ctc_beam_search(torch.full((2, 20, 256), 1 / 256, dtype=torch.float64, device=cuda), beam_size=105)
    assert e.value.status == -2


@pytest.mark.gpu
@pytest.mark.parametrize("V", [30, 64])
def test_launch_counts_at_narrow_alphabets(cuda, V):
    """At most 64 classes every call launches what it launched before: one kernel each."""
    from pgasr_b200 import functional as F
    B, T, K, L = 8, 200, 8, 30
    lg, tg, il, tl, uni = make_batch(B, T, V, K, L, seed=9, ragged=True)
    lg, tg, il, tl = dev_t(lg, cuda), dev_t(tg, cuda), dev_t(il, cuda), dev_t(tl, cuda)
    for fn in (lambda: F.softmax_sample(lg, il, K=K),
               lambda: F.pg_ctc_step(lg, tg, il, tl, K=K),
               lambda: F.ctc_loss_grad(lg, tg, il, tl),
               lambda: F.ctc_beam_search(torch.softmax(lg.double(), -1), il, beam_size=5)):
        fn()
        n0 = _launches()
        fn()
        assert _launches() - n0 == 1


# ---------------------------------------------------------------- GPU: beam search
def _softmax_rows(z):
    p = np.exp(z - z.max(-1, keepdims=True))
    return p / p.sum(-1, keepdims=True)


@pytest.mark.gpu
@pytest.mark.parametrize("V,beam,peaky,blank", [(65, 1, False, 0), (65, 5, True, 0), (128, 5, False, 3),
                                                (128, 100, True, 0), (256, 5, True, 0), (256, 100, False, 0),
                                                (256, 1, False, 255)])
def test_wide_beam_search_matches_oracle(cuda, V, beam, peaky, blank):
    from oracle import pyref
    from pgasr_b200 import functional as F
    rng = np.random.default_rng(V * 10 + beam)
    N, T = 3, (12 if beam == 100 else 30)
    z = rng.normal(size=(N, T, V)) * (4.0 if peaky else 1.5)
    if peaky:
        z[:, :, blank] += 3.0
    p = _softmax_rows(z)
    p[0, ::5, (blank + 1) % V] = 0.0                              # exact zeros
    p[1, :, V - 2] = 0.0
    lens = np.array([T, T - 1, max(T // 2, 1)], np.int32)
    labels, label_len, nll = F.ctc_beam_search(dev_t(p, cuda), dev_t(lens, cuda), beam_size=beam, blank=blank)
    labels, label_len, nll = labels.cpu().numpy(), label_len.cpu().numpy(), nll.cpu().numpy()
    for n in range(N):
        with np.errstate(divide="ignore"):
            ref_labels, ref_nll = pyref.prefix_beam_search(p[n, :lens[n]], beam_size=beam, blank=blank)
        assert tuple(labels[n, :label_len[n]]) == tuple(ref_labels), n
        assert abs(nll[n] - ref_nll) <= 1e-9 * max(1.0, abs(ref_nll)), n
