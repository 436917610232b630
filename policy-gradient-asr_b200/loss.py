"""Drop-in for upstream loss.py, plus the loss the upstream project was heading towards.

customNLLLoss(ignore_index=None).forward(inp[L,B,V], target[B,L]) -- upstream loss.py:5-17: the sum over
decoder steps of the batch-mean NLL.  Upstream's `if self.ignore_index:` makes ignore_index=0 a no-op
(loss.py:9); that behaviour is kept.

PolicyGradCTCLoss fills the same criterion slot (model.py:14,206,235: `loss = criterion(model_out, t);
loss.backward()`) with the REINFORCE + CTC step: it samples K hypotheses per utterance from the per-frame
posteriors, collapses them, scores them by edit distance against the transcript, subtracts a baseline and
returns a scalar whose backward() hands the precomputed dlogits to autograd.
"""
import torch
import torch.nn as nn

from . import functional as F


class _NLLSumFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, inp, target, ignore_index):
        ctx.save_for_backward(target)
        ctx.shape = tuple(inp.shape)
        ctx.ignore_index = ignore_index
        return F.nll_sum_forward(inp, target, ignore_index)

    @staticmethod
    def backward(ctx, grad_out):
        (target,) = ctx.saved_tensors
        L, B, V = ctx.shape
        g = F.nll_sum_backward(target, grad_out.to(torch.float32), L, B, V, ctx.ignore_index)
        return g, None, None


class customNLLLoss(nn.Module):
    def __init__(self, ignore_index=None):
        super().__init__()
        self.ignore_index = ignore_index

    def forward(self, inp, target):
        ign = self.ignore_index if self.ignore_index else F.NO_IGNORE     # upstream loss.py:9: falsy -> not ignored
        return _NLLSumFn.apply(inp, target, int(ign))


class _PGCTCFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, module, targets, input_lengths, target_lengths, uniforms):
        out = F.pg_ctc_step(logits.detach(), targets, input_lengths, target_lengths, K=module.K,
                            blank=module.blank, reward=module.reward, baseline=module.baseline,
                            baseline_value=module.baseline_value, pg_weight=module.pg_weight,
                            ctc_weight=module.ctc_weight, uniforms=uniforms, seed=module._next_seed(),
                            space_id=module.space_id, temperature=module.temperature,
                            entropy_weight=module.entropy_weight, workspace=module._workspace, want=module._want)
        module._workspace = out["workspace"]
        module.last = {k: out[k] for k in module._want}
        ctx.save_for_backward(out["dlogits"])
        return out["loss"]

    @staticmethod
    def backward(ctx, grad_out):
        (dlogits,) = ctx.saved_tensors
        return dlogits * grad_out, None, None, None, None, None


class PolicyGradCTCLoss(nn.Module):
    """loss = pg_weight * L_pg + ctc_weight * mean_b nll_b - entropy_weight * mean_b H_b
    (DESIGN.md "policy gradient spec", "CTC spec", "exploration spec")

    forward(logits[B,T,V] fp32 CUDA, targets[B,L] (pad 0), input_lengths[B]=None, target_lengths[B]=None,
            uniforms[B,K,T]=None) -> 0-d tensor attached to `logits`.
    reward: 'ed' (-edit distance), 'cer' (-edit distance / len(transcript), as metrics.evaluate's CER) or
            'ed_to_go' (upstream policy_grad.reward's per-position rewards, credited per frame as reward-to-go;
            the baseline is then taken per frame over the K samples),
            'wed' (-word edit distance) or 'wer' (-word edit distance / words in the transcript, as metrics.evaluate's
            WER): words are split at space_id as str.split(" ") does (empty words kept), which is upstream's string
            split when every alphabet entry is one character
    space_id: id of the word separator (alphabet.index(" ")); required by 'wed' / 'wer', must differ from blank
    target_lengths=None: the lengths are taken from the padding -- the number of leading non-zero ids of each row
            (upstream pads transcripts with 0 = '<pad>', data.py:99, which is also the CTC blank and never a label)
    baseline: 'mean' (over the K samples of the utterance), 'loo', 'none', or 'value' (baseline_value)
    temperature: the PG term samples from and trains softmax(logits / temperature) (finite, 0.01..100); the CTC term
            keeps the untempered logits
    entropy_weight: weight of the entropy bonus (finite, >= 0; > 0 needs pg_weight != 0); H_b is the entropy of the
            tempered policy summed over the utterance's frames, in nats
    After a call, .last holds rewards [B,K], nll [B], logp [B,K], dist [B,K] (word edit distances for 'wed' / 'wer'),
    hyp_len [B,K], and entropy [B] (H_b) when temperature or entropy_weight is not the default.
    """

    def __init__(self, K=16, blank=0, reward="ed", baseline="mean", baseline_value=0.0, pg_weight=1.0,
                 ctc_weight=1.0, seed=0, space_id=None, temperature=1.0, entropy_weight=0.0):
        super().__init__()
        F.check_explore(temperature, entropy_weight, pg_weight)
        if reward not in F.REWARD_MODES or baseline not in F.BASELINE_MODES:
            raise ValueError("unknown reward or baseline mode")
        if reward in F.WORD_REWARDS:
            if space_id is None:
                raise ValueError(f"reward={reward!r} needs space_id, the id of the word separator (alphabet.index(' '))")
            if int(space_id) == int(blank):
                raise ValueError("space_id must differ from blank")
        self.space_id = None if space_id is None else int(space_id)
        self.K, self.blank, self.reward, self.baseline = int(K), int(blank), reward, baseline
        self.baseline_value, self.pg_weight, self.ctc_weight = float(baseline_value), float(pg_weight), float(ctc_weight)
        self.temperature, self.entropy_weight = float(temperature), float(entropy_weight)
        self._want = ("rewards", "nll", "logp", "dist", "hyp_len")
        if (self.temperature != 1.0 or self.entropy_weight != 0.0) and self.pg_weight != 0.0:
            self._want += ("entropy",)
        self.seed, self._calls = int(seed), 0
        self._workspace = None
        self.last = {}

    def _next_seed(self):
        # a fresh Philox stream per call: the call counter goes into the high half of the key
        s = (self.seed & 0xFFFFFFFF) | ((self._calls & 0xFFFFFFFF) << 32)
        self._calls += 1
        return s

    def forward(self, logits, targets, input_lengths=None, target_lengths=None, uniforms=None):
        # metrics.evaluate raises ZeroDivisionError on an empty reference.  Lengths that live on the host are checked
        # here; lengths already on the GPU are not (the check would cost a device synchronisation per step) -- an
        # empty transcript then yields reward -inf / nan for that utterance instead of an exception.
        if self.reward == "cer" and target_lengths is not None:
            tl = target_lengths if isinstance(target_lengths, torch.Tensor) else torch.as_tensor(target_lengths)
            if not tl.is_cuda and bool((tl == 0).any()):
                raise ZeroDivisionError("division by zero")
        if target_lengths is None:
            # the two-argument slot criterion(model_out, t): zero padding is not a label (it is the blank), so the
            # true length is the number of leading non-pad ids -- computed on the device, no synchronisation
            tg = targets if isinstance(targets, torch.Tensor) else torch.as_tensor(targets)
            tg = tg.to(logits.device)
            target_lengths = (tg != 0).to(torch.int32).cumprod(dim=1).sum(dim=1, dtype=torch.int32)
        return _PGCTCFn.apply(logits, self, targets, input_lengths, target_lengths, uniforms)
