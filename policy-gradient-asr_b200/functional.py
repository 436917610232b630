"""Batched tensor-level operators of the PG-loss + CTC hot path (SURVEY.md 8a rows a1-a8).

Each function takes CUDA tensors, launches the sm_100a kernels of libpgasr_b200.so on torch's current
stream through the C ABI (include/pgasr.h) and returns CUDA tensors.  torch is used for device memory
and streams only.  There is no CPU path: a CPU tensor is a TypeError, a missing library a RuntimeError.
"""
import ctypes as C
import math

import torch

from . import _native

REWARD_MODES = {"ed": 0, "cer": 1, "ed_to_go": 2, "wed": 3, "wer": 4}
WORD_REWARDS = ("wed", "wer")      # word-level: need the separator id (space_id), pgasr_pg_ctc_step_multi_ws
NO_IGNORE = -2**31                  # PGASR_NO_IGNORE
OPTIONAL_OUTPUTS = ("rewards", "logp", "hyp_len", "dist", "nll", "samples", "to_go", "r_pos")
EXPLORE_OUTPUTS = ("entropy",)      # H_b [B]: pgasr_pg_ctc_step_multi_ex only (not a field of pgasr_step_io)
BASELINE_MODES = {"none": 0, "mean": 1, "loo": 2, "value": 3}


def _ptr(t):
    return None if t is None else t.data_ptr()


def _launch(ref, fn_name, *args):
    """Call a stream-taking entry point on the device of tensor `ref`: the device is made current for the call (kernel
    attributes and launches go to the current device) and the work is enqueued on THAT device's current stream."""
    dev = ref.device
    with torch.cuda.device(dev):
        _native.call(fn_name, *args, torch.cuda.current_stream(dev).cuda_stream)


def _need(t, dtype, name, ndim=None):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise TypeError(f"{name} must be a CUDA tensor (pgasr_b200 has no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if ndim is not None and t.dim() != ndim:
        raise ValueError(f"{name} must have {ndim} dims, got {tuple(t.shape)}")
    return t.contiguous()


def _opt_i32(t, name, n, device):
    if t is None:
        return None
    if not (isinstance(t, torch.Tensor) and t.dtype == torch.int32 and t.device == device and t.is_contiguous()):
        if not isinstance(t, torch.Tensor):
            t = torch.as_tensor(t)
        t = t.to(device=device, dtype=torch.int32).contiguous()
    if t.numel() != n:
        raise ValueError(f"{name} must have {n} entries, got {t.numel()}")
    return t


def as_targets(targets, device):
    """[B,Lmax] label ids, padded with 0 (upstream data.py:99) -> int32 on `device`."""
    if not isinstance(targets, torch.Tensor):
        targets = torch.as_tensor(targets)
    if targets.dim() != 2:
        raise ValueError("targets must be [B, Lmax]")
    if targets.dtype == torch.int32 and targets.device == device and targets.is_contiguous():
        return targets
    return targets.to(device=device, dtype=torch.int32).contiguous()


def softmax_sample(logits, input_lengths=None, K=16, uniforms=None, seed=0, return_probs=False):
    """Row a6.  logits [B,T,V] fp32 -> samples [B,K,T] uint8, logp [B,K] fp32 (and probs [B,T,V]).
    V <= 256 classes, K <= 64 draws."""
    logits = _need(logits, torch.float32, "logits", 3)
    B, T, V = logits.shape
    if uniforms is not None:
        uniforms = _need(uniforms, torch.float32, "uniforms", 3)
        if uniforms.shape[0] != B or uniforms.shape[2] != T:
            raise ValueError("uniforms must be [B,K,T]")
        K = uniforms.shape[1]
    in_len = _opt_i32(input_lengths, "input_lengths", B, logits.device)
    samples = torch.empty((B, K, T), dtype=torch.uint8, device=logits.device)
    logp = torch.empty((B, K), dtype=torch.float32, device=logits.device)
    probs = torch.empty_like(logits) if return_probs else None
    _launch(logits, "pgasr_softmax_sample", _ptr(logits), _ptr(in_len), _ptr(uniforms), int(seed) & (2**64 - 1),
                 B, T, V, K, _ptr(samples), _ptr(logp), _ptr(probs))
    return (samples, logp, probs) if return_probs else (samples, logp)


def collapse(seqs, lengths=None, rows_per_len=None, blank=0):
    """Row a3.  seqs [N,T] (or [B,K,T]) uint8 -> (collapsed rows, lengths); `lengths` has one entry per row or
    one per group of rows_per_len consecutive rows (e.g. [B] for [B,K,T]).  blank=None: merge repeats only
    (exactly upstream collapse_fn, CTCdecoder.py:119-131); blank=0: then drop blanks."""
    seqs = _need(seqs, torch.uint8, "seqs")
    shape = seqs.shape
    T = shape[-1]
    flat = seqs.reshape(-1, T)
    N = flat.shape[0]
    if rows_per_len is None:          # infer: one length per row, or one per group of K rows ([B,K,T] with [B] lengths)
        n_given = N if lengths is None else int(torch.as_tensor(lengths).numel())
        if n_given == 0 or N % n_given:
            raise ValueError("lengths must have one entry per row or per equal group of rows")
        rows_per_len = N // n_given
    n_len = (N + rows_per_len - 1) // rows_per_len
    lengths = _opt_i32(lengths, "lengths", n_len, seqs.device)
    out = torch.empty_like(flat)
    out_len = torch.empty((N,), dtype=torch.int32, device=seqs.device)
    _launch(seqs, "pgasr_collapse_u8", _ptr(flat), _ptr(lengths), rows_per_len, N, T,
                 -1 if blank is None else int(blank), _ptr(out), _ptr(out_len))
    return out.reshape(shape), out_len.reshape(shape[:-1])


def edit_distance(hyps, hyp_len, refs, ref_len=None, rows_per_ref=None, vocab=256, last_col=False):
    """Rows a1/a4.  hyps [N,Th] (or [B,K,Th]) uint8, hyp_len [N], refs [G,Lr] int32 with N = G*rows_per_ref
    -> dist [N] int32 (and last_col [N,Th+1]: ED(ref, hyp[:i])).  Bit-parallel kernel; len(ref) <= 512."""
    hyps = _need(hyps, torch.uint8, "hyps")
    shape = hyps.shape
    Th = shape[-1]
    flat = hyps.reshape(-1, Th)
    N = flat.shape[0]
    refs = _need(refs, torch.int32, "refs", 2)
    G, Lr = refs.shape
    if rows_per_ref is None:
        rows_per_ref = N // max(G, 1)
    if G * rows_per_ref != N:
        raise ValueError("hyps rows must be refs rows * rows_per_ref")
    hyp_len = _opt_i32(hyp_len, "hyp_len", N, hyps.device)
    ref_len = _opt_i32(ref_len, "ref_len", G, hyps.device)
    dist = torch.empty((N,), dtype=torch.int32, device=hyps.device)
    col = torch.zeros((N, Th + 1), dtype=torch.int32, device=hyps.device) if last_col else None
    _launch(hyps, "pgasr_edit_distance_u8", _ptr(flat), _ptr(hyp_len), N, Th, _ptr(refs), _ptr(ref_len),
                 rows_per_ref, Lr, int(vocab), _ptr(dist), _ptr(col))
    dist = dist.reshape(shape[:-1])
    return (dist, col.reshape(*shape[:-1], Th + 1)) if last_col else dist


def word_edit_distance(hyps, hyp_len, refs, sep, ref_len=None, rows_per_ref=None):
    """Word-level rows a1/a4: hyps [N,Th] (or [B,K,Th]) uint8, refs [G,Lr] int32, both split into words at the id
    `sep` (str.split(" ") semantics: empty words kept) -> (dist [N] int32 word edit distances, ref_words [G] int32 =
    words per reference).  len(ref) <= 511."""
    hyps = _need(hyps, torch.uint8, "hyps")
    shape = hyps.shape
    Th = shape[-1]
    flat = hyps.reshape(-1, Th)
    N = flat.shape[0]
    refs = _need(refs, torch.int32, "refs", 2)
    G, Lr = refs.shape
    if rows_per_ref is None:
        rows_per_ref = N // max(G, 1)
    if G * rows_per_ref != N:
        raise ValueError("hyps rows must be refs rows * rows_per_ref")
    hyp_len = _opt_i32(hyp_len, "hyp_len", N, hyps.device)
    ref_len = _opt_i32(ref_len, "ref_len", G, hyps.device)
    dist = torch.empty((N,), dtype=torch.int32, device=hyps.device)
    ref_words = torch.empty((G,), dtype=torch.int32, device=hyps.device)
    _launch(hyps, "pgasr_word_edit_distance_u8", _ptr(flat), _ptr(hyp_len), N, Th, _ptr(refs), _ptr(ref_len),
            rows_per_ref, Lr, int(sep), _ptr(dist), _ptr(ref_words))
    return dist.reshape(shape[:-1]), ref_words


def edit_distance_tokens(hyps, hyp_len, refs, ref_len=None, rows_per_ref=1):
    """Row a1 for arbitrary int32 tokens (word ids, code points): anti-diagonal wavefront kernel."""
    hyps = _need(hyps, torch.int32, "hyps", 2)
    refs = _need(refs, torch.int32, "refs", 2)
    N, Th = hyps.shape
    G, Lr = refs.shape
    if G * rows_per_ref != N:
        raise ValueError("hyps rows must be refs rows * rows_per_ref")
    hyp_len = _opt_i32(hyp_len, "hyp_len", N, hyps.device)
    ref_len = _opt_i32(ref_len, "ref_len", G, hyps.device)
    dist = torch.empty((N,), dtype=torch.int32, device=hyps.device)
    _launch(hyps, "pgasr_edit_distance_i32", _ptr(hyps), _ptr(hyp_len), N, Th, _ptr(refs), _ptr(ref_len),
                 rows_per_ref, Lr, _ptr(dist))
    return dist


def pg_advantages(dist, target_lengths, logp, reward="ed", baseline="mean", baseline_value=0.0, Lmax=0):
    """Row a7 (first half).  -> rewards [B,K], adv [B,K], loss_terms [B] (= -sum_k adv*logp)."""
    dist = _need(dist, torch.int32, "dist", 2)
    logp = _need(logp, torch.float32, "logp", 2)
    B, K = dist.shape
    tl = _opt_i32(target_lengths, "target_lengths", B, dist.device)
    rewards = torch.empty((B, K), dtype=torch.float32, device=dist.device)
    adv = torch.empty_like(rewards)
    terms = torch.empty((B,), dtype=torch.float32, device=dist.device)
    _launch(dist, "pgasr_pg_advantages", _ptr(dist), _ptr(tl), _ptr(logp), B, K, int(Lmax), REWARD_MODES[reward],
                 BASELINE_MODES[baseline], float(baseline_value), _ptr(rewards), _ptr(adv), _ptr(terms))
    return rewards, adv, terms


def pg_grad(samples, adv, input_lengths=None, probs=None, V=None, scale=1.0, out=None):
    """Row a7 (second half).  dlogits = scale * (probs * sum_k adv - scatter_k adv) -> [B,T,V].  With `out`
    the result is accumulated into it."""
    samples = _need(samples, torch.uint8, "samples", 3)
    adv = _need(adv, torch.float32, "adv", 2)
    B, K, T = samples.shape
    if probs is not None:
        probs = _need(probs, torch.float32, "probs", 3)
        V = probs.shape[2]
    if V is None:
        raise ValueError("V is required when probs is None")
    in_len = _opt_i32(input_lengths, "input_lengths", B, samples.device)
    acc = out is not None
    if out is None:
        out = torch.empty((B, T, V), dtype=torch.float32, device=samples.device)
    else:
        out = _need(out, torch.float32, "out", 3)
    _launch(samples, "pgasr_pg_grad", _ptr(samples), _ptr(adv), _ptr(probs), _ptr(in_len), B, T, V, K, float(scale),
                 1 if acc else 0, _ptr(out))
    return out


def ctc_loss_grad(logits, targets, input_lengths=None, target_lengths=None, blank=0, grad_scale=1.0,
                  probs=None, out=None):
    """Row a8.  -> nll [B] fp32, dlogits [B,T,V] = grad_scale * d nll_b / d logits_b.  With `out` the
    gradient is accumulated into it."""
    logits = _need(logits, torch.float32, "logits", 3)
    B, T, V = logits.shape
    targets = as_targets(targets, logits.device)
    Lmax = targets.shape[1]
    in_len = _opt_i32(input_lengths, "input_lengths", B, logits.device)
    tg_len = _opt_i32(target_lengths, "target_lengths", B, logits.device)
    if probs is not None:
        probs = _need(probs, torch.float32, "probs", 3)
    nll = torch.empty((B,), dtype=torch.float32, device=logits.device)
    acc = out is not None
    dlogits = _need(out, torch.float32, "out", 3) if acc else torch.empty_like(logits)
    nbytes = _native.lib().pgasr_ctc_workspace_bytes(B, T, V, Lmax)
    if nbytes == 0:
        raise _native.PgasrError("pgasr_ctc_workspace_bytes", -2, "unsupported size (Lmax <= 511)")
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=logits.device)
    _launch(logits, "pgasr_ctc_loss_grad", _ptr(logits), _ptr(probs), _ptr(targets), _ptr(in_len), _ptr(tg_len),
                 B, T, V, Lmax, int(blank), float(grad_scale), 1 if acc else 0, _ptr(nll), _ptr(dlogits),
                 _ptr(ws), nbytes)
    return nll, dlogits


def nll_sum_forward(inp, target, ignore_index=NO_IGNORE):
    """Row a5 (upstream loss.py:13-17).  inp [L,B,V] fp32 log-probs, target [B,L] int64 -> 0-d loss."""
    inp = _need(inp, torch.float32, "inp", 3)
    target = _need(target, torch.int64, "target", 2)
    L, B, V = inp.shape
    if target.shape[0] != B or target.shape[1] < L:
        raise IndexError("target must be [B, >=L]")
    if target.shape[1] != L:
        target = target[:, :L].contiguous()
    loss = torch.empty((1,), dtype=torch.float32, device=inp.device)
    _launch(inp, "pgasr_nll_sum_forward", _ptr(inp), _ptr(target), L, B, V, int(ignore_index), _ptr(loss))
    return loss[0]


def nll_sum_backward(target, grad_out, L, B, V, ignore_index=NO_IGNORE):
    target = _need(target, torch.int64, "target", 2)
    if target.shape[1] != L:
        target = target[:, :L].contiguous()
    grad_out = _need(grad_out.reshape(1), torch.float32, "grad_out")
    g = torch.empty((L, B, V), dtype=torch.float32, device=target.device)
    _launch(target, "pgasr_nll_sum_backward", _ptr(target), _ptr(grad_out), L, B, V, int(ignore_index), _ptr(g))
    return g


def ctc_beam_search(probs, input_lengths=None, beam_size=100, blank=0):
    """SURVEY 8f.2 (upstream CTCdecoder.py:41-116).  probs [N,T,V] fp64 post-softmax on the GPU ->
    labels [N,T] int32 (best prefix per utterance, zero padded), label_len [N] int32, nll [N] fp64."""
    probs = _need(probs, torch.float64, "probs", 3)
    N, T, V = probs.shape
    in_len = _opt_i32(input_lengths, "input_lengths", N, probs.device)
    nbytes = _native.lib().pgasr_ctc_beam_search_workspace_bytes(N, T, V, int(beam_size))
    if nbytes == 0:
        raise _native.PgasrError("pgasr_ctc_beam_search_workspace_bytes", -2,
                                 "unsupported size (V <= 256, beam <= 128; beam <= 104 at V = 256)")
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=probs.device)
    labels = torch.empty((N, T), dtype=torch.int32, device=probs.device)
    label_len = torch.empty((N,), dtype=torch.int32, device=probs.device)
    nll = torch.empty((N,), dtype=torch.float64, device=probs.device)
    _launch(probs, "pgasr_ctc_beam_search", _ptr(probs), _ptr(in_len), N, T, V, int(beam_size), int(blank),
                 _ptr(labels), _ptr(label_len), _ptr(nll), _ptr(ws), nbytes)
    return labels, label_len, nll


class StepWorkspace:
    """Device scratch of pgasr_pg_ctc_step, sized once per (B,T,V,K,Lmax) and reused across steps."""

    def __init__(self, B, T, V, K, Lmax, device):
        self.key = (B, T, V, K, Lmax)
        self.device = torch.device(device)
        self.nbytes = _native.lib().pgasr_pg_ctc_step_workspace_bytes(B, T, V, K, Lmax)
        if self.nbytes == 0:
            raise _native.PgasrError("pgasr_pg_ctc_step_workspace_bytes", -2, "unsupported size")
        self.buf = torch.empty((self.nbytes,), dtype=torch.uint8, device=device)
        _launch(self.buf, "pgasr_pg_ctc_step_workspace_init", _ptr(self.buf), self.nbytes)

    def outputs(self, want=("rewards", "nll")):
        """A fresh set of output tensors for one step on this workspace's shape (pass it as `out=` to reuse it)."""
        return _alloc_outputs(self.key, self.device, want)


_OUT_DTYPES = {"rewards": torch.float32, "logp": torch.float32, "hyp_len": torch.int32, "dist": torch.int32,
               "nll": torch.float32, "samples": torch.uint8, "to_go": torch.int16, "r_pos": torch.int8,
               "entropy": torch.float32}


def _alloc_outputs(key, dev, want):
    B, T, V, K, _ = key
    out = {"loss": torch.empty((1,), dtype=torch.float32, device=dev),
           "dlogits": torch.empty((B, T, V), dtype=torch.float32, device=dev)}
    for name in want:
        if name not in OPTIONAL_OUTPUTS + EXPLORE_OUTPUTS:
            raise ValueError(f"unknown output {name!r}; choose from {OPTIONAL_OUTPUTS + EXPLORE_OUTPUTS}")
        shape = (B,) if name in ("nll", "entropy") else (B, K, T) if name in ("samples", "to_go", "r_pos") else (B, K)
        out[name] = torch.empty(shape, dtype=_OUT_DTYPES[name], device=dev)
    return out


def _check_outputs(out, key, dev):
    B, T, V, K, _ = key
    for name, t in out.items():
        if name in ("workspace",):
            continue
        if name not in OPTIONAL_OUTPUTS + EXPLORE_OUTPUTS + ("loss", "dlogits"):
            raise ValueError(f"unknown output {name!r}")
        want_dt = torch.float32 if name in ("loss", "dlogits") else _OUT_DTYPES[name]
        n = 1 if name == "loss" else B * T * V if name == "dlogits" else B if name in ("nll", "entropy") else \
            B * K * T if name in ("samples", "to_go", "r_pos") else B * K
        if not (isinstance(t, torch.Tensor) and t.device == dev and t.dtype == want_dt and t.is_contiguous()
                and t.numel() == n):
            raise ValueError(f"out[{name!r}] must be a contiguous {want_dt} tensor of {n} elements on {dev}")


def _step_io(batch, out, seed=0):
    io = _native.StepIO()
    io.logits, io.targets = _ptr(batch["logits"]), _ptr(batch["targets"])
    io.in_len, io.tgt_len = _ptr(batch.get("in_len")), _ptr(batch.get("tgt_len"))
    io.uniforms, io.seed = _ptr(batch.get("uniforms")), int(seed) & (2**64 - 1)
    io.loss, io.dlogits = _ptr(out["loss"]), _ptr(out["dlogits"])
    for name in OPTIONAL_OUTPUTS:
        setattr(io, name, _ptr(out.get(name)))
    return io


def _prep_batch(logits, targets, input_lengths, target_lengths, uniforms, K):
    logits = _need(logits, torch.float32, "logits", 3)
    B, T, V = logits.shape
    dev = logits.device
    targets = as_targets(targets, dev)
    if targets.shape[0] != B:
        raise ValueError("targets must be [B, Lmax]")
    Lmax = targets.shape[1]
    if uniforms is not None:
        uniforms = _need(uniforms, torch.float32, "uniforms", 3)
        if uniforms.device != dev or uniforms.shape[0] != B or uniforms.shape[2] != T:
            raise ValueError(f"uniforms must be [B,K,T] = [{B},K,{T}] on {dev}, got {tuple(uniforms.shape)}")
        K = uniforms.shape[1]
    if not 1 <= int(K) <= 64:
        raise ValueError("K must be in 1..64")
    batch = {"logits": logits, "targets": targets, "in_len": _opt_i32(input_lengths, "input_lengths", B, dev),
             "tgt_len": _opt_i32(target_lengths, "target_lengths", B, dev), "uniforms": uniforms}
    return batch, (B, T, V, int(K), Lmax), dev


def check_explore(temperature, entropy_weight, pg_weight, want_entropy=False):
    """ValueError unless the exploration controls are valid (DESIGN.md "exploration spec"): temperature finite in
    [0.01, 100], entropy_weight finite and >= 0; the entropy bonus and the entropy output need the PG term."""
    t, w = float(temperature), float(entropy_weight)
    if not (math.isfinite(t) and 0.01 <= t <= 100.0):
        raise ValueError(f"temperature must be finite and in [0.01, 100], got {temperature!r}")
    if not (math.isfinite(w) and w >= 0.0):
        raise ValueError(f"entropy_weight must be finite and >= 0, got {entropy_weight!r}")
    if (w > 0.0 or want_entropy) and float(pg_weight) == 0.0:
        raise ValueError("the entropy bonus and the entropy output need the PG term (pg_weight != 0)")


def _step_entry(reward, blank, space_id, temperature=1.0, entropy_weight=0.0, want_entropy=False):
    """(entry point name, extra arguments before the workspace): non-default exploration controls or an entropy
    output go through pgasr_pg_ctc_step_multi_ex (its extra arguments follow the per-step entropy pointer array:
    word_sep, temperature, w_ent); otherwise the word rewards go through pgasr_pg_ctc_step_multi_ws with the
    separator id, every other mode through pgasr_pg_ctc_step_multi."""
    if reward not in REWARD_MODES:
        raise ValueError(f"unknown reward {reward!r}; choose from {tuple(REWARD_MODES)}")
    if reward in WORD_REWARDS:
        if space_id is None:
            raise ValueError(f"reward={reward!r} needs space_id, the id of the word separator (the space character)")
        if int(space_id) == int(blank):
            raise ValueError("space_id must differ from blank")
    if float(temperature) != 1.0 or float(entropy_weight) != 0.0 or want_entropy:
        sep = int(space_id) if reward in WORD_REWARDS else -1
        return "pgasr_pg_ctc_step_multi_ex", (sep, float(temperature), float(entropy_weight))
    if reward not in WORD_REWARDS:
        return "pgasr_pg_ctc_step_multi", ()
    return "pgasr_pg_ctc_step_multi_ws", (int(space_id),)


def _entropy_ptrs(outs):
    """The host array of per-step entropy pointers of pgasr_pg_ctc_step_multi_ex (NULL where not wanted)."""
    return (C.c_void_p * len(outs))(*[_ptr(o.get("entropy")) for o in outs])


def pg_ctc_step(logits, targets, input_lengths=None, target_lengths=None, K=16, blank=0, reward="ed",
                baseline="mean", baseline_value=0.0, pg_weight=1.0, ctc_weight=1.0, uniforms=None, seed=0,
                workspace=None, want=("rewards", "nll"), out=None, space_id=None, temperature=1.0,
                entropy_weight=0.0):
    """The whole loss step (rows a1-a8 chained) in one C-ABI call.
    Returns a dict: loss (0-d), dlogits [B,T,V], plus the optional outputs named in `want` out of
    rewards, logp, hyp_len, dist, nll, samples (and, with reward='ed_to_go', to_go and r_pos [B,K,T]).
    `out`: a dict from StepWorkspace.outputs() to write into instead of allocating (no allocation per step).
    reward='wed' / 'wer' (word edit distance, -WED / n_words): space_id is the id of the word separator; dist then
    holds word edit distances (hyp_len stays in ids).
    temperature / entropy_weight (DESIGN.md "exploration spec"): the PG term samples from and trains
    softmax(logits / temperature) and the loss gains -entropy_weight * mean_b H_b; 'entropy' in `want` returns H_b [B]
    (nats, summed over the utterance's frames).  The CTC term always uses the untempered logits."""
    want_entropy = "entropy" in (out if out is not None else want)
    check_explore(temperature, entropy_weight, pg_weight, want_entropy)
    entry, extra = _step_entry(reward, blank, space_id, temperature, entropy_weight, want_entropy)
    batch, key, dev = _prep_batch(logits, targets, input_lengths, target_lengths, uniforms, K)
    B, T, V, K, Lmax = key
    if workspace is None or workspace.key != key or workspace.device != dev:
        workspace = StepWorkspace(B, T, V, K, Lmax, dev)
    if out is None:
        out = _alloc_outputs(key, dev, want)
    else:
        _check_outputs(out, key, dev)
    io = _step_io(batch, out, seed)
    ent = (_entropy_ptrs([out]),) if entry == "pgasr_pg_ctc_step_multi_ex" else ()
    _launch(logits, entry, C.byref(io), 1, 0, B, T, V, K, Lmax, int(blank), REWARD_MODES[reward],
            BASELINE_MODES[baseline], float(baseline_value), float(pg_weight), float(ctc_weight), *ent, *extra,
            _ptr(workspace.buf), workspace.nbytes)
    res = dict(out)
    res["loss"] = out["loss"][0]
    res["workspace"] = workspace
    return res


class StepQueue:
    """n steps over a fixed set of device-resident batches with ONE C-ABI call per run() (pgasr_pg_ctc_step_multi):
    the micro-batches of one optimiser step, or a measurement loop.  Inputs are validated and every output buffer
    is allocated here, once; run() allocates nothing and costs one ctypes call however many steps it enqueues.

        q = StepQueue(batches, K=16, want=("rewards", "nll"))      # batches: dicts with logits, targets[, in_len, tgt_len, uniforms]
        q.run(first=0, n=len(batches), seed=step)                  # enqueue; results land in q.outputs[i]
    """

    def __init__(self, batches, K=16, blank=0, reward="ed", baseline="mean", baseline_value=0.0, pg_weight=1.0,
                 ctc_weight=1.0, want=("rewards", "nll"), workspace=None, space_id=None, temperature=1.0,
                 entropy_weight=0.0):
        check_explore(temperature, entropy_weight, pg_weight, "entropy" in want)
        self._entry, self._extra = _step_entry(reward, blank, space_id, temperature, entropy_weight, "entropy" in want)
        if not batches:
            raise ValueError("StepQueue needs at least one batch")
        self.batches, self.outputs = [], []
        self.key = self.device = None
        for bt in batches:
            batch, key, dev = _prep_batch(bt["logits"], bt["targets"], bt.get("in_len"), bt.get("tgt_len"),
                                          bt.get("uniforms"), K)
            if self.key is None:
                self.key, self.device = key, dev
            elif key != self.key or dev != self.device:
                raise ValueError("all batches of a StepQueue must have one shape and live on one device")
            self.batches.append(batch)
            self.outputs.append(_alloc_outputs(key, dev, want))
        B, T, V, K, Lmax = self.key
        self.workspace = workspace if workspace is not None and workspace.key == self.key else \
            StepWorkspace(B, T, V, K, Lmax, self.device)
        self.params = (int(blank), REWARD_MODES[reward], BASELINE_MODES[baseline], float(baseline_value),
                       float(pg_weight), float(ctc_weight))
        n = len(self.batches)
        # the record array holds every batch twice, so any window of up to n consecutive steps starting anywhere in
        # the cycle is one contiguous slice (no per-call marshalling); step i of a run samples with seed + i
        self._io = (_native.StepIO * (2 * n))()
        for i in range(2 * n):
            self._io[i] = _step_io(self.batches[i % n], self.outputs[i % n], seed=i)
        self._stride = C.sizeof(_native.StepIO)
        # pgasr_pg_ctc_step_multi_ex: the entropy pointers, doubled like the records
        self._ent = _entropy_ptrs(self.outputs * 2) if self._entry == "pgasr_pg_ctc_step_multi_ex" else None

    def run(self, first=0, n=None, seed=0):
        """Enqueue steps on batches first, first+1, ... (cyclically), n <= len(batches) of them; returns n."""
        nb = len(self.batches)
        n = nb if n is None else int(n)
        if not 0 <= n <= nb:
            raise ValueError(f"n must be in 0..{nb}")
        first = int(first) % nb
        B, T, V, K, Lmax = self.key
        base = C.addressof(self._io) + first * self._stride
        ent = () if self._ent is None else (C.addressof(self._ent) + first * C.sizeof(C.c_void_p),)
        _launch(self.workspace.buf, self._entry, base, n, (int(seed) - first) & (2**64 - 1), B, T, V, K,
                Lmax, *self.params, *ent, *self._extra, _ptr(self.workspace.buf), self.workspace.nbytes)
        return n
