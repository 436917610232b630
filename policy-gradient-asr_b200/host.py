"""The PG + CTC step on HOST arrays (upstream hands host arrays to its reward/metric code: model.py:317-320).

HostPipeline wraps the pgasr_host_* entry points of the C ABI: `depth` steps in flight, the H2D copy of the next
step and the D2H copy of the previous one overlapping the kernel of the current one.  Inputs and outputs are
page-locked CPU tensors (torch `pin_memory()`); pageable tensors work but make the copies synchronous.

    pipe = HostPipeline(B, T, V, K, Lmax, depth=3)
    bufs = pipe.output_buffers()                       # pinned: loss[1], dlogits[B,T,V], rewards[B,K], nll[B]
    ticket = pipe.submit(logits_h, targets_h, in_len_h, tgt_len_h, out=bufs, seed=step)
    ...                                                # submit more steps (each with its own `out`)
    pipe.wait(ticket)                                  # bufs now hold this step's results

There is no CPU fallback: constructing a pipeline without an sm_100 device raises.
"""
import ctypes as C

import torch

from . import _native
from .functional import BASELINE_MODES, REWARD_MODES, WORD_REWARDS


def _host(t, dtype, name, numel=None, optional=False):
    if t is None:
        if optional:
            return None
        raise TypeError(f"{name} is required")
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor on the CPU")
    if t.is_cuda:
        raise TypeError(f"{name} must be a HOST tensor (use functional.pg_ctc_step for device tensors)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    if numel is not None and t.numel() != numel:
        raise ValueError(f"{name} must have {numel} elements, got {t.numel()}")
    return t


class HostPipeline:
    def __init__(self, B, T, V, K, Lmax, depth=3, blank=0, reward="ed", baseline="mean", baseline_value=0.0,
                 pg_weight=1.0, ctc_weight=1.0, temperature=1.0, entropy_weight=0.0):
        if reward in WORD_REWARDS:
            raise ValueError(f"reward={reward!r} (word level) is not available on host buffers; use "
                             "functional.pg_ctc_step or PolicyGradCTCLoss with device tensors")
        if float(temperature) != 1.0 or float(entropy_weight) != 0.0:
            raise ValueError("temperature and entropy_weight are not available on host buffers; use "
                             "functional.pg_ctc_step or PolicyGradCTCLoss with device tensors")
        self.shape = (int(B), int(T), int(V), int(K), int(Lmax))
        self.depth = int(depth)
        self.blank, self.reward, self.baseline = int(blank), REWARD_MODES[reward], BASELINE_MODES[baseline]
        self.baseline_value, self.pg_weight, self.ctc_weight = float(baseline_value), float(pg_weight), float(ctc_weight)
        self._h = C.c_void_p()
        self._keep = {}                                   # ticket -> tensors the in-flight copies read/write
        _native.call("pgasr_host_create", *self.shape, self.depth, C.byref(self._h))

    def output_buffers(self):
        """A fresh set of pinned output tensors for one step."""
        B, T, V, K, _ = self.shape
        return {"loss": torch.empty((1,), dtype=torch.float32).pin_memory(),
                "dlogits": torch.empty((B, T, V), dtype=torch.float32).pin_memory(),
                "rewards": torch.empty((B, K), dtype=torch.float32).pin_memory(),
                "nll": torch.empty((B,), dtype=torch.float32).pin_memory()}

    def submit(self, logits, targets, input_lengths=None, target_lengths=None, out=None, seed=0):
        """Enqueue one step; returns its ticket.  `out` (see output_buffers) receives the results."""
        if not self._h:
            raise RuntimeError("pipeline is closed")
        B, T, V, K, Lmax = self.shape
        logits = _host(logits, torch.float32, "logits", B * T * V)
        targets = _host(targets, torch.int32, "targets", B * Lmax)
        il = _host(input_lengths, torch.int32, "input_lengths", B, optional=True)
        tl = _host(target_lengths, torch.int32, "target_lengths", B, optional=True)
        if out is None:
            out = self.output_buffers()
        loss = _host(out["loss"], torch.float32, "out['loss']", 1)
        dlog = _host(out["dlogits"], torch.float32, "out['dlogits']", B * T * V)
        rew = _host(out.get("rewards"), torch.float32, "out['rewards']", B * K, optional=True)
        nll = _host(out.get("nll"), torch.float32, "out['nll']", B, optional=True)
        ticket = C.c_int64(-1)
        ptr = lambda t: None if t is None else t.data_ptr()
        _native.call("pgasr_host_submit", self._h, ptr(logits), ptr(targets), ptr(il), ptr(tl),
                     int(seed) & (2**64 - 1), self.blank, self.reward, self.baseline, self.baseline_value,
                     self.pg_weight, self.ctc_weight, ptr(loss), ptr(dlog), ptr(rew), ptr(nll), C.byref(ticket))
        self._keep[ticket.value] = (logits, targets, il, tl, out)
        for old in [k for k in self._keep if k <= ticket.value - self.depth]:
            del self._keep[old]                            # the C side has already waited for those steps
        return ticket.value

    def wait(self, ticket=-1):
        """Block until the outputs of every step up to `ticket` (default: all) are in their host buffers."""
        if not self._h:
            raise RuntimeError("pipeline is closed")
        _native.call("pgasr_host_wait", self._h, int(ticket))
        for old in [k for k in self._keep if ticket < 0 or k <= ticket]:
            del self._keep[old]

    def step(self, logits, targets, input_lengths=None, target_lengths=None, out=None, seed=0):
        """Synchronous convenience: submit + wait; returns the output dict."""
        out = out if out is not None else self.output_buffers()
        self.wait(self.submit(logits, targets, input_lengths, target_lengths, out=out, seed=seed))
        return out

    def close(self):
        if self._h:
            _native.call("pgasr_host_destroy", self._h)
            self._h = C.c_void_p()
            self._keep.clear()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
