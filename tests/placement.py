"""Buffers at chosen element offsets, and the multi-step C entry points called on hand-built step records.

Shared by tests/test_buffer_placement.py and tools/variant_matrix.py.  torch's allocator hands out 512-byte aligned
storage, so without these helpers every device pointer the suite passes is 16-byte aligned; include/pgasr.h promises
that an array argument needs only its element's natural alignment.
"""
import ctypes as C

import numpy as np
import torch


def at_offset(array, elems, device, fill=None):
    """A contiguous device tensor that starts `elems` elements into a larger flat buffer, holding `array` (numpy or
    torch) -- or, with array a (shape, dtype) pair, uninitialised / `fill`-ed storage of that shape."""
    if isinstance(array, tuple):
        shape, dtype = array
        src = None
    else:
        src = torch.as_tensor(np.ascontiguousarray(array)) if isinstance(array, np.ndarray) else array
        shape, dtype = tuple(src.shape), src.dtype
    n = int(np.prod(shape, dtype=np.int64))
    buf = torch.empty((n + elems + 16,), dtype=dtype, device=device)
    if fill is not None:
        buf.fill_(fill)
    view = buf[elems:elems + n].view(shape)
    if src is not None:
        view.copy_(src)
    nbytes = elems * view.element_size()
    assert view.is_contiguous() and view.storage_offset() == elems
    if nbytes % 16:
        assert view.data_ptr() % 16 != 0, "the view was meant to be misaligned for 16-byte accesses"
    return view


# fill of the output buffers placed by the tests: an element the kernel never writes shows up in a bit-for-bit compare
OUT_FILL = {torch.float32: float("nan"), torch.int32: -7, torch.int16: -7, torch.int8: -7, torch.uint8: 0xEE}


def offset_outputs(F, key, device, want, elems):
    """What functional._alloc_outputs returns, with every tensor `elems` elements into its own buffer."""
    ref = F._alloc_outputs(key, device, want)
    return {k: at_offset((tuple(t.shape), t.dtype), elems, device, fill=OUT_FILL[t.dtype]) for k, t in ref.items()}


def multi_step(F, batches, outs, K, reward="ed", baseline="mean", baseline_value=0.0, w_pg=1.0, w_ctc=1.0,
               space_id=None, temperature=1.0, entropy_weight=0.0, seed=0, blank=0):
    """One call of the multi-step entry point StepQueue would use, on records built from `batches` / `outs` as given
    (step i samples with seed + i).  Unlike StepQueue this keeps every pointer where the caller put it."""
    from pgasr_b200 import _native
    want_ent = any("entropy" in o for o in outs)
    entry, extra = F._step_entry(reward, blank, space_id, temperature, entropy_weight, want_ent)
    B, T, V = batches[0]["logits"].shape
    Lmax = batches[0]["targets"].shape[1]
    dev = batches[0]["logits"].device
    n = len(batches)
    recs = (_native.StepIO * n)(*[F._step_io(b, o, seed=i) for i, (b, o) in enumerate(zip(batches, outs))])
    ent_arr = F._entropy_ptrs(outs) if entry == "pgasr_pg_ctc_step_multi_ex" else None
    ent = () if ent_arr is None else (C.addressof(ent_arr),)
    ws = F.StepWorkspace(B, T, V, K, Lmax, dev)
    with torch.cuda.device(dev):
        _native.call(entry, C.addressof(recs), n, int(seed), B, T, V, K, Lmax, int(blank), F.REWARD_MODES[reward],
                     F.BASELINE_MODES[baseline], float(baseline_value), float(w_pg), float(w_ctc), *ent, *extra,
                     ws.buf.data_ptr(), ws.nbytes, torch.cuda.current_stream(dev).cuda_stream)
    return outs
