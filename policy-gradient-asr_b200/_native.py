"""ctypes binding of libpgasr_b200.so (the C ABI declared in include/pgasr.h).

There is no CPU fallback: if the library has not been built, or a call fails, this raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PGASR_LIB") or os.path.join(_HERE, "lib", "libpgasr_b200.so")   # PGASR_LIB: tools only

_vp, _i, _f, _u64, _sz = C.c_void_p, C.c_int, C.c_float, C.c_uint64, C.c_size_t

# name -> (restype, argtypes); mirrors include/pgasr.h one to one (tests check the two against each other)
SIGNATURES = {
    "pgasr_abi_version": (_i, []),
    "pgasr_status_string": (C.c_char_p, [_i]),
    "pgasr_last_cuda_error": (_i, []),
    "pgasr_launch_count": (_u64, []),
    "pgasr_device_check": (_i, []),
    "pgasr_softmax_sample": (_i, [_vp, _vp, _vp, _u64, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "pgasr_collapse_u8": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pgasr_edit_distance_u8": (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "pgasr_word_edit_distance_u8": (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "pgasr_edit_distance_i32": (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _i, _vp, _vp]),
    "pgasr_pg_advantages": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp, _vp, _vp, _vp]),
    "pgasr_pg_grad": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _i, _vp, _vp]),
    "pgasr_ctc_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "pgasr_ctc_loss_grad": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _i, _vp, _vp, _vp, _sz, _vp]),
    "pgasr_nll_sum_forward": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "pgasr_nll_sum_backward": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "pgasr_pg_ctc_step_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "pgasr_pg_ctc_step_workspace_init": (_i, [_vp, _sz, _vp]),
    "pgasr_pg_ctc_step": (_i, [_vp, _vp, _vp, _vp, _vp, _u64, _i, _i, _i, _i, _i, _i, _i, _i, _f, _f, _f,
                               _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pgasr_pg_ctc_step_multi": (_i, [_vp, _i, _u64, _i, _i, _i, _i, _i, _i, _i, _i, _f, _f, _f, _vp, _sz, _vp]),
    "pgasr_pg_ctc_step_multi_ws": (_i, [_vp, _i, _u64, _i, _i, _i, _i, _i, _i, _i, _i, _f, _f, _f, _i, _vp, _sz, _vp]),
    "pgasr_pg_ctc_step_multi_ex": (_i, [_vp, _i, _u64, _i, _i, _i, _i, _i, _i, _i, _i, _f, _f, _f, _vp, _i, _f, _f,
                                        _vp, _sz, _vp]),
    "pgasr_ctc_beam_search_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "pgasr_ctc_beam_search": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pgasr_host_create": (_i, [_i, _i, _i, _i, _i, _i, _vp]),
    "pgasr_host_destroy": (_i, [_vp]),
    "pgasr_host_submit": (_i, [_vp, _vp, _vp, _vp, _vp, _u64, _i, _i, _i, _f, _f, _f, _vp, _vp, _vp, _vp, _vp]),
    "pgasr_host_wait": (_i, [_vp, C.c_int64]),
    "pgasr_host_pin": (_i, [_vp, _sz]),
    "pgasr_host_unpin": (_i, [_vp]),
}


class StepIO(C.Structure):
    """struct pgasr_step_io (include/pgasr.h): the device pointers of one step of pgasr_pg_ctc_step_multi."""
    _fields_ = [("logits", _vp), ("targets", _vp), ("in_len", _vp), ("tgt_len", _vp), ("uniforms", _vp),
                ("seed", _u64), ("loss", _vp), ("dlogits", _vp), ("rewards", _vp), ("logp", _vp),
                ("hyp_len", _vp), ("dist", _vp), ("nll", _vp), ("samples", _vp), ("to_go", _vp), ("r_pos", _vp)]


class PgasrError(RuntimeError):
    def __init__(self, fn, status, detail):
        super().__init__(f"{fn} failed: status {status} ({detail})")
        self.status = status


_lib = None


def lib():
    """The loaded library.  Raises if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python policy-gradient-asr_b200/build.py` "
                "(or __graft_entry__.build()); pgasr_b200 has no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.pgasr_abi_version() != 1:
            raise RuntimeError("libpgasr_b200.so ABI version mismatch; rebuild")
        _lib = L
    return _lib


def check(fn_name, status):
    if status != 0:
        L = lib()
        detail = L.pgasr_status_string(status).decode()
        if status == -5:
            detail += f", cudaError {L.pgasr_last_cuda_error()}"
        raise PgasrError(fn_name, status, detail)


def call(fn_name, *args):
    check(fn_name, getattr(lib(), fn_name)(*args))
