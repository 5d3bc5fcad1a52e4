"""ctypes binding of libhfa_align.so (the C ABI in include/hfa_align.h).

The library is built in-tree (``hubertfa_b200/libhfa_align.so``) by ``__graft_entry__.build()`` or
``make -C hubertfa_b200/csrc``.  There is no fallback of any kind: if the shared object is missing
or does not export the ABI this module raises, and every compute entry point fails without CUDA.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhfa_align.so")

HFA_OK = 0
DTYPE_F32, DTYPE_F16, DTYPE_BF16 = 0, 1, 2
UTT_OK, UTT_EMPTY, UTT_BAD_ID, UTT_NO_STATES, UTT_INFEASIBLE, UTT_TOO_MANY_STATES = range(6)
MAX_STATES = 1 << 20   # include/hfa_align.h HFA_MAX_STATES
ABI_VERSION = 2


class HfaError(RuntimeError):
    pass


class ResultLayout(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("total_bytes", "status", "n_seg", "end_state", "final_score",
                                         "total_conf", "ph_idx_seq", "ph_time_int", "intervals")]


# every symbol include/hfa_align.h declares: (restype, argtypes)
_vp, _i32, _i64, _dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
SYMBOLS = {
    "hfa_abi_version": (C.c_int, []),
    "hfa_last_error": (C.c_char_p, []),
    "hfa_launch_count": (_i64, []),
    "hfa_plan_create": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _dbl, C.POINTER(_vp)]),
    "hfa_plan_destroy": (None, [_vp]),
    "hfa_plan_workspace_bytes": (_i64, [_vp]),
    "hfa_plan_total_frames": (_i64, [_vp]),
    "hfa_plan_total_states": (_i64, [_vp]),
    "hfa_plan_total_cells": (_i64, [_vp]),
    "hfa_plan_frame_offsets": (C.POINTER(_i64), [_vp]),
    "hfa_plan_seg_offsets": (C.POINTER(_i64), [_vp]),
    "hfa_plan_result_layout": (C.c_int, [_vp, C.POINTER(ResultLayout)]),
    "hfa_plan_algorithmic_bytes": (C.c_int, [_vp, _i32, C.POINTER(_i64 * 3)]),
    "hfa_plan_debug_region": (_i64, [_vp, _i32, C.POINTER(_i64)]),
    "hfa_plan_routing": (C.c_int, [_vp, C.POINTER(_i32 * 8)]),
    "hfa_plan_pair_utterances": (_i32, [_vp]),
    "hfa_plan_skew_ctas_per_sm": (_i32, [_vp, _i32]),
    "hfa_plan_stored_emission_bytes": (_i64, [_vp]),
    "hfa_debug_unpack_emissions": (C.c_int, [_vp, _vp, _vp, _vp]),
    "hfa_plan_upload": (C.c_int, [_vp, _vp, _vp]),
    "hfa_set_inputs": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hfa_set_inputs_device": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "hfa_release_thread_resources": (None, []),
    "hfa_emission": (C.c_int, [_vp, _vp, _i32, _vp]),
    "hfa_pack_emissions": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hfa_viterbi_forward": (C.c_int, [_vp, _vp, _vp, _vp]),
    "hfa_backtrace": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "hfa_align_batch": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp]),
    "hfa_forward_fused": (C.c_int, [_vp, _vp, _i32, _vp]),
    "hfa_plan_algorithmic_bytes_fused": (_i64, [_vp, _i32]),
    "hfa_debug_unpack_backptr": (C.c_int, [_vp, _vp, _i32, _vp, _vp]),
    "hfa_debug_unpack_dp": (C.c_int, [_vp, _vp, _i32, _vp, _vp]),
    "hfa_ctc_greedy": (C.c_int, [_vp, _i32, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _vp]),
}

_lib = None


def load():
    """Loads libhfa_align.so and binds every ABI symbol; raises HfaError if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise HfaError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
                       "g.build()'` or `make -C hubertfa_b200/csrc` (there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise HfaError(f"{LIB_PATH} does not export {name}") from e
        fn.restype = res
        fn.argtypes = args
    if lib.hfa_abi_version() != ABI_VERSION:
        raise HfaError(f"ABI version mismatch: library {lib.hfa_abi_version()}, binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != HFA_OK:
        msg = load().hfa_last_error().decode("utf-8", "replace")
        raise HfaError(f"{what or 'libhfa_align'} failed with code {rc}: {msg}")
