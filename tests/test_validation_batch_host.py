"""CPU: argument checks of the batch-validation entry points (hfa_ctc_greedy_batch, hfa_frame_states) and the
layout of the ctc descriptor table the plan builds.  Every check here fails before anything touches a device."""
import ctypes as C

import numpy as np

from hubertfa_b200 import _lib, ops

ERR_ARG = -1
FAKE = 0x10000          # never dereferenced: the calls below are refused before any CUDA call


def _plan():
    return ops.AlignPlan([10, 70], [2, 1], np.array([0, 1, 0], np.int32), 8, 0.02)


def test_ctc_greedy_batch_rejects_bad_arguments():
    lib, plan = _lib.load(), _plan()
    h = plan.handle
    ok = dict(plan=h, ws=FAKE, table=FAKE, V=8, dtype=_lib.DTYPE_F32, scratch=FAKE, ids=FAKE, len=FAKE)
    bad = [dict(plan=None), dict(ws=None), dict(table=None), dict(scratch=None), dict(ids=None), dict(len=None),
           dict(V=0), dict(V=-3), dict(V=1 << 31), dict(dtype=3), dict(dtype=-1)]
    for change in bad:
        a = {**ok, **change}
        rc = lib.hfa_ctc_greedy_batch(a["plan"], a["ws"], a["table"], a["V"], a["dtype"], a["scratch"], a["ids"],
                                      a["len"], None)
        assert rc == ERR_ARG, change
        assert b"hfa_ctc_greedy_batch" in lib.hfa_last_error()


def test_frame_states_rejects_bad_arguments():
    lib, plan = _lib.load(), _plan()
    for args in ((None, FAKE, FAKE, FAKE), (plan.handle, None, FAKE, FAKE), (plan.handle, FAKE, None, FAKE),
                 (plan.handle, FAKE, FAKE, None)):
        assert lib.hfa_frame_states(*args, None) == ERR_ARG, args
        assert b"hfa_frame_states" in lib.hfa_last_error()


def test_ctc_table_is_the_c_descriptor():
    class HfaCtcDesc(C.Structure):            # include/hfa_align.h
        _fields_ = [("logits", C.c_void_p), ("stride_t", C.c_int64), ("stride_v", C.c_int64)]

    plan = _plan()
    tab = plan.ctc_table([0x1000, 0x2000], [40, 8], [1, 2])
    assert tab.dtype == np.uint8 and tab.size == 2 * C.sizeof(HfaCtcDesc)
    descs = (HfaCtcDesc * 2).from_buffer_copy(tab.tobytes())
    assert [(d.logits, d.stride_t, d.stride_v) for d in descs] == [(0x1000, 40, 1), (0x2000, 8, 2)]
