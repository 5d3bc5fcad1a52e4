"""ctypes binding of oracle/hfa_oracle_lowmem.c -- TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

The DP of ``c_oracle.decode`` at about 0.25 B per cell, for utterances whose [T][S] dp / backpointer
matrices do not fit the host: the emission rows come from a callback, chunk by chunk, so the caller can
regenerate them instead of holding them."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "hfa_oracle_lowmem.c")
_SO = os.path.join(_HERE, "_build", "libhfa_oracle_lowmem.so")
_lib = None

_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")


def build(force: bool = False) -> str:
    """Compiles the library with the flags of oracle/Makefile (the arithmetic contract needs them)."""
    if force or not os.path.isfile(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        tmp = f"{_SO}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O3", "-fPIC", "-std=c11", "-ffp-contract=off",
                               "-fno-fast-math", "-Wall", "-Wextra", "-shared", "-o", tmp, _SRC, "-lm"])
        os.replace(tmp, _SO)
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        L.hfa_lowmem_create.argtypes = [C.c_int32, C.c_int32, _i32p]
        L.hfa_lowmem_create.restype = C.c_void_p
        L.hfa_lowmem_destroy.argtypes = [C.c_void_p]
        L.hfa_lowmem_destroy.restype = None
        L.hfa_lowmem_rows.argtypes = [C.c_void_p, C.c_int32, _f32p, C.c_int64, _f32p, _f32p]
        L.hfa_lowmem_rows.restype = C.c_int
        L.hfa_lowmem_finish.argtypes = [C.c_void_p, _i32p, _i32p, _i32p, _i32p, _f32p]
        L.hfa_lowmem_finish.restype = C.c_int
        L.hfa_lowmem_path_rows.argtypes = [C.c_void_p, C.c_int32, _f32p, C.c_int64, _f32p, _f32p, _f32p]
        L.hfa_lowmem_path_rows.restype = C.c_int
        _lib = L
    return _lib


def decode_rows(ph_ids, T: int, rows, edge_log, not_edge_log, chunk: int = 4096, want_dp_path: bool = True):
    """rows(t0, t1) -> f32 [t1 - t0, S] gathered emissions of frames t0 .. t1-1 (called in order, once per
    chunk and pass; twice over all frames when ``want_dp_path``).  Returns what ``c_oracle.decode`` returns
    (rc, ph_idx_seq, ph_time_int, dp_path, end_state) plus final_score = dp[T-1][end_state]; dp_path is None
    without ``want_dp_path``."""
    L = lib()
    ids = np.ascontiguousarray(ph_ids, dtype=np.int32)
    S = len(ids)
    el = np.ascontiguousarray(edge_log, dtype=np.float32)
    ne = np.ascontiguousarray(not_edge_log, dtype=np.float32)
    assert T >= 1 and S >= 1 and len(el) == T and len(ne) == T
    h = L.hfa_lowmem_create(T, S, ids)
    if not h:
        raise MemoryError(f"hfa_lowmem_create(T={T}, S={S}) failed")
    try:
        def feed(fn, *extra):
            for t0 in range(0, T, chunk):
                t1 = min(T, t0 + chunk)
                e = np.ascontiguousarray(rows(t0, t1), dtype=np.float32)
                assert e.shape == (t1 - t0, S)
                rc = fn(h, t1 - t0, e, S, el[t0:t1], ne[t0:t1], *(x[t0:t1] for x in extra))
                assert rc == 0

        feed(L.hfa_lowmem_rows)
        idx = np.zeros(S, np.int32)
        tim = np.zeros(S, np.int32)
        n, es = np.zeros(1, np.int32), np.zeros(1, np.int32)
        fs = np.zeros(1, np.float32)
        rc = L.hfa_lowmem_finish(h, idx, tim, n, es, fs)
        dp_path = None
        if rc == 0 and want_dp_path:
            dp_path = np.zeros(T, np.float32)
            feed(L.hfa_lowmem_path_rows, dp_path)
    finally:
        L.hfa_lowmem_destroy(h)
    k = int(n[0]) if rc == 0 else 0
    return dict(rc=rc, ph_idx_seq=idx[:k].copy(), ph_time_int=tim[:k].copy(), dp_path=dp_path,
                end_state=int(es[0]), final_score=fs[0])


def decode(ph_ids, prob_log, edge_log, not_edge_log, chunk: int = 4096):
    """``c_oracle.decode`` on a [T, S] matrix in memory (the pin against the full oracle)."""
    e = np.ascontiguousarray(prob_log, dtype=np.float32)
    return decode_rows(ph_ids, e.shape[0], lambda t0, t1: e[t0:t1], edge_log, not_edge_log, chunk)
