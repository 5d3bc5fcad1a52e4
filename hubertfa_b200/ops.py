"""Thin torch-facing layer over the C ABI: an ``AlignPlan`` (collation of one ragged batch) and the
``hfa::*`` torch custom ops that forward raw device pointers and the current CUDA stream to
libhfa_align.so.  PyTorch is only plumbing here (device memory, streams); all compute is in the
hand-written sm_100a kernels under ``csrc/``.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import HfaError, ResultLayout, check


def _stream_ptr() -> int:
    return int(torch.cuda.current_stream().cuda_stream)


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise HfaError(f"{what} must be a CUDA tensor: the aligner has no CPU path")


class AlignPlan:
    """Host-side collation of one ragged batch (wraps ``hfa_plan``).

    T, S: per-utterance frame / state counts; ph_ids: concatenated phoneme ids
    (alignment_decoder.py:35); frame_length = hop_length / sample_rate (:12).
    """

    def __init__(self, T, S, ph_ids, vocab_size: int, frame_length: float):
        lib = _lib.load()
        self.T = np.ascontiguousarray(T, dtype=np.int32)
        self.S = np.ascontiguousarray(S, dtype=np.int32)
        self.ph_ids = np.ascontiguousarray(ph_ids, dtype=np.int32)
        if self.T.shape != self.S.shape or self.T.ndim != 1:
            raise ValueError("T and S must be 1-D arrays of the same length")
        if int(np.maximum(self.S, 0).sum()) != self.ph_ids.size:
            raise ValueError("ph_ids must hold sum(S) entries")
        self.n_utt = int(self.T.size)
        self.vocab_size = int(vocab_size)
        self.frame_length = float(frame_length)
        handle = C.c_void_p()
        check(lib.hfa_plan_create(self.n_utt, self.vocab_size, self.T.ctypes.data, self.S.ctypes.data,
                                  self.ph_ids.ctypes.data, self.frame_length, C.byref(handle)),
              "hfa_plan_create")
        self._h = handle
        self._lib = lib
        self.workspace_bytes = int(lib.hfa_plan_workspace_bytes(handle))
        self.total_frames = int(lib.hfa_plan_total_frames(handle))
        self.total_states = int(lib.hfa_plan_total_states(handle))
        self.total_cells = int(lib.hfa_plan_total_cells(handle))
        n1 = self.n_utt + 1
        self.frame_off = np.ctypeslib.as_array(lib.hfa_plan_frame_offsets(handle), shape=(n1,)).copy()
        self.seg_off = np.ctypeslib.as_array(lib.hfa_plan_seg_offsets(handle), shape=(n1,)).copy()
        self.layout = ResultLayout()
        check(lib.hfa_plan_result_layout(handle, C.byref(self.layout)), "hfa_plan_result_layout")
        self.result_bytes = int(self.layout.total_bytes)

    @property
    def handle(self) -> int:
        if self._h is None:
            raise HfaError("plan already destroyed")
        return int(self._h.value)

    def routing(self) -> dict:
        """Which forward-pass kernels the plan chose for this batch (hfa_plan_routing)."""
        out = (C.c_int32 * 8)()
        check(self._lib.hfa_plan_routing(self._h, C.byref(out)))
        return dict(warp_utts=out[0], band_warps=out[1], band_k=out[2], big_band_warps=out[3],
                    big_band_k=out[4], cta_utts=out[5], keeps_dp=bool(out[6]), skew_d=out[7],
                    pair_utts=int(self._lib.hfa_plan_pair_utterances(self._h)),
                    skew_ctas_per_sm=int(self._lib.hfa_plan_skew_ctas_per_sm(self._h, 0)),
                    big_skew_ctas_per_sm=int(self._lib.hfa_plan_skew_ctas_per_sm(self._h, 1)),
                    stored_emission_bytes=int(self._lib.hfa_plan_stored_emission_bytes(self._h)))

    def algorithmic_bytes_fused(self, dtype: int = _lib.DTYPE_F32) -> int:
        return int(self._lib.hfa_plan_algorithmic_bytes_fused(self._h, dtype))

    def algorithmic_bytes(self, dtype: int = _lib.DTYPE_F32):
        out = (C.c_int64 * 3)()
        check(self._lib.hfa_plan_algorithmic_bytes(self._h, dtype, C.byref(out)))
        return {"emission": int(out[0]), "dp": int(out[1]), "backtrace": int(out[2])}

    def new_workspace(self, device) -> torch.Tensor:
        return torch.empty(max(self.workspace_bytes, 256), dtype=torch.uint8, device=device)

    def new_result(self, device) -> torch.Tensor:
        return torch.empty(self.result_bytes, dtype=torch.uint8, device=device)

    def upload(self, workspace: torch.Tensor) -> None:
        _require_cuda(workspace, "workspace")
        if workspace.numel() < self.workspace_bytes:
            raise HfaError("workspace too small for this plan")
        with torch.cuda.device(workspace.device):
            check(self._lib.hfa_plan_upload(self._h, workspace.data_ptr(), _stream_ptr()),
                  "hfa_plan_upload")

    def set_inputs(self, workspace: torch.Tensor, frame_ptrs, frame_st, frame_sv, edge_ptrs, edge_st):
        """Pointer / stride tables (host int64 arrays, one entry per utterance, strides in elements)."""
        tabs = [np.ascontiguousarray(a, dtype=np.int64) for a in
                (frame_ptrs, frame_st, frame_sv, edge_ptrs, edge_st)]
        if any(a.shape != (self.n_utt,) for a in tabs):
            raise ValueError("input tables must have one entry per utterance")
        with torch.cuda.device(workspace.device):
            check(self._lib.hfa_set_inputs(self._h, workspace.data_ptr(), *[a.ctypes.data for a in tabs],
                                           _stream_ptr()), "hfa_set_inputs")

    INPUT_DESC = np.dtype([("frame", np.int64), ("edge", np.int64), ("frame_stride_t", np.int64),
                           ("frame_stride_v", np.int64), ("edge_stride", np.int64)])    # = HfaInputDesc

    def input_table(self, frame_ptrs, frame_st, frame_sv, edge_ptrs, edge_st) -> np.ndarray:
        """Host image of the per-utterance input table (HfaInputDesc[n_utt]) plus the row-stride promise
        ``set_inputs_device`` needs: returns (table as uint8 array, max_row_stride)."""
        tab = np.zeros(self.n_utt, dtype=self.INPUT_DESC)
        for name, a in zip(self.INPUT_DESC.names, (frame_ptrs, edge_ptrs, frame_st, frame_sv, edge_st)):
            tab[name] = np.asarray(a, dtype=np.int64)
        ok = self.T > 0
        tma = bool(np.all(tab["frame_stride_v"][ok] == 1) and np.all(tab["frame_stride_t"][ok] >= self.vocab_size)
                   and np.all(tab["frame"][ok] % 4 == 0))
        stride = int(tab["frame_stride_t"][ok].max()) if ok.any() else 0
        return tab.view(np.uint8), (stride if tma else 0)

    def set_inputs_device(self, workspace: torch.Tensor, table: torch.Tensor, max_row_stride: int) -> None:
        """The input table already on the device (uint8 tensor holding HfaInputDesc[n_utt]): a device-to-
        device copy, capturable into a CUDA graph (hfa_set_inputs_device)."""
        _require_cuda(table, "input table")
        if table.numel() * table.element_size() < self.n_utt * self.INPUT_DESC.itemsize:
            raise HfaError("input table too small for this plan")
        with torch.cuda.device(workspace.device):
            check(self._lib.hfa_set_inputs_device(self._h, workspace.data_ptr(), table.data_ptr(),
                                                  int(max_row_stride), _stream_ptr()), "hfa_set_inputs_device")

    def views(self, blob: np.ndarray) -> dict:
        """Typed numpy views into a host copy of the result blob."""
        L, n, ns = self.layout, self.n_utt, self.total_states

        def v(off, dtype, count):
            return blob[off:off + count * np.dtype(dtype).itemsize].view(dtype)

        return dict(status=v(L.status, np.int32, n), n_seg=v(L.n_seg, np.int32, n),
                    end_state=v(L.end_state, np.int32, n), final_score=v(L.final_score, np.float32, n),
                    total_conf=v(L.total_conf, np.float32, n),
                    ph_idx_seq=v(L.ph_idx_seq, np.int32, ns), ph_time_int=v(L.ph_time_int, np.int32, ns),
                    intervals=v(L.intervals, np.float64, 2 * ns).reshape(ns, 2))

    def debug_region(self, workspace: torch.Tensor, which: str) -> torch.Tensor:
        """Test helper: typed view of an intermediate workspace buffer."""
        code = {"emis": 0, "edge2": 1, "edge_p": 2, "bp": 3, "xchg": 4}[which]
        nb = C.c_int64()
        off = int(self._lib.hfa_plan_debug_region(self._h, code, C.byref(nb)))
        raw = workspace[off:off + int(nb.value)]
        if which in ("bp", "xchg"):
            return raw.view(torch.int32)
        v = raw.view(torch.float32)
        return v.view(-1, 2) if which == "edge2" else v

    def close(self) -> None:
        if getattr(self, "_h", None) is not None:
            self._lib.hfa_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# --------------------------------------------------------------------------------------------
# torch custom ops: (workspace, plan handle, ...) -> kernels on the current stream
# --------------------------------------------------------------------------------------------
def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


@torch.library.custom_op("hfa::emission", mutates_args=("workspace",), device_types="cuda")
def emission(workspace: torch.Tensor, plan: int, dtype: int) -> None:
    with torch.cuda.device(workspace.device):
        check(_lib.load().hfa_emission(plan, workspace.data_ptr(), dtype, _stream_ptr()), "hfa_emission")


@torch.library.custom_op("hfa::pack_emissions", mutates_args=("workspace",), device_types="cuda")
def pack_emissions(workspace: torch.Tensor, plan: int, prob_log: torch.Tensor, edge_log: torch.Tensor,
                   not_edge_log: torch.Tensor, edge_pred: Optional[torch.Tensor]) -> None:
    for t in (prob_log, edge_log, not_edge_log):
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise HfaError("pack_emissions expects contiguous float32 tensors")
    with torch.cuda.device(workspace.device):
        check(_lib.load().hfa_pack_emissions(plan, workspace.data_ptr(), prob_log.data_ptr(),
                                             edge_log.data_ptr(), not_edge_log.data_ptr(),
                                             _ptr(edge_pred), _stream_ptr()), "hfa_pack_emissions")


@torch.library.custom_op("hfa::viterbi_forward", mutates_args=("workspace", "dp_dump"),
                         device_types="cuda")
def viterbi_forward(workspace: torch.Tensor, plan: int, dp_dump: Optional[torch.Tensor]) -> None:
    with torch.cuda.device(workspace.device):
        check(_lib.load().hfa_viterbi_forward(plan, workspace.data_ptr(), _ptr(dp_dump), _stream_ptr()),
              "hfa_viterbi_forward")


@torch.library.custom_op("hfa::backtrace", mutates_args=("workspace", "result", "frame_conf", "dp_path"),
                         device_types="cuda")
def backtrace(workspace: torch.Tensor, plan: int, result: torch.Tensor,
              frame_conf: Optional[torch.Tensor], dp_path: Optional[torch.Tensor]) -> None:
    with torch.cuda.device(workspace.device):
        check(_lib.load().hfa_backtrace(plan, workspace.data_ptr(), result.data_ptr(), _ptr(frame_conf),
                                        _ptr(dp_path), _stream_ptr()), "hfa_backtrace")


@torch.library.custom_op("hfa::align_batch", mutates_args=("workspace", "result", "frame_conf"),
                         device_types="cuda")
def align_batch(workspace: torch.Tensor, plan: int, dtype: int, result: torch.Tensor,
                frame_conf: Optional[torch.Tensor]) -> None:
    with torch.cuda.device(workspace.device):
        check(_lib.load().hfa_align_batch(plan, workspace.data_ptr(), dtype, result.data_ptr(),
                                          _ptr(frame_conf), _stream_ptr()), "hfa_align_batch")


@torch.library.custom_op("hfa::forward_fused", mutates_args=("workspace",), device_types="cuda")
def forward_fused(workspace: torch.Tensor, plan: int, dtype: int) -> None:
    """Edge stream + banded DP with the emissions computed inside the kernel (small batches only;
    raises HfaError when the plan / inputs do not qualify)."""
    with torch.cuda.device(workspace.device):
        check(_lib.load().hfa_forward_fused(plan, workspace.data_ptr(), dtype, _stream_ptr()), "hfa_forward_fused")


class GraphedStep:
    """One whole step -- (optionally) the device-side input table copy, hfa_align_batch, the download of
    the result blob into pinned host memory -- captured ONCE into a CUDA graph and replayed with a single
    launch.  For fixed-shape batches that are aligned over and over (a serving loop over length buckets, the
    benchmark): the five kernel launches, the stream forks and their event records stop costing host time.

    plan / workspace must be uploaded (``plan.upload``) and, unless ``table`` is given, have their inputs
    set before the capture.  ``table``: device uint8 tensor with HfaInputDesc[n_utt]; it is re-read at every
    replay, so the caller may point the step at new logits by rewriting it (same shapes)."""

    def __init__(self, plan: AlignPlan, workspace: torch.Tensor, result: torch.Tensor, host_result: torch.Tensor,
                 dtype: int, frame_conf: Optional[torch.Tensor] = None, table: Optional[torch.Tensor] = None,
                 max_row_stride: int = 0, warmup: int = 2):
        if not host_result.is_pinned():
            raise HfaError("host_result must be pinned memory")
        self.plan, self.host_result = plan, host_result
        dev = workspace.device

        def body():
            if table is not None:
                plan.set_inputs_device(workspace, table, max_row_stride)
            align_batch(workspace, plan.handle, dtype, result, frame_conf)
            host_result.copy_(result, non_blocking=True)

        with torch.cuda.device(dev):
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):                  # warm-up outside the capture (lazy module loads)
                for _ in range(max(warmup, 1)):
                    body()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize(dev)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                body()

    def replay(self) -> None:
        """Enqueues the step on the current stream (results are in ``host_result`` once it has drained)."""
        self.graph.replay()


def unpack_backptr(plan: AlignPlan, workspace: torch.Tensor, utt: int) -> torch.Tensor:
    """Test helper: int8 [T, S] backpointers of one utterance (row 0 = -1)."""
    out = torch.empty((int(plan.T[utt]), int(plan.S[utt])), dtype=torch.int8, device=workspace.device)
    with torch.cuda.device(workspace.device):
        check(_lib.load().hfa_debug_unpack_backptr(plan.handle, workspace.data_ptr(), utt, out.data_ptr(),
                                                   _stream_ptr()), "hfa_debug_unpack_backptr")
    return out


def unpack_kept_dp(plan: AlignPlan, workspace: torch.Tensor, utt: int) -> torch.Tensor:
    """Test helper: f32 [T, S] dp cells the (production) forward pass kept for the table backtrace."""
    out = torch.empty((int(plan.T[utt]), int(plan.S[utt])), dtype=torch.float32, device=workspace.device)
    with torch.cuda.device(workspace.device):
        check(_lib.load().hfa_debug_unpack_dp(plan.handle, workspace.data_ptr(), utt, out.data_ptr(),
                                              _stream_ptr()), "hfa_debug_unpack_dp")
    return out


def unpack_emissions(plan: AlignPlan, workspace: torch.Tensor) -> torch.Tensor:
    """Test helper: the emissions the workspace holds as dense ragged f32 [sum T_b * S_b] (utterance b at its
    cell offset, [T_b, S_b] row-major), whether the rows are stored plain or compacted per distinct id."""
    out = torch.empty(max(plan.total_cells, 1), dtype=torch.float32, device=workspace.device)
    with torch.cuda.device(workspace.device):
        check(_lib.load().hfa_debug_unpack_emissions(plan.handle, workspace.data_ptr(), out.data_ptr(),
                                                     _stream_ptr()), "hfa_debug_unpack_emissions")
    return out


def launch_count() -> int:
    return int(_lib.load().hfa_launch_count())


TORCH_TO_DTYPE = {torch.float32: _lib.DTYPE_F32, torch.float16: _lib.DTYPE_F16,
                  torch.bfloat16: _lib.DTYPE_BF16}


def ctc_greedy(logits: torch.Tensor) -> torch.Tensor:
    """Greedy CTC decode of one utterance on the device (alignment_decoder.py:145-150).
    logits: CUDA tensor [T, V] (any strides; f32 / f16 / bf16).  Returns the int32 id sequence."""
    if logits.dim() != 2 or not logits.is_cuda:
        raise HfaError("ctc_greedy expects a CUDA tensor [T, V]")
    if logits.dtype not in TORCH_TO_DTYPE:
        logits = logits.float()
    T, V = int(logits.shape[0]), int(logits.shape[1])
    dev = logits.device
    scratch = torch.empty(max(T, 1), dtype=torch.int32, device=dev)
    out = torch.empty(max(T, 1), dtype=torch.int32, device=dev)
    n = torch.zeros(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(_lib.load().hfa_ctc_greedy(logits.data_ptr(), TORCH_TO_DTYPE[logits.dtype], T, V, logits.stride(0),
                                         logits.stride(1), scratch.data_ptr(), out.data_ptr(), n.data_ptr(),
                                         _stream_ptr()), "hfa_ctc_greedy")
    return out[: int(n.item())]
