"""Drop-in replacement for the reference's ``tools.alignment_decoder.AlignmentDecoder``.

Same constructor, same ``decode(...)`` signature and 5-tuple result, same attributes afterwards
(``ctc()`` / ``plot()`` keep working in ``validation_step``, networks/task/forced_alignment.py:
407-414), plus ``decode_batch`` which aligns a whole ragged batch in one pass of the sm_100a
kernels.  Everything numeric between the logits and the per-segment intervals runs on the GPU
through libhfa_align.so; there is no CPU implementation in this package.

Reference: tools/alignment_decoder.py (``ad:<line>`` below).
"""
from __future__ import annotations

from typing import Sequence

import numpy as np
import torch

from . import _lib, ops
from ._lib import HfaError


def _as_2d(frame: torch.Tensor) -> torch.Tensor:
    """[1,T,V] or [T,V] -> [T,V] view (the reference squeezes dim 0, ad:57)."""
    if frame.dim() == 3:
        if frame.shape[0] != 1:
            raise ValueError("per-utterance logits must have batch size 1 (ad:57 squeeze(0))")
        return frame[0]
    if frame.dim() != 2:
        raise ValueError("frame logits must be [1,T,V] or [T,V]")
    return frame


def _as_1d(edge: torch.Tensor) -> torch.Tensor:
    if edge.dim() == 2:
        if edge.shape[0] != 1:
            raise ValueError("per-utterance edge logits must have batch size 1")
        return edge[0]
    if edge.dim() != 1:
        raise ValueError("edge logits must be [1,T] or [T]")
    return edge


def _masked_logits(frame_logits: torch.Tensor, ph_seq_id, vocab_size: int) -> torch.Tensor:
    """ad:53-59: the frame logits with every phoneme outside the sequence (SP excepted) pushed down by 1e9."""
    drop = np.ones(vocab_size, dtype=bool)
    drop[ph_seq_id] = False
    drop[0] = False
    pen = torch.from_numpy(drop).to(frame_logits.device)[None, None, :] * 1e9
    return frame_logits.float() - pen.float()


def _ph_frame_pred(frame_logits: torch.Tensor, ph_seq_id, vocab_size: int) -> np.ndarray:
    """ad:56-59,73: softmax of the masked [1,T,V] logits -> f32 [T, V]."""
    return torch.nn.functional.softmax(_masked_logits(frame_logits, ph_seq_id, vocab_size), dim=-1
                                       ).squeeze(0).cpu().numpy().astype("float32")


def _edge_prob(edge_logits: torch.Tensor) -> np.ndarray:
    """ad:68-71,84: the edge probability of the [1,T] edge logits, spread onto the frame after it."""
    p = (((torch.sigmoid(edge_logits.float()) - 0.1) / 0.8).clamp(0.0, 1.0)).squeeze(0).cpu().numpy().astype("float32")
    return (p + np.concatenate(([0], p[:-1]))).clip(0, 1)


class BatchAlignment:
    """Result of :meth:`AlignmentDecoder.decode_batch` (host resident, numeric part vectorised).

    Ragged arrays are indexed by ``seg_off`` (raw segments, capacity S per utterance),
    ``ph_off`` (phonemes kept after the SP filter, ad:123) and ``word_off`` (merged words, ad:128).
    ``result[b]`` gives utterance ``b`` as the reference's 5-tuple.

    What ``validation_step`` reads after ``decode()`` (forced_alignment.py:407-414) is here per utterance too:
    ``ctc(b)`` (with ``ctc_logits``), ``ph_idx_frame(b)`` (``frame_state``, with ``want_frame_states``),
    ``ph_frame_pred(b)`` / ``edge_prob(b)`` (computed on demand, like the decoder's attributes) and
    ``plot(b, melspec)``.
    """

    def __init__(self, plan: ops.AlignPlan, views: dict, ph_seqs, word_seqs, ph2word, is_sp, word_idx,
                 frame_conf=None, ctc=None, frame_state=None, inputs=None):
        self.n_utt = plan.n_utt
        self.T = plan.T
        self.S = plan.S
        self.seg_off = plan.seg_off
        self.frame_off = plan.frame_off
        self.status = views["status"]
        self.n_seg = views["n_seg"]
        self.end_state = views["end_state"]
        self.final_score = views["final_score"]
        self.total_confidence = views["total_conf"]
        self.ph_idx_seq = views["ph_idx_seq"]
        self.ph_time_int = views["ph_time_int"]
        self.raw_intervals = views["intervals"]
        self.frame_confidence = frame_conf
        # ctc(): ids of utterance b at ctc_ids[frame_off[b] : frame_off[b] + ctc_len[b]]
        self.ctc_ids, self.ctc_len = ctc if ctc is not None else (None, None)
        self.frame_state = frame_state            # int32 [sum T]: state index of the best path at every frame
        self.frame_length = plan.frame_length
        self.vocab_size = plan.vocab_size
        # (frame logits, edge logits, ph_seq_id) per utterance, trimmed, on the device: for ph_frame_pred / edge_prob.
        # Kept only for validation batches (ctc_logits / want_frame_states): they hold the logits alive.
        self._inputs = inputs
        self._ph_seqs, self._word_seqs, self._ph2word = ph_seqs, word_seqs, ph2word
        self._filter_and_merge(is_sp, word_idx)

    def _filter_and_merge(self, is_sp: np.ndarray, word_idx: np.ndarray) -> None:
        # ad:121-138 for the whole batch at once.  Slot j of utterance b is a live segment when
        # j < n_seg[b]; it survives when its phoneme label is not "SP".
        n, seg_off = self.n_utt, self.seg_off
        total = int(seg_off[-1])
        utt_of = np.repeat(np.arange(n, dtype=np.int64), np.diff(seg_off))
        slot = np.arange(total, dtype=np.int64) - seg_off[:-1][utt_of]
        live = slot < self.n_seg[utt_of]
        gidx = seg_off[:-1][utt_of] + np.where(live, self.ph_idx_seq, 0)   # global state index
        keep = live & ~is_sp[gidx]
        self.keep = keep
        self.ph_utt = utt_of[keep]
        self.ph_state = self.ph_idx_seq[keep].astype(np.int64)             # index into ph_seq
        iv = self.raw_intervals[keep]
        self.ph_intervals = iv.clip(min=0)                                  # ad:136
        self.ph_off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(np.bincount(self.ph_utt, minlength=n), out=self.ph_off[1:])
        w = word_idx[gidx[keep]]
        if w.size:
            first = np.ones(w.size, dtype=bool)
            first[1:] = (w[1:] != w[:-1]) | (self.ph_utt[1:] != self.ph_utt[:-1])
            last = np.ones(w.size, dtype=bool)
            last[:-1] = first[1:]
            self.word_index = w[first]
            self.word_utt = self.ph_utt[first]
            self.word_intervals = np.stack([iv[first, 0], iv[last, 1]], axis=1).clip(min=0)  # ad:138
        else:
            self.word_index = np.zeros(0, dtype=np.int64)
            self.word_utt = np.zeros(0, dtype=np.int64)
            self.word_intervals = np.zeros((0, 2), dtype=np.float64)
        self.word_off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(np.bincount(self.word_utt, minlength=n), out=self.word_off[1:])

    def __len__(self) -> int:
        return self.n_utt

    def segments(self, b: int):
        """Raw (ph_idx_seq int64, ph_time_int int64, intervals f64 [K,2]) of utterance b (ad:99-113)."""
        o, k = int(self.seg_off[b]), int(self.n_seg[b])
        return (self.ph_idx_seq[o:o + k].astype(np.int64), self.ph_time_int[o:o + k].astype(np.int64),
                self.raw_intervals[o:o + k])

    def _require_aligned(self, b: int) -> None:
        if self.status[b] not in (_lib.UTT_OK, _lib.UTT_INFEASIBLE):
            raise HfaError(f"utterance {b} was not aligned (status {int(self.status[b])})")

    def __getitem__(self, b: int):
        """Utterance b as the reference's 5-tuple (ad:143)."""
        self._require_aligned(b)
        ph_seq, word_seq = self._ph_seqs[b], self._word_seqs[b]
        p0, p1 = int(self.ph_off[b]), int(self.ph_off[b + 1])
        w0, w1 = int(self.word_off[b]), int(self.word_off[b + 1])
        ph_pred = np.array([ph_seq[i] for i in self.ph_state[p0:p1]])
        word_pred = np.array([word_seq[i] for i in self.word_index[w0:w1]])
        ph_iv = self.ph_intervals[p0:p1] if p1 > p0 else np.array([]).clip(min=0)
        word_iv = self.word_intervals[w0:w1] if w1 > w0 else np.array([]).clip(min=0)
        return ph_pred, ph_iv, word_pred, word_iv, np.float32(self.total_confidence[b])

    def ctc(self, b: int) -> np.ndarray:
        """Greedy CTC ids of utterance b, int64: what ``decode(); ctc()`` returns (ad:145-150)."""
        self._require_aligned(b)
        if self.ctc_ids is None:
            raise HfaError("ctc() needs decode_batch(..., ctc_logits=...)")
        f0 = int(self.frame_off[b])
        return self.ctc_ids[f0:f0 + int(self.ctc_len[b])].astype(np.int64)

    def ph_idx_frame(self, b: int) -> np.ndarray:
        """State index of the best path at every frame of utterance b: the ph_idx_frame plot() builds
        (ad:156-161)."""
        self._require_aligned(b)
        if self.frame_state is None:
            raise HfaError("ph_idx_frame() needs decode_batch(..., want_frame_states=True)")
        return self.frame_state[int(self.frame_off[b]):int(self.frame_off[b + 1])].astype(np.int64)

    def _inputs_of(self, b: int):
        self._require_aligned(b)
        if self._inputs is None:
            raise HfaError("the logits are kept for decode_batch(..., ctc_logits=... or want_frame_states=True) only")
        return self._inputs[b]

    def ph_frame_pred(self, b: int) -> np.ndarray:
        """f32 [T, V] masked softmax of utterance b's frame logits (the decoder's ``ph_frame_pred``, ad:73)."""
        frame, _, ids = self._inputs_of(b)
        return _ph_frame_pred(frame[None], ids, self.vocab_size)

    def edge_prob(self, b: int) -> np.ndarray:
        """f32 [T] edge probability of utterance b (the decoder's ``edge_prob``, ad:84)."""
        return _edge_prob(self._inputs_of(b)[1][None])

    def plot(self, b: int, melspec):
        """ad:152-168 for utterance b: plot_for_valid with the arguments ``decode(); plot()`` passes.  Needs
        ``want_frame_confidence`` and ``want_frame_states``, and the reference's ``tools.plot`` on the path."""
        from tools.plot import plot_for_valid  # provided by the reference checkout

        ph_pred, ph_iv = self[b][:2]
        if self.frame_confidence is None:
            raise HfaError("plot() needs decode_batch(..., want_frame_confidence=True)")
        f0, f1 = int(self.frame_off[b]), int(self.frame_off[b + 1])
        ids = self._inputs_of(b)[2]
        return plot_for_valid(melspec.cpu().numpy(), ph_pred, (ph_iv / self.frame_length).round().astype("int32"),
                              self.frame_confidence[f0:f1].copy(), self.ph_frame_pred(b)[:, ids],
                              self.ph_idx_frame(b), self.edge_prob(b))


class AlignmentDecoder:
    """Same interface as the reference class (ad:8-168); compute runs on the current CUDA device."""

    # How decode() / decode_batch() reach hfa_align_batch.  False (default): the C ABI is called directly
    # through ctypes.  True: through the ``hfa::align_batch`` torch custom op (same entry point, same stream).
    # Measured on B200, one T=500 / S=40 utterance per call (tools/time_decode.py): 0.40 ms per decode() through
    # the op against 0.28 ms direct -- torch's Python custom-op dispatcher costs ~0.1 ms per call, more than the
    # 0.064 ms the kernels take, and predict_step (forced_alignment.py:174-176) pays it once per utterance.
    # The ops stay the interface for graph capture, the benchmark and the stage-level tests.
    dispatch_through_torch_op = False

    def __init__(self, vocab, melspec_config, device=None):
        _lib.load()                           # fail at construction if the CUDA library is missing
        self.vocab = vocab
        self.melspec_config = melspec_config
        self.frame_length = self.melspec_config["hop_length"] / (self.melspec_config["sample_rate"])
        self.device = torch.device(device) if device is not None else None

        self.ctc_logits = None
        self.ph_seq_id = None
        self.ph_idx_seq = None
        self.ph_frame_pred = None
        self.ph_time_int_pred = None
        self.ph_intervals_pred = None
        self.edge_prob = None
        self.ph_pred_seq = None
        self.frame_confidence = None

    # ----------------------------------------------------------------------------------------
    def _device_for(self, t: torch.Tensor) -> torch.device:
        if t.is_cuda:
            return t.device
        if self.device is not None:
            return self.device
        if not torch.cuda.is_available():
            raise HfaError("no CUDA device: hubertfa_b200 has no CPU fallback")
        return torch.device("cuda", torch.cuda.current_device())

    def _ids_of(self, ph_seq) -> np.ndarray:
        """ad:35 (KeyError for an unknown phoneme) and the bounds numpy enforces at ad:38 / :239: ids are
        used as indices into [V] arrays, so -V <= id < V, negative ones counting from the end."""
        V = self.vocab["vocab_size"]
        ids = np.array([self.vocab["vocab"][ph] for ph in ph_seq])
        if ids.size and (ids.min() < -V or ids.max() >= V):
            raise IndexError("phoneme id out of bounds for vocab_size")
        return np.where(ids < 0, ids + V, ids)

    def _num_frames(self, wav_length, T: int) -> int:
        if wav_length is None:
            return T
        n = int((wav_length * self.melspec_config["sample_rate"] + 0.5) / self.melspec_config["hop_length"])
        return min(T, n) if n >= 0 else max(T + n, 0)      # python slice semantics of ad:48

    def _run(self, frames, edges, ids_list, want_frame_conf: bool, ctcs=None, want_states: bool = False):
        """frames/edges: per-utterance 2-D / 1-D CUDA tensors (views allowed, already trimmed).  ctcs: None or
        per-utterance 2-D ctc logits (one dtype and width, T rows each) for hfa_ctc_greedy_batch; want_states:
        hfa_frame_states after the alignment.  Both run on the same stream, before the one synchronise."""
        dev = frames[0].device
        dtype = frames[0].dtype
        if dtype not in ops.TORCH_TO_DTYPE:
            frames = [f.float() for f in frames]
            edges = [e.float() for e in edges]
            dtype = torch.float32
        for f, e in zip(frames, edges):
            if f.dtype != dtype or e.dtype != dtype or f.device != dev or e.device != dev:
                raise HfaError("all logits of a batch must share one dtype and one device")
        T = np.array([f.shape[0] for f in frames], dtype=np.int32)
        S = np.array([len(i) for i in ids_list], dtype=np.int32)
        ids = np.concatenate(ids_list).astype(np.int32) if len(ids_list) else np.zeros(0, np.int32)
        plan = ops.AlignPlan(T, S, ids, self.vocab["vocab_size"], self.frame_length)
        # One device context, the plan's tables and ONE hfa_align_batch call (emission -> DP -> backtrace on
        # the current stream; see dispatch_through_torch_op).  Pinned result buffers are kept across calls.
        lib = _lib.load()
        n = len(frames)
        tabs = [np.fromiter((f.data_ptr() for f in frames), dtype=np.int64, count=n),
                np.fromiter((f.stride(0) for f in frames), dtype=np.int64, count=n),
                np.fromiter((f.stride(1) for f in frames), dtype=np.int64, count=n),
                np.fromiter((e.data_ptr() for e in edges), dtype=np.int64, count=n),
                np.fromiter((e.stride(0) for e in edges), dtype=np.int64, count=n)]
        with torch.cuda.device(dev):
            ws = plan.new_workspace(dev)
            res = plan.new_result(dev)
            fc = torch.empty(max(plan.total_frames, 1), dtype=torch.float32, device=dev) \
                if want_frame_conf else None
            stream = torch.cuda.current_stream()
            sp, h, wp = int(stream.cuda_stream), plan.handle, ws.data_ptr()
            _lib.check(lib.hfa_plan_upload(h, wp, sp), "hfa_plan_upload")
            _lib.check(lib.hfa_set_inputs(h, wp, *[a.ctypes.data for a in tabs], sp), "hfa_set_inputs")
            if self.dispatch_through_torch_op:
                ops.align_batch(ws, h, ops.TORCH_TO_DTYPE[dtype], res, fc)
            else:
                _lib.check(lib.hfa_align_batch(h, wp, ops.TORCH_TO_DTYPE[dtype], res.data_ptr(),
                                               fc.data_ptr() if fc is not None else None, sp), "hfa_align_batch")
            nf = max(plan.total_frames, 1)
            extra = {}                     # device outputs of the validation kernels -> pinned host copies
            if ctcs is not None:
                ctab = torch.from_numpy(plan.ctc_table(
                    np.fromiter((c.data_ptr() for c in ctcs), dtype=np.int64, count=n),
                    np.fromiter((c.stride(0) for c in ctcs), dtype=np.int64, count=n),
                    np.fromiter((c.stride(1) for c in ctcs), dtype=np.int64, count=n))).to(dev)
                ids_d = torch.empty(nf, dtype=torch.int32, device=dev)
                len_d = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
                scratch = torch.empty(nf, dtype=torch.int32, device=dev)
                Vc = int(ctcs[0].shape[1]) if n else 1
                _lib.check(lib.hfa_ctc_greedy_batch(h, wp, ctab.data_ptr(), Vc, ops.TORCH_TO_DTYPE[ctcs[0].dtype],
                                                    scratch.data_ptr(), ids_d.data_ptr(), len_d.data_ptr(), sp),
                           "hfa_ctc_greedy_batch")
                extra["ctc_ids"], extra["ctc_len"] = ids_d, len_d
            if want_states:
                st_d = torch.empty(nf, dtype=torch.int32, device=dev)
                _lib.check(lib.hfa_frame_states(h, wp, res.data_ptr(), st_d.data_ptr(), sp), "hfa_frame_states")
                extra["states"] = st_d
            host = self._pinned("res", plan.result_bytes, torch.uint8)
            host.copy_(res, non_blocking=True)
            fc_host = None
            if fc is not None:
                fc_host = self._pinned("fc", fc.numel(), torch.float32)
                fc_host.copy_(fc, non_blocking=True)
            for k, d in extra.items():
                extra[k] = self._pinned(k, d.numel(), d.dtype)
                extra[k].copy_(d, non_blocking=True)
            stream.synchronize()
        # the pinned buffers are reused by the next call: hand out copies
        host = host.numpy().copy()
        if fc_host is not None:
            fc_host = fc_host.numpy().copy()
        views = plan.views(host)
        out = dict(frame_conf=fc_host[:plan.total_frames] if fc_host is not None else None)
        if ctcs is not None:
            out["ctc"] = (extra["ctc_ids"].numpy()[:plan.total_frames].copy(), extra["ctc_len"].numpy()[:n].copy())
        if want_states:
            out["frame_state"] = extra["states"].numpy()[:plan.total_frames].copy()
        return plan, views, out, ws

    def _pinned(self, key: str, numel: int, dtype) -> torch.Tensor:
        cache = self.__dict__.setdefault("_pin_cache", {})
        buf = cache.get(key)
        if buf is None or buf.numel() < numel or buf.dtype != dtype:
            buf = torch.empty(max(int(numel * 1.5), 1024), dtype=dtype, pin_memory=True)
            cache[key] = buf
        return buf[:numel]

    # ----------------------------------------------------------------------------------------
    def decode(self,
               ph_frame_logits,
               ph_edge_logits,
               ctc_logits,
               wav_length: float | None,
               ph_seq: list[str],
               word_seq: list[str] = None,
               ph_idx_to_word_idx: list[int] = None
               ):
        ph_seq_id = self._ids_of(ph_seq)                                           # ad:35 (KeyError), :38
        self.ph_seq_id = ph_seq_id
        if word_seq is None:                                                       # ad:41-43
            word_seq = ph_seq
            ph_idx_to_word_idx = np.arange(len(ph_seq))

        if wav_length is not None:                                                 # ad:45-50
            num_frames = int(
                (wav_length * self.melspec_config["sample_rate"] + 0.5) / self.melspec_config["hop_length"])
            ph_frame_logits = ph_frame_logits[:, :num_frames, :]
            ph_edge_logits = ph_edge_logits[:, :num_frames]
            ctc_logits = ctc_logits[:, :num_frames, :] if ctc_logits is not None else None

        dev = self._device_for(ph_frame_logits)
        frame = _as_2d(ph_frame_logits).to(dev)
        edge = _as_1d(ph_edge_logits).to(dev)
        T = frame.shape[0]
        if T < 1 or len(ph_seq_id) < 1:
            raise IndexError("index 0 is out of bounds for axis 0 with size 0")    # ad:250

        plan, v, out, _ = self._run([frame], [edge], [ph_seq_id.astype(np.int32)], True)
        fc = out["frame_conf"]
        if v["status"][0] not in (_lib.UTT_OK, _lib.UTT_INFEASIBLE):
            raise HfaError(f"alignment failed with status {int(v['status'][0])}")
        k = int(v["n_seg"][0])
        ph_idx_seq = v["ph_idx_seq"][:k].astype(np.int64)
        ph_time_int_pred = v["ph_time_int"][:k].astype(np.int64)
        ph_intervals = v["intervals"][:k]
        total_confidence = np.float32(v["total_conf"][0])

        self._frame_logits, self._edge_logits, self._ctc_src = ph_frame_logits, ph_edge_logits, ctc_logits
        self._lazy = {}
        self.ph_idx_seq = ph_idx_seq
        self.ph_time_int_pred = ph_time_int_pred
        self.frame_confidence = fc.copy()
        self.final_score = np.float32(v["final_score"][0])

        # ad:115-138 for one utterance: drop the segments labelled "SP", then merge runs of consecutive
        # phonemes that belong to the same word into one [first start, last end] interval
        from itertools import groupby
        kept = [i for i, st in enumerate(ph_idx_seq) if ph_seq[st] != "SP"]
        ph_seq_pred = np.array([ph_seq[ph_idx_seq[i]] for i in kept])
        ph_intervals_pred = (ph_intervals[kept] if kept else np.array([])).clip(min=0, max=None)
        runs = [(w, list(g)) for w, g in groupby(kept, key=lambda i: ph_idx_to_word_idx[ph_idx_seq[i]])]
        word_seq_pred = np.array([word_seq[w] for w, _ in runs])
        word_intervals_pred = np.array([[ph_intervals[g[0], 0], ph_intervals[g[-1], 1]]
                                        for _, g in runs]).clip(min=0, max=None)

        self.ph_pred_seq = ph_seq_pred
        self.ph_intervals_pred = ph_intervals_pred
        return ph_seq_pred, ph_intervals_pred, word_seq_pred, word_intervals_pred, total_confidence

    # ----------------------------------------------------------------------------------------
    def decode_batch(self, ph_frame_logits, ph_edge_logits, ph_seqs: Sequence[Sequence[str]],
                     word_seqs=None, ph_idx_to_word_idxs=None, wav_lengths=None, lengths=None,
                     want_frame_confidence: bool = False, ctc_logits=None,
                     want_frame_states: bool = False) -> BatchAlignment:
        """Aligns a ragged batch in one pass.

        ph_frame_logits / ph_edge_logits: either lists of per-utterance tensors ([1,T,V] / [1,T], the
        shapes ``decode`` takes, strided views allowed), or one packed tensor [sum T, V] / [sum T]
        with ``lengths`` giving T per utterance.  Host tensors are copied to the device first.

        For validation (what ``decode(); ctc(); plot()`` give per utterance): ``ctc_logits`` in the same form
        as the frame logits (one width for the batch) is decoded greedily for every utterance in one launch,
        ``want_frame_states`` expands the best paths into per-frame state indices in one more; both run on the
        alignment's stream and come back with its single synchronise.  See ``BatchAlignment.ctc`` /
        ``ph_idx_frame`` / ``plot``.
        """
        n = len(ph_seqs)
        ids_list = [self._ids_of(seq).astype(np.int32) for seq in ph_seqs]        # same checks as decode()
        if isinstance(ph_frame_logits, torch.Tensor):
            if lengths is None:
                raise ValueError("packed logits need `lengths`")
            dev = self._device_for(ph_frame_logits)
            fcat = ph_frame_logits.to(dev, non_blocking=True)
            ecat = ph_edge_logits.to(dev, non_blocking=True)
            offs = np.concatenate([[0], np.cumsum(np.asarray(lengths, dtype=np.int64))])
            frames = [fcat[offs[b]:offs[b + 1]] for b in range(n)]
            edges = [ecat[offs[b]:offs[b + 1]] for b in range(n)]
            if ctc_logits is not None:
                ccat = ctc_logits.to(dev, non_blocking=True)
                ctcs = [ccat[offs[b]:offs[b + 1]] for b in range(n)]
        else:
            dev = self._device_for(ph_frame_logits[0])
            frames = [_as_2d(f).to(dev, non_blocking=True) for f in ph_frame_logits]
            edges = [_as_1d(e).to(dev, non_blocking=True) for e in ph_edge_logits]
            if ctc_logits is not None:
                if len(ctc_logits) != n:
                    raise ValueError("ctc_logits must hold one tensor per utterance")
                ctcs = [_as_2d(c).to(dev, non_blocking=True) for c in ctc_logits]
        # the reference applies .float() to both streams (ad:57,69): one element type per batch
        dt0 = frames[0].dtype if n else torch.float32
        if any(f.dtype != dt0 for f in frames) or dt0 not in ops.TORCH_TO_DTYPE:
            dt0 = torch.float32
        frames = [f if f.dtype == dt0 else f.to(dt0) for f in frames]
        edges = [e if e.dtype == dt0 else e.to(dt0) for e in edges]
        if wav_lengths is not None:
            for b in range(n):
                nf = self._num_frames(wav_lengths[b], frames[b].shape[0])
                frames[b], edges[b] = frames[b][:nf], edges[b][:nf]
                if ctc_logits is not None:                                       # ad:50
                    ctcs[b] = ctcs[b][:self._num_frames(wav_lengths[b], ctcs[b].shape[0])]
        if ctc_logits is None:
            ctcs = None
        elif n:
            # one element type and one width per batch; ctc() decodes the frames decode() aligns
            for b in range(n):
                if ctcs[b].shape[0] != frames[b].shape[0]:
                    raise ValueError(f"utterance {b}: {ctcs[b].shape[0]} frames of ctc logits, "
                                     f"{frames[b].shape[0]} of frame logits")
                if ctcs[b].shape[1] != ctcs[0].shape[1]:
                    raise ValueError("the ctc logits of a batch must share one width")
            ct = ctcs[0].dtype
            if any(c.dtype != ct for c in ctcs) or ct not in ops.TORCH_TO_DTYPE:
                ctcs = [c.float() for c in ctcs]
        if word_seqs is None:
            word_seqs = ph_seqs
            ph_idx_to_word_idxs = [np.arange(len(s)) for s in ph_seqs]
        is_sp = np.concatenate([np.fromiter((p == "SP" for p in s), dtype=bool, count=len(s))
                                for s in ph_seqs]) if n else np.zeros(0, bool)
        word_idx = np.concatenate([np.asarray(w, dtype=np.int64) for w in ph_idx_to_word_idxs]) \
            if n else np.zeros(0, np.int64)
        plan, views, out, _ = self._run(frames, edges, ids_list, want_frame_confidence, ctcs, want_frame_states)
        return BatchAlignment(plan, views, ph_seqs, word_seqs, ph_idx_to_word_idxs, is_sp, word_idx,
                              out["frame_conf"], out.get("ctc"), out.get("frame_state"),
                              list(zip(frames, edges, ids_list)) if ctcs is not None or want_frame_states else None)

    # ----------------------------------------------------------------------------------------
    # attributes the reference fills eagerly (ad:73-78,86) and only validation consumes: lazily here
    def _lazy_get(self, key, fn):
        if getattr(self, "_lazy", None) is None:
            return None
        if key not in self._lazy:
            self._lazy[key] = fn()
        return self._lazy[key]

    def __getattribute__(self, name):
        if name in ("ph_frame_pred", "ctc_logits", "edge_prob"):
            d = object.__getattribute__(self, "__dict__")
            if d.get("_lazy") is not None:
                if name == "ph_frame_pred":                                        # ad:56-59,73
                    return self._lazy_get(name, lambda: _ph_frame_pred(self._frame_logits, self.ph_seq_id,
                                                                       self.vocab["vocab_size"]))
                if name == "ctc_logits":                                           # ad:76-78
                    return self._lazy_get(name, lambda: None if self._ctc_src is None else
                                          self._ctc_src.float().squeeze(0).cpu().numpy().astype("float32"))
                if name == "edge_prob":                                            # ad:68-71,84
                    return self._lazy_get(name, lambda: _edge_prob(self._edge_logits))
        return object.__getattribute__(self, name)

    def ctc(self):
        src = getattr(self, "_ctc_src", None)
        if src is not None and src.is_cuda:            # same result, argmax + collapse on the device
            x = src.squeeze(0) if src.dim() == 3 else src
            return ops.ctc_greedy(x).cpu().numpy().astype(np.int64)
        ctc = np.argmax(self.ctc_logits, axis=-1)                                  # ad:145-150
        ctc_index = np.concatenate([[0], ctc])
        ctc_index = (ctc_index[1:] != ctc_index[:-1]) * ctc != 0
        ctc = ctc[ctc_index]
        return np.array([ph_id for ph_id in ctc if ph_id != 0])

    def plot(self, melspec):
        """ad:152-168.  Needs the reference's ``tools.plot.plot_for_valid`` (matplotlib) on the path."""
        from tools.plot import plot_for_valid  # provided by the reference checkout

        ph_idx_frame = np.zeros(self.ph_frame_pred.shape[0]).astype("int32")
        ph_intervals_pred_int = (self.ph_intervals_pred / self.frame_length).round().astype("int32")
        last_ph_idx = 0
        for ph_idx, ph_time in zip(self.ph_idx_seq, self.ph_time_int_pred):
            ph_idx_frame[ph_time] += ph_idx - last_ph_idx
            last_ph_idx = ph_idx
        ph_idx_frame = np.cumsum(ph_idx_frame)
        return plot_for_valid(melspec.cpu().numpy(), self.ph_pred_seq, ph_intervals_pred_int,
                              self.frame_confidence, self.ph_frame_pred[:, self.ph_seq_id], ph_idx_frame,
                              self.edge_prob)
