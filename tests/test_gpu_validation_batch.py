"""GPU: validation of a whole batch in one call -- the batched greedy CTC decode (hfa_ctc_greedy_batch) and the
per-frame path states (hfa_frame_states) behind decode_batch(..., ctc_logits=..., want_frame_states=True) and
BatchAlignment.ctc / ph_idx_frame / plot, against the reference goldens, numpy, the one-utterance kernel, and
the segments of the alignment itself."""
import sys
import types

import numpy as np
import pytest
import torch

from conftest import Golden
from hubertfa_b200 import _lib, ops, synth
from hubertfa_b200.alignment_decoder import AlignmentDecoder
from oracle import hfa_oracle_np as onp

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda")
C4_V = 74


# ---------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------
def _ctc_batch(views, S=None, ids=None, vocab=8):
    """ops.ctc_greedy_batch over per-utterance 2-D CUDA views (one width, one dtype) on a plan of their lengths.
    S / ids default to one SP state per utterance.  Returns (plan, per-utterance int32 ids, out_len)."""
    n = len(views)
    T = [int(v.shape[0]) for v in views]
    S = [1] * n if S is None else S
    ids = np.zeros(sum(max(s, 0) for s in S), np.int32) if ids is None else ids
    plan = ops.AlignPlan(T, S, ids, vocab, 0.02)
    ws = plan.new_workspace(DEV)
    plan.upload(ws)
    tab = torch.from_numpy(plan.ctc_table([v.data_ptr() for v in views], [v.stride(0) for v in views],
                                          [v.stride(1) for v in views])).to(DEV)
    nf = max(plan.total_frames, 1)
    scratch = torch.full((nf,), -7, dtype=torch.int32, device=DEV)
    out = torch.full((nf,), -7, dtype=torch.int32, device=DEV)
    n_len = torch.full((max(n, 1),), -7, dtype=torch.int32, device=DEV)
    ops.ctc_greedy_batch(ws, plan.handle, tab, int(views[0].shape[1]), ops.TORCH_TO_DTYPE[views[0].dtype],
                         scratch, out, n_len)
    torch.cuda.synchronize()
    out, n_len = out.cpu().numpy(), n_len.cpu().numpy()[:n]
    got = [out[plan.frame_off[b]:plan.frame_off[b] + n_len[b]] for b in range(n)]
    return plan, got, n_len


def _check_against_numpy_and_single(views, got):
    for b, v in enumerate(views):
        want = onp.ctc_greedy(v.float().cpu().numpy())
        assert np.array_equal(got[b], want), f"utterance {b}: batched ctc differs from numpy"
        assert np.array_equal(got[b], ops.ctc_greedy(v).cpu().numpy()), f"utterance {b}: differs from hfa_ctc_greedy"


def _coarse(T, V, seed, dtype=torch.float32):
    """Values on a grid of 0.5 in [-2, 2] (ties everywhere), every 7th row all -inf."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randint(-4, 5, (T, V), generator=g, device=DEV).float() * 0.5
    x[::7] = float("-inf")
    return x.to(dtype)


def _c4_batch(seed=synth.SEED0, V=C4_V, B=4096):
    """Seeded config-4 batch, logits drawn on the device: (T, S, ph_seqs, frame [sum T, V], edge [sum T],
    ctc [sum T, V])."""
    T, S = synth.sample_shapes(B, seed=seed)
    ids = synth.make_ids_batch(T, S, V, seed=seed)
    seqs = [["SP" if i == 0 else f"p{i}" for i in u] for u in ids]
    g = torch.Generator(device=DEV).manual_seed(seed)
    n = int(T.sum())
    frame = 3.0 * torch.randn(n, V, generator=g, device=DEV)
    edge = 2.0 * torch.randn(n, generator=g, device=DEV)
    ctc = torch.round(2.0 * torch.randn(n, V, generator=g, device=DEV)) * 0.5     # coarse: many ties
    return T, S, seqs, frame, edge, ctc


def _expected_states(res, b):
    idx, tim, _ = res.segments(b)
    T = int(res.frame_off[b + 1] - res.frame_off[b])
    return np.repeat(idx, np.diff(np.append(tim, T)))


class _PlotCapture:
    """tools.plot.plot_for_valid stand-in: records the seven arguments."""

    def __enter__(self):
        self.args = []
        fake = types.ModuleType("tools.plot")
        fake.plot_for_valid = lambda *a: self.args.append(a) or "figure"
        self.saved = {k: sys.modules.get(k) for k in ("tools", "tools.plot")}
        sys.modules["tools"] = types.ModuleType("tools")
        sys.modules["tools.plot"] = fake
        return self

    def __exit__(self, *exc):
        for k, v in self.saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def _same_plot_args(a, w):
    assert len(a) == len(w) == 7
    assert np.array_equal(a[0], w[0])
    assert list(a[1]) == list(w[1])
    assert np.array_equal(np.asarray(a[2]), np.asarray(w[2])) and np.asarray(a[2]).dtype == np.asarray(w[2]).dtype
    assert np.array_equal(a[3], w[3], equal_nan=True)
    assert a[4].shape == w[4].shape and a[4].dtype == w[4].dtype
    np.testing.assert_allclose(a[4], w[4], rtol=1e-6, atol=1e-12)
    assert np.array_equal(a[5], w[5]) and a[5].dtype == w[5].dtype
    assert a[6].dtype == w[6].dtype
    np.testing.assert_allclose(a[6], w[6], rtol=1e-6, atol=1e-12)


# ---------------------------------------------------------------------------------------------------------------
# 1. the reference goldens
# ---------------------------------------------------------------------------------------------------------------
def _golden_groups():
    g = Golden()
    groups = {}
    for m in g.meta:
        groups.setdefault((m["V"], m["hop"], m["sr"]), []).append(m["name"])
    return g, groups


def test_goldens_through_decode_batch():
    """The 18 reference cases, one decode_batch per vocabulary (and frame rate), ctc logits drawn again from each
    case's seed and trimmed by wav_length as decode() trims them: ctc ids, per-frame states and the plot()
    arguments equal the reference's / decode()'s."""
    golden, groups = _golden_groups()
    assert sum(len(v) for v in groups.values()) == len(golden.names)
    n_trimmed = 0
    for (V, hop, sr), names in groups.items():
        cases = [golden.case(nm) for nm in names]
        dec = AlignmentDecoder(synth.make_vocab(V), {"hop_length": hop, "sample_rate": sr})
        frames, edges, ctcs = [], [], []
        for c in cases:
            m = c["meta"]
            frame, edge, ctc = synth.make_logits(m["seed"], m["T"], V, c["ids"], m["planted"])
            assert np.array_equal(frame[0].numpy(), c["frame"])
            frames.append(frame.cuda())
            edges.append(edge.cuda())
            ctcs.append(ctc.cuda())
            n_trimmed += c["prob_log"].shape[0] < m["T"]
        meta = [c["meta"] for c in cases]
        res = dec.decode_batch(frames, edges, [m["ph_seq"] for m in meta], [m["word_seq"] for m in meta],
                               [m["ph_idx_to_word_idx"] for m in meta], wav_lengths=[m["wav_length"] for m in meta],
                               want_frame_confidence=True, ctc_logits=ctcs, want_frame_states=True)
        for b, c in enumerate(cases):
            m = c["meta"]
            assert np.array_equal(res.ctc(b), c["ctc_argmax"]) and res.ctc(b).dtype == np.int64, m["name"]
            assert np.array_equal(res.ph_idx_frame(b), c["plot_ph_idx_frame"]), m["name"]
            T_used = c["prob_log"].shape[0]
            mel = torch.arange(8 * T_used, dtype=torch.float32).reshape(1, 8, T_used)
            with _PlotCapture() as cap:
                assert res.plot(b, mel.cuda()) == "figure"
                dec.decode(frames[b], edges[b], ctcs[b], m["wav_length"], m["ph_seq"], m["word_seq"],
                           m["ph_idx_to_word_idx"])
                assert dec.plot(mel.cuda()) == "figure"
            _same_plot_args(cap.args[0], cap.args[1])
            assert np.array_equal(res.ctc(b), dec.ctc())
            assert np.array_equal(res.ph_frame_pred(b), dec.ph_frame_pred)
            assert np.array_equal(res.edge_prob(b), dec.edge_prob)
    assert n_trimmed >= 1, "no golden case is trimmed by wav_length"


# ---------------------------------------------------------------------------------------------------------------
# 2. ctc against numpy and the one-utterance kernel, bit for bit
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16], ids=["f32", "f16", "bf16"])
@pytest.mark.parametrize("layout", ["contiguous", "strided", "head-columns"])
def test_ctc_batch_matches_numpy(dtype, layout):
    V = 39
    Ts = [1, 2, 63, 64, 65, 128, 129, 500, 1031, 3000, 7]
    views = []
    for i, T in enumerate(Ts):
        x = _coarse(T, V, 100 + i) if i % 2 else torch.randn(T, V, device=DEV, generator=torch.Generator(
            device=DEV).manual_seed(100 + i))
        if layout == "contiguous":
            v = x.to(dtype)
        elif layout == "strided":                     # every other column of a wider tensor: stride_v = 2
            wide = torch.full((T, 3 + 2 * V), 9.0, device=DEV)
            wide[:, 3::2] = x
            v = wide.to(dtype)[:, 3::2]
        else:                                         # a [T, 2 + V + 5] head output, its ctc columns
            head = torch.randn(T, 2 + V + 5, device=DEV)
            head[:, 2:2 + V] = x
            v = head.to(dtype)[:, 2:2 + V]
        views.append(v)
    _, got, _ = _ctc_batch(views)
    _check_against_numpy_and_single(views, got)


@pytest.mark.parametrize("V", [1, 2, 31, 32, 33, 300])
def test_ctc_batch_widths_ties_and_inf_rows(V):
    views = [_coarse(T, V, 7 * V + T) for T in (1, 5, 64, 200, 777)]
    views.append(torch.full((70, V), float("-inf"), device=DEV))             # every row all -inf -> id 0
    _, got, n_len = _ctc_batch(views)
    _check_against_numpy_and_single(views, got)
    assert n_len[-1] == 0


def test_ctc_batch_skips_utterances_the_plan_did_not_accept():
    """EMPTY (T = 0) and BAD_ID utterances inside a batch: out_len 0 and no frames; decode_batch's ctc(b) raises
    for them like res[b] does, and every other utterance is decoded."""
    V = 20
    views = [_coarse(T, V, T) for T in (90, 0, 130, 40, 70)]
    S = [5, 3, 4, 6, 3]
    ids = np.concatenate([np.arange(5), np.arange(3), [1, 2, 3, 99], np.arange(6), np.arange(3)]).astype(np.int32)
    plan, got, n_len = _ctc_batch(views, S, ids, vocab=V)
    assert list(plan.T) == [90, 0, 130, 40, 70]
    assert n_len[1] == 0 and n_len[2] == 0
    for b in (0, 3, 4):
        assert np.array_equal(got[b], onp.ctc_greedy(views[b].cpu().numpy()))

    # through decode_batch (which refuses unknown phonemes itself): an utterance trimmed to T = 0 by its wav_length
    vocab = synth.make_vocab(V)
    Ts = [120, 80, 150]
    frames = [torch.randn(1, t, V, device=DEV) for t in Ts]
    edges = [torch.randn(1, t, device=DEV) for t in Ts]
    ctcs = [_coarse(t, V, 3 + t)[None] for t in Ts]
    seqs = [["SP", "p1", "p2", "SP"], ["p3", "p4"], ["SP", "p5", "p6", "p7", "SP"]]
    dec = AlignmentDecoder(vocab, synth.MELSPEC_50FPS)
    res = dec.decode_batch(frames, edges, seqs, wav_lengths=[None, -10.0, None], ctc_logits=ctcs,
                           want_frame_states=True)
    assert int(res.status[1]) == _lib.UTT_EMPTY and res.ctc_len[1] == 0
    for fn in (res.ctc, res.ph_idx_frame, res.__getitem__):
        with pytest.raises(ops.HfaError):
            fn(1)
    for b in (0, 2):
        assert np.array_equal(res.ctc(b), onp.ctc_greedy(ctcs[b][0].cpu().numpy()))
        assert np.array_equal(res.ph_idx_frame(b), _expected_states(res, b))


def test_ctc_packed_input_and_dtype_mix():
    """The packed [sum T, V] form with `lengths`, and a list whose dtypes differ (promoted to f32 like the frame
    logits): the same ids as the per-utterance list and as ctc() after decode()."""
    V = 63
    T, S = synth.sample_shapes(24, seed=11, min_s=1, max_s=6, s_lo=3, s_hi=60)
    vocab, items = synth.make_batch(T, S, V, seed=11, planted=True)
    dec = AlignmentDecoder(vocab, synth.MELSPEC_50FPS)
    seqs = [it["ph_seq"] for it in items]
    frames = [it["frame"].cuda() for it in items]
    edges = [it["edge"].cuda() for it in items]
    ctcs = [(_coarse(int(t), V, int(t)) if b % 3 == 0 else it["ctc"][0].cuda()) for b, (t, it) in
            enumerate(zip(T, items))]
    res = dec.decode_batch(frames, edges, seqs, ctc_logits=[c[None] for c in ctcs])
    packed = dec.decode_batch(torch.cat([f[0] for f in frames]), torch.cat([e[0] for e in edges]), seqs,
                              lengths=[int(t) for t in T], ctc_logits=torch.cat(ctcs))
    mixed = dec.decode_batch(frames, edges, seqs,
                             ctc_logits=[c.half()[None] if b % 2 else c[None] for b, c in enumerate(ctcs)])
    for b in range(len(items)):
        dec.decode(frames[b], edges[b], ctcs[b][None], None, seqs[b])
        want = dec.ctc()
        assert np.array_equal(want, onp.ctc_greedy(ctcs[b].cpu().numpy()))
        assert np.array_equal(res.ctc(b), want) and np.array_equal(packed.ctc(b), want)
        assert np.array_equal(mixed.ctc(b), onp.ctc_greedy(
            (ctcs[b].half() if b % 2 else ctcs[b]).float().cpu().numpy()))


def test_ctc_config4_batch():
    """4096 config-4 utterances (V = 74) in one launch: every utterance equals numpy and hfa_ctc_greedy."""
    T, S, seqs, frame, edge, ctc = _c4_batch()
    offs = np.concatenate([[0], np.cumsum(T)])
    views = [ctc[offs[b]:offs[b + 1]] for b in range(len(T))]
    _, got, _ = _ctc_batch(views)
    host = ctc.cpu().numpy()
    for b in range(len(T)):
        want = onp.ctc_greedy(host[offs[b]:offs[b + 1]])
        assert np.array_equal(got[b], want), b
        assert np.array_equal(got[b], ops.ctc_greedy(views[b]).cpu().numpy()), b


# ---------------------------------------------------------------------------------------------------------------
# 3. per-frame states
# ---------------------------------------------------------------------------------------------------------------
def test_frame_states_config4_and_config2():
    T, S, seqs, frame, edge, ctc = _c4_batch()
    dec = AlignmentDecoder(synth.make_vocab(C4_V), synth.MELSPEC_50FPS)
    res = dec.decode_batch(frame, edge, seqs, lengths=T, want_frame_states=True, ctc_logits=ctc)
    assert (res.status == _lib.UTT_OK).all()
    for b in range(len(T)):
        assert np.array_equal(res.ph_idx_frame(b), _expected_states(res, b)), b
    V = 63
    T2, S2 = synth.sample_shapes(256, seed=synth.SEED0)
    vocab, items = synth.make_batch(T2, S2, V, seed=synth.SEED0, planted=True)
    dec = AlignmentDecoder(vocab, synth.MELSPEC_50FPS)
    res = dec.decode_batch([it["frame"].cuda() for it in items], [it["edge"].cuda() for it in items],
                           [it["ph_seq"] for it in items], want_frame_states=True)
    assert res.ctc_ids is None
    for b in range(len(items)):
        assert np.array_equal(res.ph_idx_frame(b), _expected_states(res, b)), b
    with pytest.raises(ops.HfaError):
        res.ctc(0)


def test_frame_states_infeasible_utterance():
    V = 30
    vocab = synth.make_vocab(V)
    seqs = [[f"p{i}" for i in range(1, 11)], ["SP", "p1", "SP", "p2", "SP"]]
    Ts = [4, 60]                                      # ten phonemes without SP in 4 frames: no path
    frames = [torch.randn(1, t, V, device=DEV) for t in Ts]
    edges = [torch.randn(1, t, device=DEV) for t in Ts]
    dec = AlignmentDecoder(vocab, synth.MELSPEC_50FPS)
    res = dec.decode_batch(frames, edges, seqs, want_frame_states=True)
    assert int(res.status[0]) == _lib.UTT_INFEASIBLE and int(res.n_seg[0]) == 1
    assert np.array_equal(res.ph_idx_frame(0), np.full(4, res.segments(0)[0][0]))
    assert np.array_equal(res.ph_idx_frame(1), _expected_states(res, 1))


@pytest.mark.parametrize("bt_walk", ["0", None], ids=["tables", "default"])
def test_frame_states_giant_in_both_backtrace_routes(bt_walk, monkeypatch):
    """An S = 8200 giant (jump tables in both routes) next to small utterances (walked from shared memory by
    default, jump tables with HFA_BT_WALK=0)."""
    if bt_walk is None:
        monkeypatch.delenv("HFA_BT_WALK", raising=False)
    else:
        monkeypatch.setenv("HFA_BT_WALK", bt_walk)
    V = 63
    T = np.array([9000, 300, 500, 200], np.int32)
    S = np.array([8200, 40, 90, 30], np.int32)
    vocab, items = synth.make_batch(T, S, V, seed=8200, style="nosp", planted=True)
    dec = AlignmentDecoder(vocab, synth.MELSPEC_50FPS)
    res = dec.decode_batch([it["frame"].cuda() for it in items], [it["edge"].cuda() for it in items],
                           [it["ph_seq"] for it in items], want_frame_states=True,
                           ctc_logits=[it["ctc"].cuda() for it in items])
    plan = ops.AlignPlan(T, S, np.concatenate([it["ids"] for it in items]), V, dec.frame_length)
    walked = plan.routing()["bt_walk_utts"]
    assert walked == 0 if bt_walk == "0" else walked > 0
    for b, it in enumerate(items):
        assert int(res.status[b]) == _lib.UTT_OK
        assert np.array_equal(res.ph_idx_frame(b), _expected_states(res, b)), b
        assert np.array_equal(res.ctc(b), onp.ctc_greedy(it["ctc"][0].numpy())), b
    assert int(res.n_seg[0]) > 8192


# ---------------------------------------------------------------------------------------------------------------
# 4. one launch each, and nothing more without the new arguments
# ---------------------------------------------------------------------------------------------------------------
def test_launch_counts_do_not_grow_with_the_batch():
    deltas = {}
    for B in (24, 4096):
        T, S = synth.sample_shapes(B, seed=3)
        ids = np.concatenate(synth.make_ids_batch(T, S, C4_V, seed=3))
        plan = ops.AlignPlan(T, S, ids, C4_V, 0.02)
        ws, res = plan.new_workspace(DEV), plan.new_result(DEV)
        plan.upload(ws)
        n = int(T.sum())
        ctc = torch.randn(n, C4_V, device=DEV)
        offs = np.concatenate([[0], np.cumsum(T)])
        tab = torch.from_numpy(plan.ctc_table(ctc.data_ptr() + offs[:-1] * C4_V * 4, [C4_V] * B, [1] * B)).to(DEV)
        i32 = lambda k: torch.empty(k, dtype=torch.int32, device=DEV)
        res.zero_()
        c0 = ops.launch_count()
        ops.ctc_greedy_batch(ws, plan.handle, tab, C4_V, _lib.DTYPE_F32, i32(n), i32(n), i32(B))
        c1 = ops.launch_count()
        ops.frame_states(ws, plan.handle, res, i32(n))
        c2 = ops.launch_count()
        torch.cuda.synchronize()
        deltas[B] = (c1 - c0, c2 - c1)
    assert deltas[24] == deltas[4096] == (1, 1)


def test_decode_batch_launches_only_what_it_asks_for():
    V = 39
    T, S = synth.sample_shapes(24, seed=5, min_s=1, max_s=6, s_lo=3, s_hi=60)
    vocab, items = synth.make_batch(T, S, V, seed=5)
    dec = AlignmentDecoder(vocab, synth.MELSPEC_50FPS)
    args = ([it["frame"].cuda() for it in items], [it["edge"].cuda() for it in items], [it["ph_seq"] for it in items])
    ctcs = [it["ctc"].cuda() for it in items]
    dec.decode_batch(*args)                                          # warm-up
    # what hfa_align_batch launches for this batch on its own
    plan = ops.AlignPlan(T, S, np.concatenate([it["ids"] for it in items]), V, dec.frame_length)
    ws, res = plan.new_workspace(DEV), plan.new_result(DEV)
    plan.upload(ws)
    fr, ed = [f[0] for f in args[0]], [e[0] for e in args[1]]
    plan.set_inputs(ws, [f.data_ptr() for f in fr], [f.stride(0) for f in fr], [f.stride(1) for f in fr],
                    [e.data_ptr() for e in ed], [e.stride(0) for e in ed])
    c0 = ops.launch_count()
    ops.align_batch(ws, plan.handle, _lib.DTYPE_F32, res, None)
    align = ops.launch_count() - c0
    counts = {}
    for key, kw in (("plain", {}), ("ctc", dict(ctc_logits=ctcs)), ("states", dict(want_frame_states=True)),
                    ("both", dict(ctc_logits=ctcs, want_frame_states=True))):
        c0 = ops.launch_count()
        dec.decode_batch(*args, **kw)
        counts[key] = ops.launch_count() - c0
    assert counts == dict(plain=align, ctc=align + 1, states=align + 1, both=align + 2), (counts, align)


# ---------------------------------------------------------------------------------------------------------------
# 5. one CUDA graph: alignment, frame states and ctc
# ---------------------------------------------------------------------------------------------------------------
def test_graph_capture_with_device_tables():
    V = 63
    T, S = synth.sample_shapes(48, seed=21, min_s=1, max_s=8, s_lo=3, s_hi=150)
    vocab, items = synth.make_batch(T, S, V, seed=21, planted=True)
    _, items2 = synth.make_batch(T, S, V, seed=21, planted=False)          # same sequences, other logits
    B = len(items)
    plan = ops.AlignPlan(T, S, np.concatenate([it["ids"] for it in items]), V, 0.02)
    n = plan.total_frames

    def heads(its, ctc_sign):    # [T, 1 + V + V] per utterance: edge | frame logits | ctc logits
        return [torch.cat([it["edge"][0][:, None], it["frame"][0], ctc_sign * it["ctc"][0]], 1).to(DEV)
                for it in its]

    def tables(hs):
        W = 1 + 2 * V
        tab, stride = plan.input_table([h[:, 1:].data_ptr() for h in hs], [W] * B, [1] * B,
                                       [h[:, 0].data_ptr() for h in hs], [W] * B)
        ctab = plan.ctc_table([h[:, 1 + V:].data_ptr() for h in hs], [W] * B, [1] * B)
        return torch.from_numpy(tab.copy()).to(DEV), torch.from_numpy(ctab.copy()).to(DEV), stride

    i32 = lambda k: torch.empty(k, dtype=torch.int32, device=DEV)

    def run(ws, res, tab, ctab, stride, states, ids, lens, scratch):
        plan.set_inputs_device(ws, tab, stride)
        ops.align_batch(ws, plan.handle, _lib.DTYPE_F32, res, None)
        ops.frame_states(ws, plan.handle, res, states)
        ops.ctc_greedy_batch(ws, plan.handle, ctab, V, _lib.DTYPE_F32, scratch, ids, lens)

    def snapshot(res, states, ids, lens):
        torch.cuda.synchronize()
        lens_h, ids_h = lens.cpu().numpy(), ids.cpu().numpy()
        return (plan.views(res.cpu().numpy().copy()), states.cpu().numpy().copy(),
                [ids_h[plan.frame_off[b]:plan.frame_off[b] + lens_h[b]].copy() for b in range(B)])

    def eager(hs):
        ws, res = plan.new_workspace(DEV), plan.new_result(DEV)
        plan.upload(ws)
        bufs = (i32(n), i32(n), i32(B), i32(n))
        run(ws, res, *tables(hs), *bufs)
        return snapshot(res, *bufs[:3])

    h1, h2 = heads(items, 1.0), heads(items2, -1.0)     # make_batch draws the same ctc logits for both
    want1, want2 = eager(h1), eager(h2)
    assert any(not np.array_equal(a, b) for a, b in zip(want1[2], want2[2]))

    ws, res = plan.new_workspace(DEV), plan.new_result(DEV)
    plan.upload(ws)
    tab, ctab, stride = tables(h1)
    bufs = (i32(n), i32(n), i32(B), i32(n))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run(ws, res, tab, ctab, stride, *bufs)                     # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        run(ws, res, tab, ctab, stride, *bufs)

    def same(got, want):
        for key in ("status", "n_seg"):
            assert np.array_equal(got[0][key], want[0][key]), key
        for b in range(B):                            # slots past n_seg are never written
            o, k = int(plan.seg_off[b]), int(want[0]["n_seg"][b])
            for key in ("ph_idx_seq", "ph_time_int"):
                assert np.array_equal(got[0][key][o:o + k], want[0][key][o:o + k]), (b, key)
        assert np.array_equal(got[1], want[1])
        for a, b in zip(got[2], want[2]):
            assert np.array_equal(a, b)

    for b in bufs:
        b.fill_(-1)
    graph.replay()
    same(snapshot(res, *bufs[:3]), want1)
    t2, c2, _ = tables(h2)
    tab.copy_(t2)
    ctab.copy_(c2)
    graph.replay()
    same(snapshot(res, *bufs[:3]), want2)
