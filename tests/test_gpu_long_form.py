"""GPU: long-form utterances, S > 8192 phoneme states (the skewed strips, or the halo bands without tensor maps).

Tier 1 is the C oracle DP run on OUR emissions, through the low-memory oracle (oracle/lowmem_oracle.py, pinned
bit for bit against the full one in tests/test_long_form_host.py) wherever the [T][S] matrices would be large."""
import numpy as np
import pytest
import torch

from gpu_util import bits, check_core_against_oracle, run_core_gpu, synth_core_inputs
from hubertfa_b200 import ops, synth
from hubertfa_b200.alignment_decoder import AlignmentDecoder
from oracle import c_oracle as oc
from oracle import hfa_oracle_np as onp
from oracle import lowmem_oracle as lo
from test_gpu_full_size import emissions_of, planted_head

pytestmark = pytest.mark.gpu


def tier1(ids, e, el, ne):
    """lowmem oracle on our dense emissions [T, S] (host)."""
    return lo.decode(ids, e, el, ne, chunk=2048)


@pytest.mark.parametrize("S", [8193, 16_000])
def test_long_form_from_logits_through_decode(S):
    """decode() from planted [1, T, V] logits, T = 4 S: the protocol of test_config3_from_logits_through_decode."""
    V, T = 63, 4 * S
    rng = np.random.default_rng(S)
    vocab = synth.make_vocab(V)
    ph_seq, word_seq, ph2w = synth.make_ph_seq(rng, S, V, "dictionary")
    ids = np.array([vocab["vocab"][p] for p in ph_seq], dtype=np.int32)
    head = planted_head([T], [ids], V, seed=S + 1)
    head_dev = head.cuda()
    dec = AlignmentDecoder(vocab, synth.MELSPEC_50FPS)
    rt = ops.AlignPlan([T], [S], ids, V, dec.frame_length).routing()
    assert rt["cta_utts"] == 0 and rt["big_band_k"] == 1 and rt["skew_d"] > 0 and rt["keeps_dp"], rt
    ctc = torch.zeros(1, 16, V, device="cuda")
    out = dec.decode(head_dev[None, :, 2:], head_dev[None, :, 0], ctc, None, ph_seq, word_seq, ph2w)
    # tier 1: the oracle DP on our emissions
    (e, el, ne), = emissions_of(dec, [head_dev[:, 2:]], [head_dev[:, 0]], [ids], V)
    r = tier1(ids, e, el, ne)
    assert r["rc"] == 0
    assert np.array_equal(dec.ph_idx_seq, r["ph_idx_seq"]) and np.array_equal(dec.ph_time_int_pred, r["ph_time_int"])
    assert bits(dec.final_score) == bits(r["final_score"])
    fc, tot = oc.confidence(r["dp_path"])
    np.testing.assert_allclose(dec.frame_confidence, fc, rtol=2e-6, atol=1e-30)
    np.testing.assert_allclose(out[4], tot, rtol=1e-4)
    # tier 2: the reference's own arithmetic (torch softmax on the CPU, numpy) from the logits
    want, ex = onp.decode(vocab, synth.MELSPEC_50FPS, head[None, :, 2:], head[None, :, 0], None, None,
                          ph_seq, word_seq, ph2w, full=True)
    assert np.array_equal(dec.ph_idx_seq, ex["ph_idx_seq"]) and np.array_equal(dec.ph_time_int_pred, ex["ph_time_int"])
    assert list(out[0]) == list(want[0]) and list(out[2]) == list(want[2])
    np.testing.assert_allclose(out[1], want[1], rtol=0, atol=1e-7)
    np.testing.assert_allclose(out[3], want[3], rtol=0, atol=1e-7)


MODES = {
    "strips-D2": dict(HFA_SKEW_D="2"),
    "strips-D3": dict(HFA_SKEW_D="3"),
    "halo-bands": dict(HFA_LAT_KERNEL="band"),
    "no-tensormap": dict(HFA_NO_TENSORMAP="1"),
    "no-kept-dp": dict(HFA_KEEP_DP="0"),
}


@pytest.mark.parametrize("mode", list(MODES))
def test_giant_at_the_decode_boundary(mode, monkeypatch):
    """One S = 8200 utterance, T = 3 S, through every forward route it can take: dp, backpointers of the dump and
    of the production instantiation, kept dp (where kept), path, dp_path and confidences, bit for bit."""
    for k, v in MODES[mode].items():
        monkeypatch.setenv(k, v)
    S, T, V = 8200, 24_600, 63
    d = synth_core_inputs(T, S, V, seed=8200, planted=True)
    plan = ops.AlignPlan([T], [S], d["ids"], V, 0.02)
    rt = plan.routing()
    assert rt["cta_utts"] == 0 and rt["warp_utts"] == 0 and rt["keeps_dp"] == (mode != "no-kept-dp"), rt
    assert rt["big_band_k"] == (1 if mode in ("strips-D2", "strips-D3", "no-kept-dp") else 2), rt
    if mode == "strips-D3":
        assert rt["skew_d"] == 3
    g, = run_core_gpu([d["ids"]], [d["prob_log"]], [d["el"]], [d["ne"]], [d["p"]], vocab=V)
    assert ("dp_kept" in g) == (mode != "no-kept-dp")
    check_core_against_oracle(d["ids"], d["prob_log"], d["el"], d["ne"], g, p=d["p"], full=True)


def test_config4_batch_with_two_giants():
    """decode_batch of the 4096 config-4 utterances plus two giants: the giants pass tier 1, and every other
    utterance's results are bit-identical to a decode_batch of the 4096 alone."""
    V, B = 63, 4096
    T, S = synth.sample_shapes(B, seed=synth.SEED0 + V)
    ids_list = list(synth.make_ids_batch(T, S, V, seed=synth.SEED0 + V))
    giants = [(36_000, 9_000), (48_000, 12_000)]
    g_ids = list(synth.make_ids_batch([t for t, _ in giants], [s for _, s in giants], V, seed=77))
    T2 = np.concatenate([T, [t for t, _ in giants]]).astype(np.int64)
    S2 = np.concatenate([S, [s for _, s in giants]]).astype(np.int64)
    ids2 = ids_list + g_ids
    head = planted_head(T2, ids2, V, seed=4242)
    head_dev = head.cuda()
    row_off = np.concatenate([[0], np.cumsum(T2)])
    vocab = synth.make_vocab(V)
    dec = AlignmentDecoder(vocab, synth.MELSPEC_50FPS)
    names = np.array(["SP"] + [f"p{i}" for i in range(1, V)])
    frames = [head_dev[row_off[i]:row_off[i + 1], 2:] for i in range(len(T2))]
    edges = [head_dev[row_off[i]:row_off[i + 1], 0] for i in range(len(T2))]
    seqs = [list(names[i]) for i in ids2]
    rt = ops.AlignPlan(T2, S2, np.concatenate(ids2), V, dec.frame_length).routing()
    assert rt["warp_utts"] == B and rt["cta_utts"] == 0 and rt["big_band_k"] == 1 and rt["keeps_dp"], rt
    both = dec.decode_batch(frames, edges, seqs)
    alone = dec.decode_batch(frames[:B], edges[:B], seqs[:B])
    assert (both.status == 0).all() and (alone.status == 0).all()
    for k in ("status", "n_seg", "end_state"):
        assert np.array_equal(getattr(both, k)[:B], getattr(alone, k)), k
    for k in ("final_score", "total_confidence"):
        assert np.array_equal(bits(getattr(both, k)[:B]), bits(getattr(alone, k))), k
    for b in range(B):                            # the written entries: n_seg of the S slots of each utterance
        o, k = int(alone.seg_off[b]), int(alone.n_seg[b])
        assert np.array_equal(both.ph_idx_seq[o:o + k], alone.ph_idx_seq[o:o + k]), b
        assert np.array_equal(both.ph_time_int[o:o + k], alone.ph_time_int[o:o + k]), b
        assert np.array_equal(both.raw_intervals[o:o + k].view(np.uint64), alone.raw_intervals[o:o + k].view(np.uint64)), b
    for j, b in enumerate(range(B, B + len(giants))):
        (e, el, ne), = emissions_of(dec, [frames[b]], [edges[b]], [ids2[b]], V)
        r = tier1(ids2[b], e, el, ne)
        idx, tim, _ = both.segments(b)
        assert np.array_equal(idx, r["ph_idx_seq"]) and np.array_equal(tim, r["ph_time_int"]), f"giant {j}"
        assert both.end_state[b] == r["end_state"] and bits(both.final_score[b]) == bits(r["final_score"])
        _, tot = oc.confidence(r["dp_path"])
        np.testing.assert_allclose(both.total_confidence[b], tot, rtol=1e-4)


def seeded_rows(xp, t0, t1, S, T):
    """Emissions of frames t0 .. t1-1, [t1 - t0, S] f32, from integer hashes: the same bits from numpy on the
    host and torch on the device.  Values are multiples of 2^-9 in [-16, 0], near 0 on a diagonal band."""
    if xp is np:
        t = np.arange(t0, t1, dtype=np.int64)[:, None]
        s = np.arange(S, dtype=np.int64)[None, :]
    else:
        t = torch.arange(t0, t1, dtype=torch.int64, device="cuda")[:, None]
        s = torch.arange(S, dtype=torch.int64, device="cuda")[None, :]
    h = (t * 1103515245 + s * 12345 + 17) % 2147483647
    h = (h * 48271) % 2147483647
    diag = (s == (t * S) // T) | (s == (t * S) // T + 1)
    v = xp.where(diag, h % 64, h % 8192)
    return (-v).to(torch.float32) / 512.0 if xp is torch else (-v).astype(np.float32) / np.float32(512.0)


def seeded_edges(T):
    t = np.arange(T, dtype=np.int64)
    h = ((t * 69069 + 1) % 2147483647 * 48271) % 2147483647
    el = (-(h % 4096)).astype(np.float32) / np.float32(256.0)
    ne = (-((h >> 12) % 256)).astype(np.float32) / np.float32(1024.0)
    return el, ne


def test_beyond_2_pow_31_cells():
    """S = 8200, T = 262 000: 2.15e9 DP cells, 8.6 GB of emissions, at the _decode boundary through
    hfa_pack_emissions.  The low-memory oracle regenerates the same seeded rows on the host."""
    S, T, V = 8200, 262_000, 63
    assert T * S > 2 ** 31
    rng = np.random.default_rng(31)
    ids = rng.integers(1, V, size=S).astype(np.int32)
    ids[rng.random(S) < 0.3] = 0
    plan = ops.AlignPlan([T], [S], ids, V, 0.02)
    rt = plan.routing()
    assert rt["big_band_k"] == 1 and rt["cta_utts"] == 0 and rt["keeps_dp"], rt
    need = plan.workspace_bytes + T * S * 4 + plan.result_bytes + 5 * T * 4
    free, total = torch.cuda.mem_get_info()
    print(f"T*S = {T * S} cells; device memory needed {need / 2**30:.2f} GiB "
          f"(workspace {plan.workspace_bytes / 2**30:.2f} GiB + dense emissions {T * S * 4 / 2**30:.2f} GiB), "
          f"free {free / 2**30:.2f} of {total / 2**30:.2f} GiB")
    if free < need + (1 << 30):
        pytest.skip(f"needs {need} bytes of device memory (+1 GiB headroom), {free} free")
    dev = torch.device("cuda")
    ws = torch.empty(plan.workspace_bytes, dtype=torch.uint8, device=dev)
    plan.upload(ws)
    el, ne = seeded_edges(T)
    pl = torch.empty(T * S, dtype=torch.float32, device=dev)
    step = 8192
    for t0 in range(0, T, step):
        t1 = min(T, t0 + step)
        pl[t0 * S:t1 * S] = seeded_rows(torch, t0, t1, S, T).reshape(-1)
    ops.pack_emissions(ws, plan.handle, pl, torch.from_numpy(el).to(dev), torch.from_numpy(ne).to(dev), None)
    del pl
    ops.viterbi_forward(ws, plan.handle, None)
    res = torch.empty(plan.result_bytes, dtype=torch.uint8, device=dev)
    fc = torch.empty(T, dtype=torch.float32, device=dev)
    dpp = torch.empty(T, dtype=torch.float32, device=dev)
    ops.backtrace(ws, plan.handle, res, fc, dpp)
    torch.cuda.synchronize()
    v = plan.views(res.cpu().numpy())
    del ws
    r = lo.decode_rows(ids, T, lambda a, b: seeded_rows(np, a, b, S, T), el, ne, chunk=2048, want_dp_path=False)
    assert r["rc"] == 0
    k = int(v["n_seg"][0])
    assert int(v["status"][0]) == 0 and k == len(r["ph_idx_seq"]) > S // 2
    assert np.array_equal(v["ph_idx_seq"][:k], r["ph_idx_seq"]) and np.array_equal(v["ph_time_int"][:k], r["ph_time_int"])
    assert int(v["end_state"][0]) == r["end_state"]
    assert bits(v["final_score"][0]) == bits(r["final_score"])
    assert bits(dpp[-1].cpu().numpy()) == bits(r["final_score"])
    print(f"beyond 2^31 cells: {k} segments, end state {r['end_state']}, final score {r['final_score']!r}: "
          f"bit-identical to the low-memory oracle")
