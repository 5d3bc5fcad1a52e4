"""CPU: both oracles reproduce the reference outputs stored in tests/golden (and the live reference
where its tree is provided, see oracle/reference_import.py).  This is what pins the oracle; the GPU
tests then compare the CUDA path with the oracle."""
import numpy as np
import pytest
import torch

from conftest import golden_names
from hubertfa_b200 import synth
from oracle import c_oracle as oc
from oracle import hfa_oracle_np as onp
from oracle.reference_import import load_reference_decoder


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.mark.parametrize("name", golden_names())
def test_numpy_oracle_matches_golden_decode(golden, name):
    c = golden.case(name)
    m = c["meta"]
    vocab = synth.make_vocab(m["V"])
    mel = {"hop_length": m["hop"], "sample_rate": m["sr"]}
    frame = torch.from_numpy(c["frame"])[None]
    edge = torch.from_numpy(c["edge"])[None]
    out, ex = onp.decode(vocab, mel, frame, edge, None, m["wav_length"], m["ph_seq"], m["word_seq"],
                         m["ph_idx_to_word_idx"], full=True)
    assert list(out[0]) == list(c["ph_seq_pred"])
    assert np.array_equal(np.asarray(out[1], dtype=np.float64).reshape(c["ph_intervals_pred"].shape),
                          c["ph_intervals_pred"])
    assert list(out[2]) == list(c["word_seq_pred"])
    assert np.array_equal(np.asarray(out[3], dtype=np.float64).reshape(c["word_intervals_pred"].shape),
                          c["word_intervals_pred"])
    assert np.array_equal(np.float32(out[4]), c["total_confidence"], equal_nan=True)
    assert np.array_equal(ex["ph_idx_seq"], c["ph_idx_seq"])
    assert np.array_equal(ex["ph_time_int"], c["ph_time_int"])
    assert np.array_equal(_bits(ex["frame_confidence"]), _bits(c["frame_confidence"]))
    assert np.array_equal(_bits(ex["prob_log"]), _bits(c["prob_log"]))
    assert np.array_equal(ex["edge_prob"], c["edge_prob"])


@pytest.mark.parametrize("name", golden_names())
def test_c_oracle_matches_golden_at_decode_core(golden, name):
    """`_decode` boundary: identical emissions in -> identical path, bit-identical scores."""
    c = golden.case(name)
    el, ne = oc.edge_logs(c["edge_prob"])
    eln, nen = onp.edge_logs(c["edge_prob"])
    assert np.array_equal(_bits(el), _bits(eln)) and np.array_equal(_bits(ne), _bits(nen))
    r = oc.decode(c["ids"], c["prob_log"], el, ne, full=True)
    assert r["rc"] == 0
    assert np.array_equal(r["ph_idx_seq"], c["ph_idx_seq"])
    assert np.array_equal(r["ph_time_int"], c["ph_time_int"])
    dp, bt, _ = onp.forward_dp(c["ids"], c["prob_log"], el, ne)
    assert np.array_equal(_bits(r["dp"]), _bits(dp))
    assert np.array_equal(r["bt"], bt)
    fc, tot = oc.confidence(r["dp_path"])
    ok = np.isfinite(c["frame_confidence"])
    np.testing.assert_allclose(fc[ok], c["frame_confidence"][ok], rtol=2e-6, atol=0)
    if np.isfinite(c["total_confidence"]):
        np.testing.assert_allclose(tot, c["total_confidence"], rtol=1e-5)
    # O(T) path-only rescoring (what the CUDA finalize kernel does) reproduces dp on the path
    rs = onp.path_rescore(c["ids"], c["prob_log"], el, ne, r["ph_idx_seq"], r["ph_time_int"])
    assert np.array_equal(_bits(rs), _bits(r["dp_path"]))


@pytest.mark.parametrize("name", golden_names())
def test_c_oracle_front_end_close_to_torch(golden, name):
    """Emission / edge stages replace torch's exp/log by libm: compare with a tolerance."""
    c = golden.case(name)
    m = c["meta"]
    T = c["prob_log"].shape[0]
    e = oc.emission(c["frame"][:T], c["ids"])
    np.testing.assert_allclose(e, c["prob_log"], rtol=0, atol=4e-6)
    p = oc.edge_pred(c["edge"][:T])
    ed, ep = oc.edge_prob(p)
    np.testing.assert_allclose(ep, c["edge_prob"], rtol=0, atol=5e-7)
    # intervals from the golden path with the oracle's own edge_pred: bit-equal when p is bit-equal
    pt = onp.edge_pred(torch.from_numpy(c["edge"][:T])[None])
    iv = oc.intervals(T, c["ph_time_int"], pt, m["hop"] / m["sr"])
    edt, _ = onp.edge_streams(pt)
    assert np.array_equal(iv, onp.intervals_from_path(c["ph_time_int"], edt, T, m["hop"] / m["sr"]))


def test_c_oracle_batch_driver_matches_single(golden):
    names = ["c1_T500_S40_V63", "c1_planted", "short_T3_S7", "S2"]
    cs = [golden.case(n) for n in names]
    T = [c["frame"].shape[0] for c in cs]
    S = [len(c["ids"]) for c in cs]
    out = oc.align_batch(T, S, 63, np.concatenate([c["frame"].reshape(-1) for c in cs]),
                         np.concatenate([c["edge"] for c in cs]), np.concatenate([c["ids"] for c in cs]),
                         512 / 44100, n_threads=2)
    assert out["bad"] == 0
    for b, c in enumerate(cs):
        o, k = int(out["seg_off"][b]), int(out["n_seg"][b])
        e = oc.emission(c["frame"], c["ids"])
        p = oc.edge_pred(c["edge"])
        _, ep = oc.edge_prob(p)
        el, ne = oc.edge_logs(ep)
        r = oc.decode(c["ids"], e, el, ne)
        assert np.array_equal(out["ph_idx_seq"][o:o + k], r["ph_idx_seq"])
        assert np.array_equal(out["ph_time_int"][o:o + k], r["ph_time_int"])


@pytest.mark.parametrize("name", golden_names())
def test_ctc_greedy_matches_golden(golden, name):
    """The reference's greedy CTC decode (ad:145-150) of its ctc logits, trimmed to the frames it aligned.
    The logits are drawn again from the case's seed; the same draw must reproduce the stored inputs."""
    c = golden.case(name)
    m = c["meta"]
    frame, edge, ctc = synth.make_logits(m["seed"], m["T"], m["V"], c["ids"], m["planted"])
    assert np.array_equal(_bits(frame[0].numpy()), _bits(c["frame"]))
    assert np.array_equal(_bits(edge[0].numpy()), _bits(c["edge"]))
    T = c["prob_log"].shape[0]
    assert np.array_equal(onp.ctc_greedy(ctc[0, :T].numpy()), c["ctc_argmax"])


@pytest.mark.skipif(load_reference_decoder() is None, reason="reference tree not present")
def test_oracles_match_live_reference_on_random_shapes():
    import warnings
    warnings.filterwarnings("ignore")
    Ref = load_reference_decoder()
    mel = {"hop_length": 512, "sample_rate": 44100}
    T, S = synth.sample_shapes(12, seed=77, min_s=1, max_s=8)
    for i, (t, s) in enumerate(zip(T, S)):
        rng = np.random.default_rng(500 + i)
        V = [63, 39, 74][i % 3]
        vocab = synth.make_vocab(V)
        ph_seq, word_seq, ph2w = synth.make_ph_seq(rng, int(s), V, ["dictionary", "alternate", "nosp"][i % 3])
        ids = np.array([vocab["vocab"][p] for p in ph_seq])
        frame, edge, ctc = synth.make_logits(500 + i, int(t), V, ids, planted=bool(i & 1))
        ref = Ref(vocab, mel)
        r = ref.decode(frame, edge, ctc, None, ph_seq, word_seq, ph2w)
        o, ex = onp.decode(vocab, mel, frame, edge, ctc, None, ph_seq, word_seq, ph2w, full=True)
        for a, b in zip(r, o):
            a, b = np.asarray(a), np.asarray(b)
            assert a.shape == b.shape
            assert np.array_equal(a, b, equal_nan=True) if a.dtype.kind == "f" else np.array_equal(a, b)
        assert np.array_equal(ref.ph_idx_seq, ex["ph_idx_seq"])
        c = oc.decode(ids, ex["prob_log"], ex["edge_log"], ex["not_edge_log"], full=True)
        assert np.array_equal(c["ph_idx_seq"], ref.ph_idx_seq)
        assert np.array_equal(c["ph_time_int"], ref.ph_time_int_pred)
        assert np.array_equal(_bits(c["dp"]), _bits(ex["dp"]))
        assert np.array_equal(onp.ctc_greedy(ref.ctc_logits), ref.ctc())
