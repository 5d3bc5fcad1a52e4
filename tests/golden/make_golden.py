"""Generates tests/golden/reference_cases.npz by running the UNMODIFIED reference decoder
(tools/alignment_decoder.py of the reference tree, see oracle/reference_import.py; imported with a
matplotlib stub) on seeded synthetic logits.  Only runs where the reference tree exists:

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

Every case stores its inputs (so nothing depends on RNG reproducibility), the reference's values at
the `_decode` boundary (ph_prob_log gathered by ph_seq_id, in the compact form of
golden_format.pack_prob_log; edge_prob) and every output of `decode`.  The ctc logits are not stored: the
test of `ctc()` draws them again from the case's seed and first checks that the same draw reproduces
the stored frame and edge logits.
"""
import json
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from golden_format import pack_prob_log  # noqa: E402  (next to this script)
from hubertfa_b200 import synth  # noqa: E402
from oracle.reference_import import load_reference_decoder  # noqa: E402

# (name, T, S, V, style, planted, wav_length_frames or None, hop, sr)
CASES = [
    ("c1_T500_S40_V63", 500, 40, 63, "dictionary", False, None, 882, 44100),
    ("c1_planted", 500, 41, 63, "dictionary", True, None, 512, 44100),
    ("alt_T37_S7_V39", 37, 7, 39, "alternate", False, None, 512, 44100),
    ("short_T3_S7", 3, 7, 63, "alternate", False, None, 512, 44100),
    ("T1_S3", 1, 3, 63, "alternate", False, None, 512, 44100),
    ("T1_S3_trunc", 1, 3, 63, "dictionary", False, None, 512, 44100),
    ("S1_nonsp", 5, 1, 63, "nosp", False, None, 512, 44100),
    ("S1_sp", 5, 1, 63, "dictionary", False, None, 512, 44100),
    ("S2", 9, 2, 63, "dictionary", False, None, 512, 44100),
    ("nosp_T200_S33_V74", 200, 33, 74, "nosp", False, None, 512, 44100),
    ("infeasible_T2_S5", 2, 5, 63, "nosp", False, None, 512, 44100),
    ("T64_S64", 64, 64, 63, "alternate", False, None, 512, 44100),
    ("wavlen_trim", 300, 31, 63, "dictionary", True, 257, 512, 44100),
    ("k5_T700_S150", 700, 150, 63, "dictionary", True, None, 882, 44100),
    ("cta_T400_S300", 400, 300, 74, "alternate", False, None, 882, 44100),
    ("T17_S33", 17, 33, 39, "alternate", False, None, 512, 44100),
    ("T16_S32", 16, 32, 39, "alternate", True, None, 512, 44100),
    ("T33_S12", 33, 12, 39, "dictionary", True, None, 512, 44100),
]


def main():
    Ref = load_reference_decoder()
    if Ref is None:
        raise SystemExit("reference tree not available: cannot generate goldens")
    warnings.filterwarnings("ignore")
    out, meta = {}, []
    for ci, (name, T, S, V, style, planted, wav_frames, hop, sr) in enumerate(CASES):
        rng = np.random.default_rng(9000 + ci)
        vocab = synth.make_vocab(V)
        ph_seq, word_seq, ph2w = synth.make_ph_seq(rng, S, V, style)
        ids = np.array([vocab["vocab"][p] for p in ph_seq])
        frame, edge, ctc = synth.make_logits(9000 + ci, T, V, ids, planted)
        mel = {"hop_length": hop, "sample_rate": sr}
        wav_length = None if wav_frames is None else (wav_frames * hop + 0.25 * hop) / sr
        dec = Ref(vocab, mel)
        captured = {}
        orig = dec._decode

        def spy(ph_seq_id, ph_prob_log, edge_prob, _o=orig, _c=captured):
            _c["ph_prob_log"] = ph_prob_log.copy()
            _c["edge_prob"] = edge_prob.copy()
            return _o(ph_seq_id, ph_prob_log, edge_prob)

        dec._decode = spy
        r = dec.decode(frame, edge, ctc, wav_length, ph_seq, word_seq, ph2w)
        # validation-time consumers (forced_alignment.py:413-414): the seven arguments plot() hands to
        # tools.plot.plot_for_valid (ad:152-168), captured with a stand-in for the matplotlib function
        import tools.alignment_decoder as ref_mod
        import torch
        plot_args = {}

        def fake_plot(*a, _p=plot_args):
            _p["args"] = a
            return "figure"

        real_plot, ref_mod.plot_for_valid = ref_mod.plot_for_valid, fake_plot
        try:
            n_fr = dec.ph_frame_pred.shape[0]
            assert dec.plot(torch.zeros(1, 8, n_fr)) == "figure"
        finally:
            ref_mod.plot_for_valid = real_plot
        pre = f"{name}/"
        out[pre + "frame"] = frame[0].numpy()
        out[pre + "edge"] = edge[0].numpy()
        out[pre + "ctc_argmax"] = dec.ctc().astype(np.int64)
        out[pre + "ids"] = ids.astype(np.int32)
        packed = pack_prob_log(frame[0].numpy(), captured["ph_prob_log"][:, ids], ids)      # ad:239
        out.update({pre + k: v for k, v in packed.items()})
        out[pre + "edge_prob"] = captured["edge_prob"]
        out[pre + "ph_seq_pred"] = np.asarray(r[0]).astype("U")
        out[pre + "ph_intervals_pred"] = np.asarray(r[1], dtype=np.float64)
        out[pre + "word_seq_pred"] = np.asarray(r[2]).astype("U")
        out[pre + "word_intervals_pred"] = np.asarray(r[3], dtype=np.float64)
        out[pre + "total_confidence"] = np.asarray(r[4], dtype=np.float32)
        out[pre + "ph_idx_seq"] = dec.ph_idx_seq.astype(np.int64)
        out[pre + "ph_time_int"] = dec.ph_time_int_pred.astype(np.int64)
        out[pre + "frame_confidence"] = dec.frame_confidence.astype(np.float32)
        if T <= 64 or name in ("c1_planted", "wavlen_trim"):      # [T, V] f32: kept for the small cases only
            out[pre + "ph_frame_pred"] = dec.ph_frame_pred.astype(np.float32)     # ad:56-59,73
        a = plot_args["args"]
        out[pre + "plot_ph_seq"] = np.asarray(a[1]).astype("U")
        out[pre + "plot_ph_intervals_int"] = np.asarray(a[2]).astype(np.int32)
        out[pre + "plot_ph_idx_frame"] = np.asarray(a[5]).astype(np.int64)
        out[pre + "plot_ph_frame_prob_sum"] = np.asarray(a[4], dtype=np.float64).sum(axis=0)   # [S]: a digest of [T, S]
        meta.append(dict(name=name, seed=9000 + ci, T=T, S=S, V=V, style=style, planted=planted, hop=hop, sr=sr,
                         wav_length=wav_length, ph_seq=ph_seq, word_seq=word_seq,
                         ph_idx_to_word_idx=[int(x) for x in ph2w]))
        print(name, "segments", len(dec.ph_idx_seq), "conf", float(r[4]))
    out["meta_json"] = np.array(json.dumps(meta))
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_cases.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
