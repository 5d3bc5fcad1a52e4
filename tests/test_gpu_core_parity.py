"""GPU, tier 1: identical emissions in -> bit-identical DP cells, backpointers, paths and path
scores out, against the C oracle and the reference's golden outputs (SURVEY.md 8c)."""
import numpy as np
import pytest

from conftest import golden_names
from gpu_util import bits, check_core_against_oracle, pairable_ids, run_core_gpu, synth_core_inputs
from oracle import c_oracle as oc
from oracle import hfa_oracle_np as onp

pytestmark = pytest.mark.gpu


@pytest.fixture(params=["0", "0p2", "0p0", "2k4", "2k8", "2nk", "2rc", "2s2", "2s3", "2s2slow", "2s2nk", "auto"],
                ids=["warp-per-utterance", "warp-pair-layout-forced", "warp-plain-layout-only", "banded-k2-k4", "banded-k2-k8",
                     "banded-no-dp-store", "banded-row-copies", "skew-d2", "skew-d3", "skew-d2-guarded-body",
                     "skew-d2-no-dp-store", "auto"])
def routing(request, monkeypatch):
    """HFA_LATENCY_MODE: 0 = every S <= 256 utterance in the warp kernel (all 8 state classes) and
    S > 256 in the CTA kernel -- the SP-aware pair layout where the plan's cost rule picks it, wherever it is
    possible (HFA_PAIR=2) or nowhere (HFA_PAIR=0);
    2 = everything in the banded (halo) kernel, S > 256 with 4 / 8 states per lane, the backtrace
    reading the dp the forward pass kept -- or (no-dp-store) re-scoring the path, or (row-copies)
    without the TMA tensor maps; skew-* = everything (S > 256 included) in the skewed-wavefront kernel
    with 2 / 3 frames of skew per state, through its unrolled steady-state body or (guarded-body) only
    the guarded one; auto = the plan's own choice (the skewed kernel for these small batches)."""
    if request.param != "auto":
        monkeypatch.setenv("HFA_LATENCY_MODE", request.param[0])
        monkeypatch.setenv("HFA_BIG_KERNEL", "band" if request.param[0] == "2" else "cta")
        monkeypatch.setenv("HFA_LAT_KERNEL", "skew" if request.param.startswith("2s") else "band")
    if request.param in ("0p2", "0p0"):
        monkeypatch.setenv("HFA_PAIR", request.param[2])
    if request.param in ("2k4", "2k8"):
        monkeypatch.setenv("HFA_BIG_K", request.param[2])
    if request.param.startswith("2s"):
        monkeypatch.setenv("HFA_SKEW_D", request.param[2])
    if request.param == "2s2slow":
        monkeypatch.setenv("HFA_SKEW_SLOW", "1")
    if request.param in ("2nk", "2s2nk"):
        monkeypatch.setenv("HFA_KEEP_DP", "0")
    if request.param == "2rc":                     # 1-D row copies instead of the TMA tensor-tile loads
        monkeypatch.setenv("HFA_NO_TENSORMAP", "1")
    return request.param


def test_golden_cases_one_batch(golden, routing):
    """All golden cases in ONE ragged batch: every state class incl. the CTA kernel, T=1, S=1,
    infeasible alignments.  Paths must equal the reference's, scores the oracle's bit for bit."""
    import torch
    cs = [golden.case(n) for n in golden.names]
    els, nes, ps = [], [], []
    for c in cs:
        el, ne = oc.edge_logs(c["edge_prob"])
        els.append(el)
        nes.append(ne)
        T = c["prob_log"].shape[0]
        ps.append(onp.edge_pred(torch.from_numpy(c["edge"][:T])[None]))
    fl = 512 / 44100
    out = run_core_gpu([c["ids"] for c in cs], [c["prob_log"] for c in cs], els, nes, ps, fl)
    for c, g, el, ne, p in zip(cs, out, els, nes, ps):
        assert np.array_equal(g["ph_idx_seq"], c["ph_idx_seq"]), c["meta"]["name"]
        assert np.array_equal(g["ph_time_int"], c["ph_time_int"]), c["meta"]["name"]
        check_core_against_oracle(c["ids"], c["prob_log"], el, ne, g, p, fl)
        fin = np.isfinite(c["frame_confidence"])
        np.testing.assert_allclose(g["frame_conf"][fin], c["frame_confidence"][fin], rtol=3e-6)


SHAPES = [  # (T, S, style) -- every K class of the warp kernel, tile-boundary T, the CTA kernel
    (1, 1, "dictionary"), (2, 2, "dictionary"), (15, 5, "alternate"), (16, 9, "alternate"),
    (17, 12, "dictionary"), (31, 31, "alternate"), (32, 32, "alternate"), (33, 33, "alternate"),
    (100, 20, "dictionary"), (257, 64, "dictionary"), (300, 65, "dictionary"), (480, 96, "nosp"),
    (333, 97, "dictionary"), (500, 128, "dictionary"), (512, 129, "dictionary"), (700, 160, "dictionary"),
    (640, 161, "dictionary"), (650, 192, "dictionary"), (600, 200, "alternate"), (800, 224, "dictionary"),
    (801, 225, "dictionary"), (900, 256, "dictionary"), (600, 257, "alternate"), (700, 300, "alternate"),
    (1000, 513, "alternate"), (1300, 1030, "alternate"), (40, 7, "nosp"), (3, 7, "alternate"), (2, 5, "nosp"),
]


def test_random_shapes_all_classes(routing):
    ins = [synth_core_inputs(T, S, 63, 4000 + i, style, planted=bool(i % 2))
           for i, (T, S, style) in enumerate(SHAPES)]
    out = run_core_gpu([x["ids"] for x in ins], [x["prob_log"] for x in ins], [x["el"] for x in ins],
                       [x["ne"] for x in ins], [x["p"] for x in ins], 0.02)
    for x, g, shp in zip(ins, out, SHAPES):
        try:
            check_core_against_oracle(x["ids"], x["prob_log"], x["el"], x["ne"], g, x["p"], 0.02)
        except AssertionError as e:
            raise AssertionError(f"shape {shp}: {e}") from e


def test_cta_per_utterance_kernel(monkeypatch):
    """S > 256 in a batch that is never cut into strips: the CTA-per-utterance kernel (8 states per thread, one
    barrier per frame), 256 / 512 / 1024 threads."""
    monkeypatch.setenv("HFA_LATENCY_MODE", "0")
    monkeypatch.setenv("HFA_BIG_KERNEL", "cta")
    shapes = [(600, 257, "alternate"), (700, 300, "alternate"), (1000, 513, "alternate"),
              (1300, 1030, "alternate"), (50, 2100, "dictionary"), (1, 300, "alternate"), (40, 5000, "dictionary")]
    ins = [synth_core_inputs(T, S, 63, 7000 + i, style, planted=bool(i % 2)) for i, (T, S, style) in enumerate(shapes)]
    out = run_core_gpu([x["ids"] for x in ins], [x["prob_log"] for x in ins], [x["el"] for x in ins],
                       [x["ne"] for x in ins], [x["p"] for x in ins], 0.02)
    for x, g in zip(ins, out):
        check_core_against_oracle(x["ids"], x["prob_log"], x["el"], x["ne"], g, x["p"], 0.02)


def test_ties_go_to_the_earlier_candidate(routing):
    """Constant emissions and edge logs make stay/advance/skip tie everywhere: the strict '>' scan
    (alignment_decoder.py:210-218) must be reproduced exactly."""
    T, S = 64, 21
    ids = np.array([0, 3, 0, 4, 5, 0, 6, 0, 7, 8, 0, 9, 0, 1, 0, 2, 0, 3, 4, 0, 0][:S], dtype=np.int32)
    cases = []
    for val, e, n in [(-1.0, -0.5, -0.5), (0.0, 0.0, 0.0), (-2.0, -1.0, -3.0)]:
        cases.append((ids, np.full((T, S), val, np.float32), np.full(T, e, np.float32), np.full(T, n, np.float32)))
    out = run_core_gpu([c[0] for c in cases], [c[1] for c in cases], [c[2] for c in cases], [c[3] for c in cases])
    for c, g in zip(cases, out):
        check_core_against_oracle(c[0], c[1], c[2], c[3], g)


@pytest.mark.parametrize("pair", ["2", "0"], ids=["pair-layout", "plain-layout"])
def test_sp_pair_layout_edge_cases(pair, monkeypatch):
    """The SP-aware pair layout of the warp kernel (hfa_dp_pair_body) on the shapes its regrouping has to get
    right: with / without a leading SP (frame 1 is the one frame where an SP's curr is not 0, quirk q1), with /
    without a trailing SP (a pair without a phoneme), words of 1..4 phonemes (pairs without an SP), 1..4 pairs per
    lane, T = 1 / 2 / tile boundaries, coarse-grid values (ties), sprinkled -inf, and -0.0 everywhere (the SP
    shortcut must still give f32(f64(a) + 0.0) = +0.0 for a = -0.0).  Every dp cell and backpointer vs the oracle."""
    from hubertfa_b200 import ops
    monkeypatch.setenv("HFA_LATENCY_MODE", "0")
    monkeypatch.setenv("HFA_PAIR", pair)
    rng = np.random.default_rng(424242)
    ids_l, e_l, el_l, ne_l, p_l = [], [], [], [], []
    shapes = [(1, 1), (1, 2), (2, 1), (2, 2), (2, 3), (3, 2), (7, 3), (8, 5), (9, 4), (16, 8), (17, 30), (24, 33),
              (25, 64), (40, 65), (33, 100), (64, 128), (70, 150), (50, 200), (41, 213), (90, 256), (300, 90)]
    for i, (T, S) in enumerate(shapes * 3):
        lead, trail, mw = bool(i & 1), bool(i & 2), 1 + i % 4
        ids = pairable_ids(rng, S, lead, trail, mw)
        mode = i % 4
        if mode == 0:
            e = (-rng.exponential(3.0, (T, S))).astype(np.float32)
            p = rng.random(T).astype(np.float32)
        elif mode == 1:
            e = (-rng.integers(0, 4, (T, S)) * 0.5).astype(np.float32)
            p = (rng.integers(0, 3, T) * 0.5).astype(np.float32)
        elif mode == 2:
            e = np.full((T, S), -1.0, np.float32)
            p = np.full(T, 0.25, np.float32)
        else:
            e = np.where(rng.random((T, S)) < 0.5, -0.0, 0.0).astype(np.float32)
            p = rng.random(T).astype(np.float32)
        if i % 5 == 0:
            e[rng.random((T, S)) < 0.05] = -np.inf
        _, ep = onp.edge_streams(p)
        el, ne = onp.edge_logs(ep)
        if mode == 3:                                  # -0.0 edge logs: only reachable at this boundary
            el = np.where(rng.random(T) < 0.5, -0.0, 0.0).astype(np.float32)
            ne = np.where(rng.random(T) < 0.5, -0.0, 0.0).astype(np.float32)
        ids_l.append(ids); e_l.append(e); el_l.append(el); ne_l.append(ne); p_l.append(p)
    plan = ops.AlignPlan([e.shape[0] for e in e_l], [len(i) for i in ids_l], np.concatenate(ids_l), 4096, 0.02)
    r = plan.routing()
    n_pairable = sum(1 for ids in ids_l if ((ids != 0).sum() + (ids[-1] == 0) + 31) // 32 <= 4)
    assert r["warp_utts"] == len(ids_l) and r["pair_utts"] == (n_pairable if pair == "2" else 0)
    assert n_pairable >= 40
    out = run_core_gpu(ids_l, e_l, el_l, ne_l, p_l, 0.02)
    for i, g in enumerate(out):
        try:
            check_core_against_oracle(ids_l[i], e_l[i], el_l[i], ne_l[i], g, p_l[i], 0.02)
        except AssertionError as err:
            raise AssertionError(f"utterance {i} (T={e_l[i].shape[0]}, S={len(ids_l[i])}, ids={ids_l[i][:12]}): {err}") from err


def test_minus_inf_emissions_do_not_create_nan():
    T, S = 40, 9
    x = synth_core_inputs(T, S, 39, 77, "alternate")
    pl = x["prob_log"].copy()
    pl[5:9, 3] = -np.inf
    pl[20, :] = -np.inf
    out = run_core_gpu([x["ids"]], [pl], [x["el"]], [x["ne"]])
    check_core_against_oracle(x["ids"], pl, x["el"], x["ne"], out[0])


def test_invalid_utterances_get_a_status():
    import torch
    from hubertfa_b200 import ops
    good = synth_core_inputs(50, 9, 39, 5, "alternate")
    ids_bad = good["ids"].copy()
    ids_bad[2] = 1000
    plan = ops.AlignPlan([50, 0, 50], [9, 3, 9], np.concatenate([good["ids"], [0, 1, 0], ids_bad]), 39, 0.02)
    dev = torch.device("cuda")
    ws, res = plan.new_workspace(dev), plan.new_result(dev)
    plan.upload(ws)
    cat = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32).reshape(-1)).to(dev)
    ops.pack_emissions(ws, plan.handle, cat(good["prob_log"]), cat(good["el"]), cat(good["ne"]), None)
    ops.viterbi_forward(ws, plan.handle, None)
    ops.backtrace(ws, plan.handle, res, None, None)
    torch.cuda.synchronize()
    v = plan.views(res.cpu().numpy())
    assert list(v["status"]) == [0, 1, 2]
    assert v["n_seg"][1] == 0 and v["n_seg"][2] == 0
    r = oc.decode(good["ids"], good["prob_log"], good["el"], good["ne"])
    assert np.array_equal(v["ph_idx_seq"][:v["n_seg"][0]], r["ph_idx_seq"])


@pytest.mark.parametrize("big", ["cta", "band2", "band4", "band8", "skew2", "skew3"])
def test_long_form_c3_stress(big, monkeypatch):
    """BASELINE config 3: one 10-minute utterance, T=30000, S=2000 (1875 word rows): the CTA-per-
    utterance kernel, the banded kernel with 2 / 4 / 8 states per lane (63 / 21 / 9 warps) and the
    skewed-wavefront kernel (67 strips) with 2 / 3 frames of skew per state."""
    monkeypatch.setenv("HFA_BIG_KERNEL", "cta" if big == "cta" else "band")
    monkeypatch.setenv("HFA_LAT_KERNEL", "skew" if big.startswith("skew") else "band")
    if big.startswith("band"):
        monkeypatch.setenv("HFA_BIG_K", big[4:])
    if big.startswith("skew"):
        monkeypatch.setenv("HFA_SKEW_D", big[4:])
    x = synth_core_inputs(30000, 2000, 63, 31337, "dictionary", planted=True)
    out = run_core_gpu([x["ids"]], [x["prob_log"]], [x["el"]], [x["ne"]], [x["p"]], dump=False)
    r = check_core_against_oracle(x["ids"], x["prob_log"], x["el"], x["ne"], out[0], x["p"], full=False)
    assert len(r["ph_idx_seq"]) > 1000


def test_many_small_tie_heavy_utterances(routing):
    """300 small utterances in one batch: random SP patterns, coarse-grid values (ties everywhere),
    constant emissions, sprinkled -inf, T < S -- every dp cell, backpointer and path vs the C oracle."""
    from oracle import hfa_oracle_np as onp
    rng = np.random.default_rng(20241018)
    ids_l, e_l, el_l, ne_l, p_l = [], [], [], [], []
    for i in range(300):
        T, S = int(rng.integers(1, 70)), int(rng.integers(1, 90))
        sp_rate = [0.0, 0.3, 0.5, 0.8, 1.0][i % 5]
        ids = np.where(rng.random(S) < sp_rate, 0, rng.integers(1, 30, S)).astype(np.int32)
        mode = i % 3
        if mode == 0:
            e = (-rng.exponential(3.0, (T, S))).astype(np.float32)
            p = rng.random(T).astype(np.float32)
        elif mode == 1:
            e = (-rng.integers(0, 4, (T, S)) * 0.5).astype(np.float32)
            p = (rng.integers(0, 3, T) * 0.5).astype(np.float32)
        else:
            e = np.full((T, S), -1.0, np.float32)
            p = np.full(T, 0.25, np.float32)
        if i % 4 == 0:
            e[rng.random((T, S)) < 0.05] = -np.inf
        _, ep = onp.edge_streams(p)
        el, ne = onp.edge_logs(ep)
        ids_l.append(ids); e_l.append(e); el_l.append(el); ne_l.append(ne); p_l.append(p)
    out = run_core_gpu(ids_l, e_l, el_l, ne_l, p_l, 0.0116)
    for i, g in enumerate(out):
        try:
            check_core_against_oracle(ids_l[i], e_l[i], el_l[i], ne_l[i], g, p_l[i], 0.0116)
        except AssertionError as err:
            raise AssertionError(f"utterance {i} (T={e_l[i].shape[0]}, S={len(ids_l[i])}): {err}") from err
