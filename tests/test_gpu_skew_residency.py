"""GPU, tier 1: the skewed-wavefront kernel at both residencies -- 4 strips per SM (a 6-stage ring) and 5 (a
5-stage ring) -- bit for bit against the C oracle in its DUMP and production instantiations, the exchange table
all-zero after every call, and the residency the plan picks for the bench batches."""
import numpy as np
import pytest

from gpu_util import check_core_against_oracle, run_core_gpu, synth_core_inputs

pytestmark = pytest.mark.gpu

SHAPES = [  # (T, S, style): one strip, several strips, ramps longer than the utterance, S > 256
    (1, 1, "dictionary"), (2, 5, "nosp"), (17, 12, "dictionary"), (33, 33, "alternate"), (100, 20, "dictionary"),
    (257, 64, "dictionary"), (300, 65, "dictionary"), (40, 150, "alternate"), (480, 96, "nosp"),
    (700, 160, "dictionary"), (1000, 513, "alternate"), (1475, 149, "dictionary"),
]


def _skew_env(monkeypatch, d, ctas):
    monkeypatch.setenv("HFA_LATENCY_MODE", "2")
    monkeypatch.setenv("HFA_BIG_KERNEL", "band")
    monkeypatch.setenv("HFA_LAT_KERNEL", "skew")
    monkeypatch.setenv("HFA_SKEW_D", d)
    if ctas:
        monkeypatch.setenv("HFA_SKEW_CTAS", ctas)


@pytest.mark.parametrize("d", ["2", "3"])
@pytest.mark.parametrize("ctas", ["4", "5"])
def test_both_residencies_match_the_oracle(ctas, d, monkeypatch):
    from hubertfa_b200 import ops
    _skew_env(monkeypatch, d, ctas)
    ins = [synth_core_inputs(T, S, 63, 9100 + i, style, planted=bool(i % 2)) for i, (T, S, style) in enumerate(SHAPES)]
    plan = ops.AlignPlan([x["prob_log"].shape[0] for x in ins], [len(x["ids"]) for x in ins],
                         np.concatenate([x["ids"] for x in ins]), 4096, 0.02)
    r = plan.routing()
    assert r["skew_d"] == int(d) and r["skew_ctas_per_sm"] == int(ctas) and r["big_skew_ctas_per_sm"] == int(ctas)
    out = run_core_gpu([x["ids"] for x in ins], [x["prob_log"] for x in ins], [x["el"] for x in ins],
                       [x["ne"] for x in ins], [x["p"] for x in ins], 0.02)
    for x, g, shp in zip(ins, out, SHAPES):
        try:
            check_core_against_oracle(x["ids"], x["prob_log"], x["el"], x["ne"], g, x["p"], 0.02)
        except AssertionError as e:
            raise AssertionError(f"shape {shp}: {e}") from e


@pytest.mark.parametrize("d", ["2", "3"])
@pytest.mark.parametrize("ctas", ["4", "5"])
def test_exchange_table_is_zero_after_every_call(ctas, d, monkeypatch):
    """Tags are frame numbers, the same in every call: a slot left set would be taken for the next call's value.
    Three calls of the production kernel over one workspace, then its paths, segment times and path scores."""
    import torch
    from hubertfa_b200 import ops
    _skew_env(monkeypatch, d, ctas)
    ins = [synth_core_inputs(T, S, 63, 9300 + i, "dictionary", planted=True)
           for i, (T, S) in enumerate([(900, 150), (333, 97), (1475, 149)])]
    plan = ops.AlignPlan([x["prob_log"].shape[0] for x in ins], [len(x["ids"]) for x in ins],
                         np.concatenate([x["ids"] for x in ins]), 4096, 0.02)
    r = plan.routing()
    assert r["skew_d"] == int(d) and r["skew_ctas_per_sm"] + r["big_skew_ctas_per_sm"] == int(ctas)
    dev = torch.device("cuda")
    ws, res = plan.new_workspace(dev), plan.new_result(dev)
    plan.upload(ws)
    cat = lambda k: torch.from_numpy(np.concatenate([np.ascontiguousarray(x[k], np.float32).reshape(-1)
                                                     for x in ins])).to(dev)
    ops.pack_emissions(ws, plan.handle, cat("prob_log"), cat("el"), cat("ne"), None)
    xchg = plan.debug_region(ws, "xchg")
    assert xchg.numel() > 0
    for call in range(3):
        ops.viterbi_forward(ws, plan.handle, None)
        torch.cuda.synchronize()
        assert int((xchg != 0).sum()) == 0, f"call {call}: exchange slots left set"
    ops.backtrace(ws, plan.handle, res, None, None)
    v = plan.views(res.cpu().numpy())
    from oracle import c_oracle as oc
    for b, x in enumerate(ins):
        want = oc.decode(x["ids"], x["prob_log"], x["el"], x["ne"])
        o, k = int(plan.seg_off[b]), int(v["n_seg"][b])
        assert np.array_equal(v["ph_idx_seq"][o:o + k], want["ph_idx_seq"])
        assert np.array_equal(v["ph_time_int"][o:o + k], want["ph_time_int"])
        assert abs(v["final_score"][b] - want["dp_path"][-1]) <= 1e-4 * abs(want["dp_path"][-1])


@pytest.mark.parametrize("n_utt,want", [(1, 4), (256, 4), (512, 5)])
def test_residency_follows_the_list_schedule(n_utt, want):
    """4 strips per SM where the list schedule of the strips is no longer with them (one utterance, the
    256-utterance bench batch), 5 where it is (512 utterances: 106 vs 93 blocks on 148 SMs)."""
    import torch
    from hubertfa_b200 import ops, synth
    if torch.cuda.get_device_properties(0).multi_processor_count != 148:
        pytest.skip("the expected choices are worked out for 148 SMs")
    if n_utt == 1:
        T, S = np.array([30000], np.int32), np.array([2000], np.int32)
    else:
        T, S = synth.sample_shapes(n_utt, seed=synth.SEED0, min_s=5, max_s=30, s_lo=20, s_hi=150)
    ids = np.concatenate(synth.make_ids_batch(T, S, 63, seed=synth.SEED0))
    r = ops.AlignPlan(T, S, ids, 63, synth.FRAME_SECONDS).routing()
    assert r["skew_d"] == 2 and max(r["skew_ctas_per_sm"], r["big_skew_ctas_per_sm"]) == want
