"""GPU: the kept-dp backtrace walked out of shared memory (hfa_backtrace_walk_kernel, HFA_BT_WALK=2) against the
jump-table backtrace (HFA_BT_WALK=0): every result the caller sees -- the result blob's fields, frame_conf and
dp_path -- bit for bit the same, and both against the C oracle.  Row boundaries of the 16-frame backpointer words,
one- and two-state sequences, SP at either end and SP jumps on consecutive frames, an infeasible utterance, the
walk/table split at the size cap inside one batch, a giant, and every dp-store layout of the latency kernels."""
import numpy as np
import pytest

from oracle import c_oracle as oc
from gpu_util import bits, check_core_against_oracle, run_core_gpu, synth_core_inputs

pytestmark = pytest.mark.gpu

FIELDS = ("status", "n_seg", "end_state", "ph_idx_seq", "ph_time_int", "intervals")
FLOATS = ("final_score", "total_conf", "frame_conf", "dp_path")


def _latency_env(monkeypatch, extra=None):
    monkeypatch.setenv("HFA_LATENCY_MODE", "2")
    monkeypatch.setenv("HFA_BIG_KERNEL", "band")
    for k, v in (extra or {}).items():
        monkeypatch.setenv(k, v)


def _plan(ins):
    from hubertfa_b200 import ops
    return ops.AlignPlan([x["prob_log"].shape[0] for x in ins], [len(x["ids"]) for x in ins],
                         np.concatenate([x["ids"] for x in ins]), 4096, 0.02)


def _run(ins, monkeypatch, mode):
    monkeypatch.setenv("HFA_BT_WALK", mode)
    r = _plan(ins).routing()
    out = run_core_gpu([x["ids"] for x in ins], [x["prob_log"] for x in ins], [x["el"] for x in ins],
                       [x["ne"] for x in ins], [x["p"] for x in ins], 0.02, dump=False)
    return r, out


def _same(a, b, what):
    for x, y in zip(a, b):
        for k in FIELDS:
            assert np.array_equal(np.asarray(x[k]), np.asarray(y[k])), f"{what}: {k} differs"
        for k in FLOATS:
            assert np.array_equal(bits(np.atleast_1d(x[k])), bits(np.atleast_1d(y[k]))), f"{what}: {k} differs"


def _both_routes(ins, monkeypatch, n_walk):
    r0, tab = _run(ins, monkeypatch, "0")
    r2, walk = _run(ins, monkeypatch, "2")
    assert r0["keeps_dp"] and r0["bt_walk_utts"] == 0
    assert r2["bt_walk_utts"] == n_walk
    _same(tab, walk, "walk vs tables")
    for i, (x, g) in enumerate(zip(ins, walk)):
        if np.isneginf(x["prob_log"]).all():
            r = oc.decode(x["ids"], x["prob_log"], x["el"], x["ne"])
            assert np.isneginf(r["dp_path"][-1]) and g["status"] == 4
            continue
        try:
            check_core_against_oracle(x["ids"], x["prob_log"], x["el"], x["ne"], g, x["p"], 0.02)
        except AssertionError as e:
            raise AssertionError(f"utterance {i} (T={x['prob_log'].shape[0]}, S={len(x['ids'])}): {e}") from e
    return walk


def _with_ids(x, ids, seed):
    """Inputs of synth_core_inputs re-targeted at a given id sequence (same frames)."""
    rng = np.random.default_rng(seed)
    T = x["prob_log"].shape[0]
    lp = np.log(rng.dirichlet(np.ones(64), size=T)).astype(np.float32)
    y = dict(x)
    y["ids"] = np.asarray(ids, np.int32)
    y["prob_log"] = np.ascontiguousarray(lp[:, y["ids"]])
    return y


EDGE_SHAPES = [  # (T, S, style): row boundaries of the backpointer words, tiny sequences
    (1, 1, "dictionary"), (15, 1, "nosp"), (16, 2, "dictionary"), (17, 2, "alternate"), (31, 7, "dictionary"),
    (47, 12, "alternate"), (63, 20, "dictionary"), (16, 16, "nosp"), (257, 64, "dictionary"),
    (1475, 149, "dictionary"), (900, 300, "alternate"),
]


def _edge_batch():
    ins = [synth_core_inputs(T, S, 63, 7700 + i, style, planted=bool(i % 2))
           for i, (T, S, style) in enumerate(EDGE_SHAPES)]
    base = synth_core_inputs(40, 9, 63, 7790, "dictionary")
    # SP at both ends, then SP between every phoneme with as many frames as phonemes: the path jumps an SP on
    # consecutive frames
    ins.append(_with_ids(base, [0, 5, 0, 7, 0, 9, 0, 11, 0], 7791))
    fast = synth_core_inputs(20, 5, 63, 7792, "alternate")
    ins.append(_with_ids(fast, [0] + [v for k in range(20) for v in (3 + k, 0)], 7793))
    ins.append(_with_ids(synth_core_inputs(33, 6, 63, 7794, "nosp"), [0, 4, 6, 8, 10, 0], 7795))
    # infeasible: every kept logit -inf (status 4)
    dead = synth_core_inputs(50, 8, 63, 7796, "dictionary")
    dead["prob_log"] = np.full_like(dead["prob_log"], -np.inf)
    ins.append(dead)
    return ins


@pytest.mark.parametrize("layout", [
    {}, {"HFA_SKEW_D": "3"}, {"HFA_SKEW_CTAS": "4"}, {"HFA_SKEW_CTAS": "5"}, {"HFA_LAT_KERNEL": "band"},
], ids=["skew_d2", "skew_d3", "ctas4", "ctas5", "band"])
def test_walk_matches_tables_and_oracle(layout, monkeypatch):
    _latency_env(monkeypatch, layout)
    ins = _edge_batch()
    walk = _both_routes(ins, monkeypatch, len(ins))
    assert walk[-1]["status"] == 4


def _cap_rows(monkeypatch, S):
    """Most 16-frame rows an S-state utterance may have and still take the walk (its words fit in one CTA's shared
    memory; found from the plan's routing, so the test follows the limit wherever it is set)."""
    from hubertfa_b200 import ops
    lo, hi = 1, 4096
    while lo < hi:
        mid = (lo + hi + 1) // 2
        r = ops.AlignPlan([16 * mid], [S], np.arange(S, dtype=np.int32) % 7 + 1, 4096, 0.02).routing()
        lo, hi = (mid, hi) if r["bt_walk_utts"] == 1 else (lo, mid - 1)
    return lo


def test_cap_splits_one_batch_and_giant_keeps_tables(monkeypatch):
    """An utterance at the cap walks, one a row above it and a giant (S > 8192) take the jump tables, all in one
    call, and every result equals the all-tables route's."""
    _latency_env(monkeypatch)
    monkeypatch.delenv("HFA_BT_WALK", raising=False)
    S = 148
    rows = _cap_rows(monkeypatch, S)
    assert 1 < rows < 4096
    ins = [synth_core_inputs(16 * rows, S, 63, 7800, "dictionary", planted=True),
           synth_core_inputs(16 * rows + 1, S, 63, 7801, "dictionary", planted=True),
           synth_core_inputs(400, 60, 63, 7802, "alternate"),
           synth_core_inputs(8300, 8200, 63, 7803, "nosp", planted=True)]
    _both_routes(ins, monkeypatch, 2)                 # the one at the cap and the short one
