"""Long-form utterances (S > 8192 phoneme states) on the host: plan statuses, routing, workspace layout, and
the low-memory oracle the GPU long-form tests check against.  No GPU needed."""
import numpy as np
import pytest

from hubertfa_b200 import _lib, ops, sharding, synth

V = 63


def giant_ids(S, seed):
    """A dictionary-style id row: words of 2-6 phonemes separated by SP (id 0)."""
    rng = np.random.default_rng(seed)
    ids = rng.integers(1, V, size=S).astype(np.int32)
    ids[rng.random(S) < 0.25] = 0
    ids[1:][(ids[1:] == 0) & (ids[:-1] == 0)] = 5          # no two SPs in a row
    return ids


def plan_of(T, S, ids):
    return ops.AlignPlan(T, S, ids, V, 0.02)


@pytest.mark.parametrize("S", [8192, 8193, 20_000, _lib.MAX_STATES, _lib.MAX_STATES + 1])
def test_plan_status_of_long_sequences(S):
    T = 3 * S
    p = plan_of([T], [S], np.ones(S, np.int32))
    accepted = S <= _lib.MAX_STATES
    assert p.total_cells == (T * S if accepted else 0)
    assert list(p.frame_off) == [0, T if accepted else 0]
    rt = p.routing()
    assert rt["cta_utts"] == 0 and rt["warp_utts"] == 0
    if accepted and S > 8192:
        # strips (one state per lane) with the TMA tensor maps, 2-states-per-lane halo bands without them
        assert rt["big_band_k"] == (1 if rt["skew_d"] > 0 else 2)
        assert rt["big_band_warps"] >= S // 64 and rt["keeps_dp"]


def test_header_and_python_agree_on_max_states():
    import os
    import re
    hdr = open(os.path.join(os.path.dirname(__file__), "..", "include", "hfa_align.h")).read()
    assert re.search(r"#define HFA_MAX_STATES \(1 << 20\)", hdr)
    assert _lib.MAX_STATES == 1 << 20


def _config4(seed=synth.SEED0 + V):
    T, S = synth.sample_shapes(4096, seed=seed)
    ids = synth.make_ids_batch(T, S, V, seed=seed)
    return list(T), list(S), list(ids)


def _giants():
    return [(40_000, 12_000, giant_ids(12_000, 1)), (70_000, 20_000, giant_ids(20_000, 2))]


def test_giant_alone_and_inside_a_big_batch_is_never_in_the_cta_kernel():
    t, s, ids = _giants()[0]
    alone = plan_of([t], [s], ids).routing()
    assert alone["cta_utts"] == 0 and alone["warp_utts"] == 0 and alone["big_band_warps"] > 0
    T, S, I = _config4()
    base = plan_of(T, S, np.concatenate(I)).routing()
    assert base["warp_utts"] == 4096 and base["big_band_warps"] == 0 and base["cta_utts"] == 0
    giants = _giants()
    T2, S2, I2 = T + [g[0] for g in giants], S + [g[1] for g in giants], I + [g[2] for g in giants]
    mixed = plan_of(T2, S2, np.concatenate(I2))
    rt = mixed.routing()
    # every other utterance: same kernel, same pair layout, same stored emission rows as without the giants
    for k in ("warp_utts", "band_warps", "band_k", "cta_utts", "pair_utts"):
        assert rt[k] == base[k], k
    assert rt["stored_emission_bytes"] == base["stored_emission_bytes"] + sum(4 * g[0] * g[1] for g in giants)
    # the giants: strips (or halo bands without tensor maps), dp kept for the table backtrace
    k = rt["big_band_k"]
    assert k == (1 if rt["skew_d"] > 0 else 2) and rt["keeps_dp"]
    per = (lambda sp: 1 + (sp - 32 + 29) // 30) if k == 1 else (lambda sp: (sp - 32 + 31) // 32)
    assert rt["big_band_warps"] == sum(per((g[1] + 3) // 4 * 4) for g in giants)


def test_giant_routing_ignores_the_band_budget(monkeypatch):
    monkeypatch.setenv("HFA_BAND_MAX", "1")
    t, s, ids = _giants()[1]
    rt = plan_of([t, 500], [s, 400], np.concatenate([ids, giant_ids(400, 3)])).routing()
    assert rt["cta_utts"] == 1 and rt["big_band_warps"] > 1     # the S = 400 one stays in the CTA kernel
    monkeypatch.setenv("HFA_KEEP_DP", "0")
    assert not plan_of([t], [s], ids).routing()["keeps_dp"]


def test_workspace_and_result_layout_beyond_4_gib():
    T, S = 400_000, 20_000
    p = plan_of([T], [S], giant_ids(S, 4))
    assert p.total_cells == T * S > 2 ** 32
    emis_off, emis_bytes = p._lib.hfa_plan_debug_region(p._h, 0, None), T * S * 4
    n = ops.C.c_int64()
    for which, want in ((0, emis_bytes), (1, T * 8), (2, T * 4), (3, (T + 15) // 16 * S * 4)):
        off = p._lib.hfa_plan_debug_region(p._h, which, ops.C.byref(n))
        assert n.value == want and 0 <= off and off + want <= p.workspace_bytes
    assert emis_off >= 0 and p.workspace_bytes > emis_bytes > 2 ** 32
    L = p.layout
    offs = [L.status, L.n_seg, L.end_state, L.final_score, L.total_conf, L.ph_idx_seq, L.ph_time_int, L.intervals]
    assert offs == sorted(offs) and L.ph_time_int == L.ph_idx_seq + 4 * S and L.intervals >= L.ph_time_int + 4 * S
    assert L.total_bytes >= L.intervals + 16 * S


def test_chunk_by_bytes_gives_an_over_budget_utterance_a_chunk_of_its_own():
    T = [100, 200, 180_000, 50, 60]
    S = [10, 20, 12_000, 5, 6]
    chunks = sharding.chunk_by_bytes(T, S, max_cells=1_000_000)
    assert [list(c) for c in chunks] == [[0, 1], [2], [3, 4]]


def _rand_inputs(T, S, seed, sp_frac=0.3):
    rng = np.random.default_rng(seed)
    ids = rng.integers(1, 9, size=S).astype(np.int32)
    ids[rng.random(S) < sp_frac] = 0
    e = (-rng.exponential(2.0, size=(T, S))).astype(np.float32)
    e[rng.random((T, S)) < 0.02] = -np.inf
    el = np.log(rng.random(T) + 1e-6).astype(np.float32)
    ne = np.log(1 - rng.random(T) + 1e-6).astype(np.float32)
    return ids, e, el, ne


def _same(a):
    from oracle import c_oracle as oc
    from oracle import lowmem_oracle as lo
    ids, e, el, ne = a
    r = oc.decode(ids, e, el, ne)
    for chunk in (1, 7, 4096):
        q = lo.decode(ids, e, el, ne, chunk=chunk)
        assert q["rc"] == r["rc"]
        if r["rc"] != 0:
            continue
        assert np.array_equal(q["ph_idx_seq"], r["ph_idx_seq"]) and np.array_equal(q["ph_time_int"], r["ph_time_int"])
        assert q["end_state"] == r["end_state"]
        assert np.array_equal(q["dp_path"].view(np.uint32), r["dp_path"].view(np.uint32))
        assert q["final_score"].view(np.uint32) == r["dp_path"][-1].view(np.uint32)
        fq, tq = oc.confidence(q["dp_path"])
        fr, tr = oc.confidence(r["dp_path"])
        assert np.array_equal(fq.view(np.uint32), fr.view(np.uint32)) and np.array_equal(tq, tr, equal_nan=True)


@pytest.mark.parametrize("shape", [(1, 1), (1, 5), (2, 1), (7, 3), (40, 40), (100, 13), (300, 77), (64, 200)])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_lowmem_oracle_equals_full_oracle_on_random_shapes(shape, seed):
    _same(_rand_inputs(*shape, seed=seed))


def test_lowmem_oracle_equals_full_oracle_on_golden_cases(golden):
    from oracle import c_oracle as oc
    assert golden.names
    for name in golden.names:
        c = golden.case(name)
        el, ne = oc.edge_logs(c["edge_prob"])
        _same((c["ids"], c["prob_log"], el, ne))
