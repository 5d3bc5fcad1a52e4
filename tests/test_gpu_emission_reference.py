"""GPU: the logits -> emission / edge stage (hfa_emission.cu, the fused band producer in hfa_dp.cu) against
the float64 reference of oracle/emission_f64.py, within its derived per-element bound, and bit for bit
where two routes must agree; tier 1 (every dp cell and backpointer against the C oracle) on compacted rows.

Contract (DESIGN.md 4.1): finite logits with |x| < 5e8, and -inf anywhere.  A row whose kept logits are
all -inf gives -inf emissions, as in the reference (its masked logits stay finite); a row in which EVERY
logit is -inf gives -inf too, where the reference gives NaN (a deliberate divergence).  NaN, +inf and
|x| >= 5e8 are out of contract.

Which kernel runs follows from the inputs (HFA_EMISSION_NO_TMA and HFA_FUSED are read once per process):
  stream  unit column stride and a 64-row stage of at most 48 KiB (f32 head views [T, V+2] up to V = 189)
  block   column stride != 1 (a transposed view), or a larger stage (f32 head views, V = 190 .. 255)
  wide    V >= 256
Compacted rows (one column per distinct id) are written for the utterances the plan puts into the warp
kernel's pair layout (HFA_PAIR=2, HFA_LATENCY_MODE=0 force it; HFA_COMPACT=0 keeps plain rows)."""
import time

import numpy as np
import pytest
import torch

from gpu_util import bits, check_core_against_oracle, pairable_ids, run_core_from_logits
from hubertfa_b200 import _lib, ops, synth
from oracle import c_oracle as oc
from oracle import emission_f64 as ef

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda")
DTYPES = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
STYLES = ["gauss", "planted", "range80", "grid", "neginf_kept", "neginf_masked", "dead_rows"]


@pytest.fixture(scope="module", autouse=True)
def _module_time():
    t0 = time.perf_counter()
    yield
    print(f"\n{__name__}: {time.perf_counter() - t0:.1f} s")


# ------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------
def make_ids(rng, S, n_kept, V, pairable=False):
    """S phoneme ids that keep exactly min(n_kept, V, S + 1) vocabulary ids (id 0 always counts).  pairable:
    no two SPs adjacent and at most 125 phonemes (the pair layout's conditions); otherwise SP runs occur."""
    n_kept = max(1, min(n_kept, V, S + 1))
    if n_kept == 1:
        return np.zeros(S, np.int32)
    kept = rng.choice(np.arange(1, V), n_kept - 1, replace=False)
    n_phon = min(S, max(n_kept - 1, (S + 1) // 2 if pairable else S - S // 3))
    phon = rng.permutation(np.concatenate([kept, rng.choice(kept, n_phon - (n_kept - 1))]))
    n_sp = S - n_phon
    gaps = np.zeros(n_phon + 1, np.int64)                  # SPs before phoneme g (g = n_phon: trailing)
    if pairable:
        gaps[rng.choice(n_phon + 1, n_sp, replace=False)] = 1
    else:
        np.add.at(gaps, rng.integers(0, n_phon + 1, n_sp), 1)
    ids = []
    for g in range(n_phon + 1):
        ids += [0] * int(gaps[g])
        if g < n_phon:
            ids.append(int(phon[g]))
    return np.array(ids, np.int32)


def make_head(rng, T, V, ids, style):
    """One utterance's network head [T, V + 2] in f32: column 0 the edge logit, 2.. the frame logits."""
    keep = ef.keep_mask(ids, V)
    if style == "range80":
        x = rng.uniform(-80.0, 80.0, (T, V))
    elif style == "grid":                             # coarse grid: the row max ties, emissions tie
        x = rng.integers(-3, 2, (T, V)) * 0.5
    else:
        x = 3.0 * rng.standard_normal((T, V))
    if style == "planted":                            # a monotone path of clear winners
        s = (np.arange(T) * len(ids)) // max(T, 1)
        x[np.arange(T), ids[s]] += 8.0
    elif style == "neginf_kept":
        x[(rng.random((T, V)) < 0.2) & keep] = -np.inf
    elif style == "neginf_masked":
        x[(rng.random((T, V)) < 0.3) & ~keep] = -np.inf
    elif style == "dead_rows":                        # every kept logit -inf / every logit -inf
        r = rng.random(T)
        x[np.ix_(r < 0.25, keep)] = -np.inf
        x[r > 0.85] = -np.inf
    head = np.zeros((T, V + 2), np.float32)
    head[:, 2:] = x
    head[:, 0] = np.where(rng.random(T) < 0.1, rng.uniform(-30.0, 30.0, T), 2.0 * rng.standard_normal(T))
    head[:, 1] = 7.0                                  # never read
    return head


def run_emission(heads, ids_list, V, dtype, view="head"):
    """hfa_emission on `heads` (host f32 arrays, cast to `dtype` on the device).  view: "head" = the [T, V+2]
    head views (unit column stride), "transposed" = the same values with column stride T.  Returns (plan,
    per-utterance (emissions [T, S], edge2 [T, 2], edge_p [T]), device heads)."""
    dh = [torch.from_numpy(h).to(DEV).to(dtype) for h in heads]
    if view == "head":
        frames = [h[:, 2:] for h in dh]
    else:
        frames = [h[:, 2:].t().contiguous().t() for h in dh]
    edges = [h[:, 0] for h in dh]
    T = [h.shape[0] for h in heads]
    plan = ops.AlignPlan(T, [len(i) for i in ids_list], np.concatenate(ids_list), V, 0.02)
    ws = plan.new_workspace(DEV)
    plan.upload(ws)
    plan.set_inputs(ws, [f.data_ptr() for f in frames], [f.stride(0) for f in frames], [f.stride(1) for f in frames],
                    [e.data_ptr() for e in edges], [e.stride(0) for e in edges])
    ops.emission(ws, plan.handle, ops.TORCH_TO_DTYPE[dtype])
    emis = ops.unpack_emissions(plan, ws).cpu().numpy()
    edge2 = plan.debug_region(ws, "edge2").cpu().numpy()
    edgep = plan.debug_region(ws, "edge_p").cpu().numpy()
    out, cell, eo = [], 0, 0
    for t, ids in zip(T, ids_list):
        S = len(ids)
        out.append((emis[cell:cell + t * S].reshape(t, S).copy(), edge2[eo:eo + t].copy(), edgep[eo:eo + t].copy()))
        cell += t * S
        eo += (t + 15) // 16 * 16
    return plan, out, dh


def check_against_f64(head_vals, ids, V, got, what):
    """One utterance: emissions within the bound (exact -inf where the reference has -inf, -inf for rows of
    all -inf logits), edge_p within its bound, edge logs within 1 f32 ulp of the f64 logs of OUR p."""
    e, e2, p = got
    x = head_vals[:, 2:]
    out, xm, lse, n = ef.emission_f64(x, ids, V)
    depth = ef.sum_depth(n, V, "wide" if V > 255 else "stream")
    dead = np.isneginf(x).all(axis=1)
    assert np.isnan(out[dead]).all() and not np.isnan(out[~dead]).any(), what
    assert not np.isnan(e).any(), f"{what}: NaN emissions in rows {np.unique(np.nonzero(np.isnan(e))[0])[:8]}"
    assert np.isneginf(e[dead]).all(), f"{what}: rows of all -inf logits must give -inf"
    ok = ~dead[:, None] & np.ones_like(e, dtype=bool)
    assert np.array_equal(np.isneginf(e[ok]), np.isneginf(out[ok])), f"{what}: -inf pattern differs"
    fin = ok & np.isfinite(out)
    err = np.abs(e[fin].astype(np.float64) - out[fin])
    bound = ef.emission_bound(out, xm, lse, n, depth)[fin]
    if err.size:
        worst = int(np.argmax(err / bound))
        assert (err <= bound).all(), (f"{what}: emission error {err[worst]:.3e} > bound {bound[worst]:.3e} "
                                      f"(n_kept={n}, ratio {err[worst] / bound[worst]:.2f})")
    pw, pb = ef.edge_pred_f64(head_vals[:, 0])
    assert (np.abs(p.astype(np.float64) - pw) <= pb).all(), f"{what}: edge_p outside its bound"
    wl, wn = ef.edge_logs_f64(p)
    assert (np.abs(e2[:, 0] - wl) <= ef.f32_ulp(wl)).all(), f"{what}: edge_log"
    assert (np.abs(e2[:, 1] - wn) <= ef.f32_ulp(wn)).all(), f"{what}: not_edge_log"


def values_of(dh):
    """The values the kernel read (exact f32 of the f16 / bf16 logits)."""
    return [h.float().cpu().numpy() for h in dh]


S_AXIS = [1, 4, 32, 33, 64, 65, 128, 129, 256, 257, 1030]
KEPT_AXIS = [1, 32, 33, 40, 41, 48, 49, 56, 57, 64, 65, 200]
T_AXIS = [1, 63, 64, 65, 129]


def matrix_batch(V, seed):
    """Every S and every kept-id count of the axes above (clipped to what V and S allow), T and value style
    cycling, in ONE ragged batch."""
    rng = np.random.default_rng(seed)
    cases = [(S, KEPT_AXIS[i % len(KEPT_AXIS)]) for i, S in enumerate(S_AXIS)]
    cases += [(max(k + 20, 40), k) for k in KEPT_AXIS]
    heads, ids_list = [], []
    for i, (S, k) in enumerate(cases):
        ids = make_ids(rng, S, k, V)
        ids_list.append(ids)
        heads.append(make_head(rng, T_AXIS[i % len(T_AXIS)], V, ids, STYLES[i % len(STYLES)]))
    return heads, ids_list


# ------------------------------------------------------------------------------------------------
# B. emissions and edge stream against the f64 reference
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("V", [2, 39, 63, 74, 189, 190, 255, 256, 300])
def test_emission_matrix_vs_f64(V, dt):
    """Head views [T, V+2]: stream kernel (f32 to V = 189, f16 / bf16 to 255), block kernel (f32 V = 190 / 255:
    the 64-row stage exceeds 48 KiB), wide kernel (V = 256 / 300).  Sp 4 .. 1032, kept ids 1 .. 200 (the 8 .. 16
    register slots of the normaliser and its generic loop past 64), T = 1 / 63 / 64 / 65 / 129, all value styles.
    Odd row strides of f16 / bf16 views give non-zero 16-byte shifts in the stream kernel's bulk copies."""
    heads, ids_list = matrix_batch(V, 1000 + V)
    _, got, dh = run_emission(heads, ids_list, V, DTYPES[dt])
    for i, (h, ids, g) in enumerate(zip(values_of(dh), ids_list, got)):
        check_against_f64(h, ids, V, g, f"V={V} {dt} utterance {i} (T={h.shape[0]}, S={len(ids)})")


@pytest.mark.parametrize("V", [39, 74, 200, 255])
def test_block_kernel_strided_views_vs_f64_and_stream_bits(V):
    """Column stride != 1 takes the thread-loaded block kernel.  Against the f64 reference, and -- same kept-id
    summation order -- bit-identical to the stream kernel (f16 head views: a stage of at most 48 KiB)."""
    heads, ids_list = matrix_batch(V, 2000 + V)
    _, got_b, dh = run_emission(heads, ids_list, V, torch.float16, view="transposed")
    for i, (h, ids, g) in enumerate(zip(values_of(dh), ids_list, got_b)):
        check_against_f64(h, ids, V, g, f"block V={V} utterance {i}")
    _, got_s, _ = run_emission(heads, ids_list, V, torch.float16, view="head")
    for i, (a, b) in enumerate(zip(got_b, got_s)):
        for j in range(3):
            assert np.array_equal(bits(a[j]), bits(b[j])), f"utterance {i}: stream and block kernels differ"


@pytest.mark.parametrize("V,dt,view", [(63, "f32", "head"), (63, "bf16", "head"), (63, "f32", "transposed"),
                                       (300, "f16", "head")])
def test_ids_past_the_staged_8192(V, dt, view):
    """S = 8200: the ids of states 8192 .. 8199 are read from global memory in the gather (stream, block) and in
    the wide kernel's loop."""
    rng = np.random.default_rng(V + len(dt))
    ids_list = [make_ids(rng, 8200, min(V, 57), V), make_ids(rng, 37, 20, V), make_ids(rng, 300, 41, V)]
    ids_list[0][8190:] = rng.choice(np.arange(1, V), 10)       # distinct ids out there
    heads = [make_head(rng, T, V, ids, st) for T, ids, st in zip((3, 65, 2), ids_list, ("gauss", "neginf_kept", "grid"))]
    _, got, dh = run_emission(heads, ids_list, V, DTYPES[dt], view)
    for i, (h, ids, g) in enumerate(zip(values_of(dh), ids_list, got)):
        check_against_f64(h, ids, V, g, f"utterance {i}")


def test_persistent_ctas_span_many_utterances():
    """2400 short utterances: every persistent stream CTA walks several utterances and must redo the per-
    utterance setup (ids, keep mask, kept list, register slots, lanes per row) at each boundary."""
    V = 63
    rng = np.random.default_rng(77)
    heads, ids_list = [], []
    for i in range(2400):
        T, S = int(rng.integers(1, 90)), int(rng.integers(1, 70))
        ids = make_ids(rng, S, int(rng.choice([1, 2, 9, 33, 41, 49, 57, 63])), V)
        ids_list.append(ids)
        heads.append(make_head(rng, T, V, ids, STYLES[i % len(STYLES)]))
    plan, got, dh = run_emission(heads, ids_list, V, torch.float32)
    for i, (h, ids, g) in enumerate(zip(values_of(dh), ids_list, got)):
        check_against_f64(h, ids, V, g, f"utterance {i}")


@pytest.mark.parametrize("dt", list(DTYPES))
def test_f16_bf16_logits_give_the_bits_of_their_f32_values(dt):
    """The kernels convert each logit to f32 and do nothing else with its type: an f16 / bf16 head gives the same
    bits as the f32 tensor of the same values (stream kernel; the transposed views: block kernel)."""
    V = 200
    heads, ids_list = matrix_batch(V, 3000)
    for view in ("head", "transposed"):
        _, got_h, dh = run_emission(heads, ids_list, V, DTYPES[dt], view)
        _, got_f, _ = run_emission(values_of(dh), ids_list, V, torch.float32, view)
        for i, (a, b) in enumerate(zip(got_h, got_f)):
            for j in range(3):
                assert np.array_equal(bits(a[j]), bits(b[j])), f"{view} utterance {i}: {dt} != f32 of its values"


# ------------------------------------------------------------------------------------------------
# compacted rows
# ------------------------------------------------------------------------------------------------
def pair_batch(rng, V, shapes, kept):
    heads, ids_list = [], []
    for i, (T, S) in enumerate(shapes):
        ids = make_ids(rng, S, kept[i % len(kept)], V, pairable=True)
        ids_list.append(ids)
        heads.append(make_head(rng, T, V, ids, STYLES[i % len(STYLES)]))
    return heads, ids_list


def assert_compacted(plan, n_pair):
    r = plan.routing()
    full = 4 * int(sum(int(t) * ((int(s) + 3) // 4 * 4) for t, s in zip(plan.T, plan.S)))
    assert r["pair_utts"] == n_pair and r["stored_emission_bytes"] < full, r


PAIR_SHAPES = [(1, 8), (2, 33), (63, 32), (64, 64), (65, 65), (129, 100), (70, 128), (33, 200), (90, 250), (7, 13)]


@pytest.mark.parametrize("dt,V,view", [("f32", 63, "head"), ("f16", 74, "head"), ("bf16", 200, "head"),
                                       ("f32", 190, "head"), ("f32", 63, "transposed")])
def test_compacted_rows_vs_f64_and_plain_bits(dt, V, view, monkeypatch):
    """Pair layout forced: the emission kernels write one column per distinct id (8 / 16 / 32 lanes per row
    at Dp <= 32 / <= 64 / more).  Unpacked, within the f64 bound, and bit-identical to plain rows
    (HFA_COMPACT=0)."""
    monkeypatch.setenv("HFA_PAIR", "2")
    monkeypatch.setenv("HFA_LATENCY_MODE", "0")
    rng = np.random.default_rng(V + 7)
    heads, ids_list = pair_batch(rng, V, PAIR_SHAPES, [5, 9, 32, 33, 41, 57, 64, 65, 120])
    plan, got, dh = run_emission(heads, ids_list, V, DTYPES[dt], view)
    assert_compacted(plan, len(ids_list))
    for i, (h, ids, g) in enumerate(zip(values_of(dh), ids_list, got)):
        check_against_f64(h, ids, V, g, f"compacted utterance {i} (S={len(ids)})")
    monkeypatch.setenv("HFA_COMPACT", "0")
    plan0, got0, _ = run_emission(heads, ids_list, V, DTYPES[dt], view)
    assert plan0.routing()["stored_emission_bytes"] > plan.routing()["stored_emission_bytes"]
    for i, (a, b) in enumerate(zip(got, got0)):
        for j in range(3):
            assert np.array_equal(bits(a[j]), bits(b[j])), f"utterance {i}: compacted != plain rows"


def test_batch_mixing_compacted_plain_and_long_rows(monkeypatch):
    """One batch: compacted rows (pairable), plain rows (adjacent SPs: no pair layout) and S > 256 (CTA
    kernel), so the persistent CTAs switch between row layouts and the gather widths."""
    monkeypatch.setenv("HFA_PAIR", "2")
    monkeypatch.setenv("HFA_LATENCY_MODE", "0")
    V = 63
    rng = np.random.default_rng(99)
    heads, ids_list, n_pair = [], [], 0
    for i in range(60):
        kind = i % 3
        T = int(rng.integers(1, 140))
        if kind == 0:
            ids = make_ids(rng, int(rng.integers(8, 250)), int(rng.integers(2, 60)), V, pairable=True)
            n_pair += 1
        elif kind == 1:
            ids = make_ids(rng, int(rng.integers(8, 200)), int(rng.integers(2, 60)), V)
            ids[1:3] = 0                                           # two adjacent SPs
        else:
            ids = make_ids(rng, int(rng.integers(257, 700)), int(rng.integers(2, 64)), V)
        ids_list.append(ids)
        heads.append(make_head(rng, T, V, ids, STYLES[i % len(STYLES)]))
    plan, got, dh = run_emission(heads, ids_list, V, torch.float32)
    assert_compacted(plan, n_pair)
    for i, (h, ids, g) in enumerate(zip(values_of(dh), ids_list, got)):
        check_against_f64(h, ids, V, g, f"utterance {i} (S={len(ids)})")


# ------------------------------------------------------------------------------------------------
# fused band producer
# ------------------------------------------------------------------------------------------------
def test_fused_equals_three_stage_route_with_many_kept_ids(monkeypatch):
    """hfa_forward_fused (emissions computed in the band kernel's producer warps) against hfa_emission +
    hfa_viterbi_forward at V = 200, where the normaliser runs its generic loop over more than 64 kept ids,
    with rows whose kept logits are all -inf: backpointers, frame confidence, dp on the path, results."""
    monkeypatch.setenv("HFA_LAT_KERNEL", "band")
    V = 200
    rng = np.random.default_rng(2024)
    shapes = [(500, 150), (130, 90), (257, 200), (64, 70), (17, 33), (1, 3), (333, 120)]
    kept = [120, 80, 150, 66, 30, 3, 100]
    ids_list = [make_ids(rng, S, k, V) for (T, S), k in zip(shapes, kept)]
    heads = [make_head(rng, T, V, ids, st) for (T, S), ids, st in
             zip(shapes, ids_list, ["planted", "gauss", "planted", "grid", "dead_rows", "gauss", "neginf_kept"])]
    dh = [torch.from_numpy(h).to(DEV) for h in heads]
    T = np.array([s[0] for s in shapes], np.int32)
    S = np.array([len(i) for i in ids_list], np.int32)
    outs = []
    for fused in (False, True):
        plan = ops.AlignPlan(T, S, np.concatenate(ids_list), V, 0.02)
        rt = plan.routing()
        assert rt["warp_utts"] == 0 and rt["cta_utts"] == 0 and rt["keeps_dp"]
        ws, res = plan.new_workspace(DEV), plan.new_result(DEV)
        plan.upload(ws)
        plan.set_inputs(ws, [h[:, 2:].data_ptr() for h in dh], [V + 2] * len(dh), [1] * len(dh),
                        [h[:, 0].data_ptr() for h in dh], [V + 2] * len(dh))
        if fused:
            ops.forward_fused(ws, plan.handle, _lib.DTYPE_F32)
        else:
            ops.emission(ws, plan.handle, _lib.DTYPE_F32)
            ops.viterbi_forward(ws, plan.handle, None)
        fc = torch.empty(plan.total_frames, dtype=torch.float32, device=DEV)
        dpp = torch.empty(plan.total_frames, dtype=torch.float32, device=DEV)
        ops.backtrace(ws, plan.handle, res, fc, dpp)
        torch.cuda.synchronize()
        outs.append((plan.debug_region(ws, "bp").cpu().numpy().copy(), res.cpu().numpy().copy(),
                     fc.cpu().numpy(), dpp.cpu().numpy()))
    for j in (0, 2, 3):
        assert np.array_equal(outs[0][j].view(np.uint8), outs[1][j].view(np.uint8))
    va, vb = plan.views(outs[0][1]), plan.views(outs[1][1])
    for key in ("status", "n_seg", "end_state", "final_score", "total_conf"):
        assert np.array_equal(va[key].view(np.uint8), vb[key].view(np.uint8)), key
    assert not np.isnan(vb["final_score"]).any()
    assert va["status"][4] == 4                       # the dead rows make that utterance infeasible
    for b in range(plan.n_utt):
        o, k = int(plan.seg_off[b]), int(va["n_seg"][b])
        for key in ("ph_idx_seq", "ph_time_int", "intervals"):
            assert np.array_equal(va[key][o:o + k], vb[key][o:o + k]), (b, key)


# ------------------------------------------------------------------------------------------------
# D. rows whose kept logits are all -inf, end to end
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("route", ["skew-f32", "skew-bf16", "band-fused-f32", "wide-f32"])
def test_row_of_minus_inf_kept_logits_makes_the_utterance_infeasible(route, monkeypatch):
    """decode_batch on an utterance with one frame whose kept logits are all -inf (caller-side masking, f16
    overflow): status 4 (infeasible), as the C oracle gives on oc.emission of the same logits -- not a NaN
    DP.  The other utterances align as the oracle does.  band-fused: the emissions come from the fused band
    producer (decode_batch takes the fused route for unsplit banded batches)."""
    from hubertfa_b200.alignment_decoder import AlignmentDecoder
    if route.startswith("band"):
        monkeypatch.setenv("HFA_LAT_KERNEL", "band")
    V = 300 if route.startswith("wide") else 63
    dtype = torch.bfloat16 if route.endswith("bf16") else torch.float32
    T = np.array([200, 150, 120], np.int32)
    S = np.array([30, 21, 40], np.int32)
    vocab, items = synth.make_batch(T, S, V, seed=515, style="dictionary", planted=True)
    frames = [it["frame"].to(dtype).float() for it in items]
    keep = ef.keep_mask(items[0]["ids"], V)
    frames[0][0, 77, torch.from_numpy(keep)] = -float("inf")
    frames[2][0, 0, torch.from_numpy(ef.keep_mask(items[2]["ids"], V))] = -float("inf")
    dec = AlignmentDecoder(vocab, synth.MELSPEC_50FPS)
    res = dec.decode_batch([f.to(dtype).to(DEV) for f in frames], [it["edge"].to(dtype).to(DEV) for it in items],
                           [it["ph_seq"] for it in items])
    for b, it in enumerate(items):
        x = frames[b][0].numpy()
        e = oc.emission(np.ascontiguousarray(x), it["ids"])
        assert not np.isnan(e).any()
        p = oc.edge_pred(it["edge"][0].to(dtype).float().numpy())
        el, ne = oc.edge_logs(oc.edge_prob(p)[1])
        r = oc.decode(it["ids"], e, el, ne)
        want = 4 if np.isneginf(r["dp_path"][-1]) else 0
        assert int(res.status[b]) == want, f"utterance {b}: status {int(res.status[b])}, oracle {want}"
        if want == 0:
            idx, tim, _ = res.segments(b)
            assert np.array_equal(idx, r["ph_idx_seq"]) and np.array_equal(tim, r["ph_time_int"])
    assert int(res.status[0]) == 4 and int(res.status[2]) == 4 and int(res.status[1]) == 0


# ------------------------------------------------------------------------------------------------
# C. tier 1 on compacted rows
# ------------------------------------------------------------------------------------------------
def _tier1(frames, edges, ids_list, V, sample=None):
    plan, out, inputs = run_core_from_logits(frames, edges, ids_list, V, 0.02, sample)
    for b, (e, el, ne, p) in inputs.items():
        try:
            check_core_against_oracle(ids_list[b], e, el, ne, out[b], p, 0.02)
        except AssertionError as err:
            raise AssertionError(f"utterance {b} (T={e.shape[0]}, S={len(ids_list[b])}): {err}") from err
    return plan


def test_tier1_on_compacted_rows_pair_layout_edge_cases(monkeypatch):
    """The shapes and id patterns of the pair-layout edge cases (leading / trailing SP, words of 1..4 phonemes,
    T = 1 / 2 / tile boundaries), coarse-grid logits (many tied states), emissions from the logits in
    compacted rows: every dp cell, DUMP and production backpointer, path, dp_path, final score and frame
    confidence against the C oracle run on the emissions the DP read."""
    monkeypatch.setenv("HFA_LATENCY_MODE", "0")
    monkeypatch.setenv("HFA_PAIR", "2")
    V = 63
    rng = np.random.default_rng(31337)
    shapes = [(1, 1), (1, 2), (2, 1), (2, 2), (2, 3), (3, 2), (7, 3), (8, 5), (9, 4), (16, 8), (17, 30), (24, 33),
              (25, 64), (40, 65), (33, 100), (64, 128), (70, 150), (50, 200), (41, 213), (90, 256), (300, 90)]
    ids_list, heads = [], []
    for i, (T, S) in enumerate(shapes * 3):
        ids = pairable_ids(rng, S, bool(i & 1), bool(i & 2), 1 + i % 4)
        ids_list.append(ids)
        h = make_head(rng, T, V, ids, "grid" if i % 3 else "gauss")
        if i % 7 == 3:
            h[T // 2, 2:][ef.keep_mask(ids, V)] = -np.inf                # one dead frame: infeasible
        heads.append(h)
    n_pairable = sum(1 for ids in ids_list if ((ids != 0).sum() + (ids[-1] == 0) + 31) // 32 <= 4)
    dh = [torch.from_numpy(h).to(DEV) for h in heads]
    plan = _tier1([h[:, 2:] for h in dh], [h[:, 0] for h in dh], ids_list, V)
    r = plan.routing()
    assert r["pair_utts"] == n_pairable and n_pairable >= 40
    full = 4 * int(sum(int(t) * ((int(s) + 3) // 4 * 4) for t, s in zip(plan.T, plan.S)))
    assert r["stored_emission_bytes"] < full


def test_tier1_on_a_config4_batch():
    """A config-4-sized batch (4096 utterances, 5-30 s, 20-150 phonemes, V = 74), routed by the plan itself:
    every utterance in the pair layout with compacted rows; tier 1 bit-exact on a seeded sample of 256."""
    V = 74
    T, S = synth.sample_shapes(4096, seed=404, min_s=5, max_s=30, s_lo=20, s_hi=150)
    rng = np.random.default_rng(404)
    ids_list = [pairable_ids(rng, int(s), bool(rng.random() < 0.5), bool(rng.random() < 0.5), 4) for s in S]
    g = torch.Generator(device=DEV).manual_seed(404)
    head = 3.0 * torch.randn(int(T.sum()), V + 2, device=DEV, generator=g)
    offs = np.concatenate([[0], np.cumsum(T.astype(np.int64))])
    hv = [head[offs[b]:offs[b + 1]] for b in range(len(T))]
    sample = set(int(b) for b in rng.choice(len(T), 256, replace=False))
    plan = _tier1([h[:, 2:] for h in hv], [h[:, 0] for h in hv], ids_list, V, sample)
    r = plan.routing()
    assert r["pair_utts"] == len(T), r
    assert r["stored_emission_bytes"] < 4 * int((T.astype(np.int64) * ((S + 3) // 4 * 4)).sum())
