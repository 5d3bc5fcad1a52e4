"""Helpers shared by the GPU parity tests: run the CUDA stages through the C ABI (torch custom ops)
and run the CPU oracle on the same inputs."""
import numpy as np
import torch

from hubertfa_b200 import ops
from oracle import c_oracle as oc
from oracle import hfa_oracle_np as onp


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def run_core_gpu(ids_list, prob_logs, els, nes, ps=None, frame_length=0.02, vocab=4096,
                 dump=True):
    """forward_pass-boundary inputs (per-utterance numpy arrays) -> per-utterance result dicts."""
    dev = torch.device("cuda")
    T = [p.shape[0] for p in prob_logs]
    S = [len(i) for i in ids_list]
    plan = ops.AlignPlan(T, S, np.concatenate(ids_list), vocab, frame_length)
    cat = lambda xs, dt: torch.from_numpy(np.concatenate([np.asarray(x, dtype=dt).reshape(-1) for x in xs])).to(dev)
    pl, el, ne = cat(prob_logs, np.float32), cat(els, np.float32), cat(nes, np.float32)
    pp = cat(ps, np.float32) if ps is not None else None
    return _run_plan(plan, lambda ws: ops.pack_emissions(ws, plan.handle, pl, el, ne, pp), dump)


def run_core_from_logits(frames, edges, ids_list, vocab, frame_length=0.02, sample=None):
    """Tier 1 from logits: hfa_emission fills the workspace from the logits views `frames` / `edges` (CUDA
    tensors, one per utterance), then the DP and backtrace run as in run_core_gpu.  Returns (plan, results,
    inputs): inputs[b] = (emissions [T, S], edge_log, not_edge_log, edge_p) exactly as the DP read them, for
    check_core_against_oracle.  `sample`: the utterances to return (default all)."""
    T = [int(f.shape[0]) for f in frames]
    S = [len(i) for i in ids_list]
    plan = ops.AlignPlan(T, S, np.concatenate(ids_list), vocab, frame_length)
    got = {}

    def fill(ws):
        plan.set_inputs(ws, [f.data_ptr() for f in frames], [f.stride(0) for f in frames],
                        [f.stride(1) for f in frames], [e.data_ptr() for e in edges], [e.stride(0) for e in edges])
        ops.emission(ws, plan.handle, ops.TORCH_TO_DTYPE[frames[0].dtype])
        got["emis"] = ops.unpack_emissions(plan, ws).cpu().numpy()
        got["edge2"] = plan.debug_region(ws, "edge2").cpu().numpy().copy()
        got["edge_p"] = plan.debug_region(ws, "edge_p").cpu().numpy().copy()

    out = _run_plan(plan, fill, True, sample)
    inputs, cell, eo = {}, 0, 0
    for b in range(plan.n_utt):
        if T[b] < 1 or S[b] < 1:
            continue
        if sample is None or b in sample:
            e2 = got["edge2"][eo:eo + T[b]]
            inputs[b] = (got["emis"][cell:cell + T[b] * S[b]].reshape(T[b], S[b]).copy(), e2[:, 0].copy(),
                         e2[:, 1].copy(), got["edge_p"][eo:eo + T[b]].copy())
        cell += T[b] * S[b]
        eo += (T[b] + 15) // 16 * 16
    return plan, out, inputs


def _run_plan(plan, fill, dump, sample=None):
    dev = torch.device("cuda")
    T, S = [int(t) for t in plan.T], [int(s) for s in plan.S]
    # compute-sanitizer is closed on this pool: the workspace and the result blob sit between guard zones
    # filled with a pattern, checked after the kernels have run (an out-of-bounds write of any kernel in any
    # routing fails the test)
    G = 1 << 16
    ws_all = torch.full((G + max(plan.workspace_bytes, 256) + G,), 0xA5, dtype=torch.uint8, device=dev)
    res_all = torch.full((G + plan.result_bytes + G,), 0x5A, dtype=torch.uint8, device=dev)
    ws, res = ws_all[G:G + max(plan.workspace_bytes, 256)], res_all[G:G + plan.result_bytes]
    plan.upload(ws)
    fill(ws)
    dp_dump = torch.full((max(plan.total_cells, 1),), float("nan"), dtype=torch.float32, device=dev) if dump else None
    ops.viterbi_forward(ws, plan.handle, dp_dump)
    bt_dump = None
    if dump:
        # the dump run used the DUMP instantiations of the kernels; keep its backpointers, then run the
        # PRODUCTION instantiation (what decode_batch launches) over the same workspace: its backpointer
        # words and -- where the plan keeps dp -- its dp cells are compared with the oracle as well
        torch.cuda.synchronize()
        bt_dump = []
        for b in range(plan.n_utt):
            try:
                bt_dump.append(ops.unpack_backptr(plan, ws, b).cpu().numpy() if sample is None or b in sample
                               else None)
            except ops.HfaError:                      # invalid utterance: no backpointers
                bt_dump.append(None)
        plan.debug_region(ws, "bp").fill_(-1)
        ops.viterbi_forward(ws, plan.handle, None)
    fc = torch.empty(max(plan.total_frames, 1), dtype=torch.float32, device=dev)
    dpp = torch.empty(max(plan.total_frames, 1), dtype=torch.float32, device=dev)
    ops.backtrace(ws, plan.handle, res, fc, dpp)
    torch.cuda.synchronize()
    for buf, pat, what in ((ws_all, 0xA5, "workspace"), (res_all, 0x5A, "result blob")):
        assert bool((buf[:G] == pat).all()) and bool((buf[-G:] == pat).all()), f"a kernel wrote outside the {what}"
    v = plan.views(res.cpu().numpy())
    fc, dpp = fc.cpu().numpy(), dpp.cpu().numpy()
    dump_h = dp_dump.cpu().numpy() if dump else None
    out, cell = [], 0
    for b in range(plan.n_utt):
        if sample is not None and b not in sample:
            if int(v["status"][b]) in (0, 4):
                cell += T[b] * S[b]
            out.append(None)
            continue
        o, k = int(plan.seg_off[b]), int(v["n_seg"][b])
        f0, f1 = int(plan.frame_off[b]), int(plan.frame_off[b + 1])
        d = dict(status=int(v["status"][b]), n_seg=k, end_state=int(v["end_state"][b]),
                 final_score=v["final_score"][b], total_conf=v["total_conf"][b],
                 ph_idx_seq=v["ph_idx_seq"][o:o + k].copy(), ph_time_int=v["ph_time_int"][o:o + k].copy(),
                 intervals=v["intervals"][o:o + k].copy(), frame_conf=fc[f0:f1], dp_path=dpp[f0:f1])
        if dump and d["status"] in (0, 4):
            n = T[b] * S[b]
            d["dp"] = dump_h[cell:cell + n].reshape(T[b], S[b])
            cell += n
            d["bt"] = bt_dump[b]
            d["bt_prod"] = ops.unpack_backptr(plan, ws, b).cpu().numpy()
            if plan.routing()["keeps_dp"]:
                d["dp_kept"] = ops.unpack_kept_dp(plan, ws, b).cpu().numpy()
        out.append(d)
    return out


def check_core_against_oracle(ids, prob_log, el, ne, g, p=None, frame_length=0.02, full=True):
    """Bit-exact comparison of one utterance's GPU result `g` with the C oracle."""
    r = oc.decode(ids, prob_log, el, ne, full=full)
    assert r["rc"] == 0
    assert g["n_seg"] == len(r["ph_idx_seq"])
    assert np.array_equal(g["ph_idx_seq"], r["ph_idx_seq"])
    assert np.array_equal(g["ph_time_int"], r["ph_time_int"])
    assert g["end_state"] == r["end_state"]
    assert np.array_equal(bits(g["dp_path"]), bits(r["dp_path"]))
    assert bits(g["final_score"]) == bits(r["dp_path"][-1])
    if full and "dp" in g:
        assert np.array_equal(bits(g["dp"]), bits(r["dp"]))
        assert np.array_equal(g["bt"][1:], r["bt"][1:])
        assert (g["bt"][0] == -1).all()
        assert np.array_equal(g["bt_prod"][1:], r["bt"][1:]), "production kernel: backpointers differ"
        if "dp_kept" in g:
            assert np.array_equal(bits(g["dp_kept"]), bits(r["dp"])), "production kernel: kept dp differs"
    fc, tot = oc.confidence(r["dp_path"])
    fin = np.isfinite(fc)
    np.testing.assert_allclose(g["frame_conf"][fin], fc[fin], rtol=2e-6, atol=1e-30)
    assert g["status"] == (4 if np.isneginf(r["dp_path"][-1]) else 0)   # HFA_UTT_INFEASIBLE
    if np.isfinite(tot):
        np.testing.assert_allclose(g["total_conf"], tot, rtol=1e-4)
    else:
        assert np.isnan(g["total_conf"])
    if p is not None:
        iv = oc.intervals(prob_log.shape[0], r["ph_time_int"], p, frame_length)
        assert np.array_equal(g["intervals"], iv)
    return r


def synth_core_inputs(T, S, V, seed, style="dictionary", planted=False):
    """Emissions through the numpy/torch oracle front end (the reference's own third-party calls)."""
    from hubertfa_b200 import synth
    rng = np.random.default_rng(seed)
    vocab = synth.make_vocab(V)
    ph_seq, word_seq, ph2w = synth.make_ph_seq(rng, S, V, style)
    ids = np.array([vocab["vocab"][x] for x in ph_seq], dtype=np.int32)
    frame, edge, _ = synth.make_logits(seed, T, V, ids, planted)
    lp = onp.frame_log_probs(frame, ids, V)
    p = onp.edge_pred(edge)
    _, ep = onp.edge_streams(p)
    el, ne = onp.edge_logs(ep)
    return dict(ids=ids, prob_log=np.ascontiguousarray(lp[:, ids]), el=el, ne=ne, p=p, frame=frame,
                edge=edge, ph_seq=ph_seq, word_seq=word_seq, ph2w=ph2w, vocab=vocab)


def pairable_ids(rng, S, lead, trail, max_word):
    """Random sequence without adjacent SPs: [SP] word SP word ... [SP], words of 1..max_word phonemes."""
    ids = [0] if lead else []
    while len(ids) < S:
        ids += [int(x) for x in rng.integers(1, 30, int(rng.integers(1, max_word + 1)))]
        ids.append(0)
    ids = ids[:S]
    if trail:
        if S >= 2 and ids[-2] == 0:
            ids[-2] = 7
        ids[-1] = 0
    elif ids[-1] == 0 and (S == 1 or ids[-2] != 0):
        ids[-1] = 9 if not (S == 1 and lead) else 0
    return np.array(ids, dtype=np.int32)
