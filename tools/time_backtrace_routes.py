"""Backtrace stage of the kept-dp (latency) plans under both routes: the serial walk out of shared memory
(HFA_BT_WALK=2) against the jump tables (HFA_BT_WALK=0).

For every batch both plans run the same emissions through the forward pass once; then `ops.backtrace` is timed with
CUDA events over many launches, the two routes alternating (A B A B), and the two result blobs are compared byte for
byte.  Batches: single-length batches of 256 utterances (T x S grid) and the bench workloads c1, c2, c3 and m512.
Emissions are random log-probabilities generated on the device (the stage reads backpointers and kept dp only).
Prints one JSON line per batch, the first line names the card, its power limit and SM clock.

    python tools/time_backtrace_routes.py [--launches 200] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GRID_T = [500, 1000, 1500, 2000, 3000, 4000, 6000]
GRID_S = [40, 80, 150, 256]
MODES = ["0", "2"]


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), [x.strip() for x in out.stdout.strip().splitlines()[0].split(",")])) \
        if out.returncode == 0 else {"error": out.stderr.strip()}


def run_batch(name, T, S, V, launches, reps=2):
    import torch
    from hubertfa_b200 import ops, synth
    dev = torch.device("cuda")
    T, S = np.asarray(T, np.int32), np.asarray(S, np.int32)
    ids = np.concatenate(synth.make_ids_batch(T, S, V, seed=synth.SEED0))
    g = torch.Generator(device=dev).manual_seed(1234)
    cells = int((T.astype(np.int64) * S).sum())
    pl = (torch.randn(cells, device=dev, generator=g) * 2.0 - 4.0).contiguous()
    el = torch.log(torch.rand(int(T.sum()), device=dev, generator=g) * 0.98 + 0.01)
    ne = torch.log1p(-torch.exp(el))
    arms = {}
    for mode in MODES:
        os.environ["HFA_BT_WALK"] = mode
        plan = ops.AlignPlan(T, S, ids, V, synth.FRAME_SECONDS)
        ws, res = plan.new_workspace(dev), plan.new_result(dev)
        res.zero_()                      # segment slots past n_seg are never written: compare them as zeros
        plan.upload(ws)
        ops.pack_emissions(ws, plan.handle, pl, el, ne, None)
        ops.viterbi_forward(ws, plan.handle, None)
        n0 = ops.launch_count()
        ops.backtrace(ws, plan.handle, res, None, None)
        torch.cuda.synchronize()
        arms[mode] = dict(plan=plan, ws=ws, res=res, launches=ops.launch_count() - n0, ms=[],
                          walk_utts=plan.routing()["bt_walk_utts"], keeps_dp=plan.routing()["keeps_dp"])
    os.environ.pop("HFA_BT_WALK", None)
    for _ in range(reps):
        for mode in MODES:
            a = arms[mode]
            for _ in range(10):
                ops.backtrace(a["ws"], a["plan"].handle, a["res"], None, None)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(launches):
                ops.backtrace(a["ws"], a["plan"].handle, a["res"], None, None)
            e1.record()
            torch.cuda.synchronize()
            a["ms"].append(e0.elapsed_time(e1) / launches)
    same = bool(torch.equal(arms["0"]["res"], arms["2"]["res"]))
    staged = ((T.astype(np.int64) + 15) // 16) * ((S.astype(np.int64) + 3) // 4 * 4) * 4
    line = dict(batch=name, utts=int(len(T)), max_T=int(T.max()), max_S=int(S.max()), max_staged_bytes=int(staged.max()),
                keeps_dp=arms["0"]["keeps_dp"], results_identical=same)
    for mode in MODES:
        a = arms[mode]
        line[f"walk{mode}"] = dict(ms=[round(x, 5) for x in a["ms"]], ms_min=round(min(a["ms"]), 5),
                                   walk_utts=a["walk_utts"], launches=a["launches"])
    for a in arms.values():
        a["plan"].close()
    del arms
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench
    from hubertfa_b200 import synth
    if not torch.cuda.is_available():
        raise RuntimeError("needs a CUDA device")
    out = open(args.out, "w") if args.out else None

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
            out.flush()

    emit({"card": card(), "torch": torch.__version__})
    for wl in ["c1", "c2", "c3", "m512"]:
        T, S, V, _ = bench.workload_shapes(wl, synth.SEED0)
        emit(run_batch(wl, T, S, V, args.launches if len(T) > 1 or wl == "c1" else 20))
    for t in GRID_T:
        for s in GRID_S:
            emit(run_batch(f"T{t}_S{s}", [t] * 256, [s] * 256, 63, args.launches))
    emit({"card_after": card()})


if __name__ == "__main__":
    main()
