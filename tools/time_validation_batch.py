"""Validation of a whole batch: the per-utterance loop against one decode_batch, and the batched ctc kernel alone.

For the seeded config-2 (256 utterances, V = 63) and config-4 (4096 utterances, V = 74) batches, logits drawn on the
device:
  (a) loop   -- what validation_step does per utterance: decode() + ctc() (forced_alignment.py:407-414);
  (b) batch  -- one decode_batch(..., ctc_logits=..., want_frame_states=True) on the same per-utterance views.
Each is timed with a host clock around work that ends in a device synchronise; (a) and (b) alternate.  Their ctc
ids and paths are compared utterance by utterance.
  (c) kernel -- hfa_ctc_greedy_batch alone (the out_len memset and one kernel), f32 and bf16 logits: CUDA events
around replays of a CUDA graph of many calls, the calls cycling over enough copies of the logits that they do not
fit the 126 MB L2.  Algorithmic bytes = sum T * V * elem (logits, read once) + 8 * sum T (argmax written and read
back), over kernel time, against the data-sheet 7.7 TB/s of one B200.
Prints one JSON line per measurement; the first and last lines name the card, its power limit and SM clock.

    python tools/time_validation_batch.py [--out FILE] [--reps 3]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK = 7.7e12          # B/s, NVIDIA HGX B200 data sheet, one GPU
L2_BYTES = 126 << 20


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), [x.strip() for x in out.stdout.strip().splitlines()[0].split(",")])) \
        if out.returncode == 0 else {"error": out.stderr.strip()}


def make_batch(B, V, seed):
    import torch
    from hubertfa_b200 import synth
    T, S = synth.sample_shapes(B, seed=seed)
    ids = synth.make_ids_batch(T, S, V, seed=seed)
    seqs = [["SP" if i == 0 else f"p{i}" for i in u] for u in ids]
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(seed)
    n = int(T.sum())
    frame = 3.0 * torch.randn(n, V, generator=g, device=dev)
    edge = 2.0 * torch.randn(n, generator=g, device=dev)
    ctc = torch.randn(n, V, generator=g, device=dev)
    return T, S, ids, seqs, frame, edge, ctc


def time_loop_vs_batch(name, B, V, reps, seed):
    import torch
    from hubertfa_b200 import synth
    from hubertfa_b200.alignment_decoder import AlignmentDecoder
    T, S, _, seqs, frame, edge, ctc = make_batch(B, V, seed)
    offs = np.concatenate([[0], np.cumsum(T)])
    fr = [frame[offs[b]:offs[b + 1]][None] for b in range(B)]
    ed = [edge[offs[b]:offs[b + 1]][None] for b in range(B)]
    cc = [ctc[offs[b]:offs[b + 1]][None] for b in range(B)]
    dec = AlignmentDecoder(synth.make_vocab(V), synth.MELSPEC_50FPS)

    def loop(count):
        out = []
        for b in range(count):
            dec.decode(fr[b], ed[b], cc[b], None, seqs[b])
            out.append((dec.ph_idx_seq, dec.ctc()))
        torch.cuda.synchronize()
        return out

    def batch():
        r = dec.decode_batch(fr, ed, seqs, ctc_logits=cc, want_frame_states=True)
        torch.cuda.synchronize()
        return r

    loop(min(B, 32))                                  # warm-up: modules, pinned buffers, allocator
    batch()
    t_loop, t_batch = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        ref = loop(B)
        t_loop.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        res = batch()
        t_batch.append(time.perf_counter() - t0)
    same_ctc = all(np.array_equal(res.ctc(b), ref[b][1]) for b in range(B))
    same_path = all(np.array_equal(res.segments(b)[0], ref[b][0]) for b in range(B))
    return dict(batch=name, utts=B, V=V, sum_T=int(T.sum()), loop_s=[round(x, 4) for x in t_loop],
                batch_s=[round(x, 4) for x in t_batch], loop_s_min=round(min(t_loop), 4),
                batch_s_min=round(min(t_batch), 5), speedup=round(min(t_loop) / min(t_batch), 1),
                ctc_identical=same_ctc, paths_identical=same_path)


def time_ctc_kernel(name, B, V, dtype, seed, calls=40, replays=5):
    import torch
    from hubertfa_b200 import _lib, ops
    T, S, ids, _, _, _, ctc = make_batch(B, V, seed)
    dev = torch.device("cuda")
    ctc = ctc.to(dtype)
    n = int(T.sum())
    elem = ctc.element_size()
    logit_bytes = n * V * elem
    copies = max(1, -(-2 * L2_BYTES // logit_bytes))  # together at least twice the L2
    bufs = [ctc] + [ctc.clone() for _ in range(copies - 1)]
    plan = ops.AlignPlan(T, S, np.concatenate(ids), V, 0.02)
    ws = plan.new_workspace(dev)
    plan.upload(ws)
    offs = np.concatenate([[0], np.cumsum(T)]).astype(np.int64)
    tabs = [torch.from_numpy(plan.ctc_table(x.data_ptr() + offs[:-1] * V * elem, [V] * B, [1] * B)).to(dev)
            for x in bufs]
    i32 = lambda k: torch.empty(k, dtype=torch.int32, device=dev)
    scratch, out, lens = i32(n), i32(n), i32(B)
    code = ops.TORCH_TO_DTYPE[dtype]
    lib = _lib.load()

    def call(i):
        _lib.check(lib.hfa_ctc_greedy_batch(plan.handle, ws.data_ptr(), tabs[i % copies].data_ptr(), V, code,
                                            scratch.data_ptr(), out.data_ptr(), lens.data_ptr(),
                                            int(torch.cuda.current_stream().cuda_stream)), "hfa_ctc_greedy_batch")

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(copies + 2):
            call(i)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    # correctness of the timed configuration against the one-utterance kernel (first 64 utterances)
    lens_h, out_h = lens.cpu().numpy(), out.cpu().numpy()
    ok = all(np.array_equal(out_h[offs[b]:offs[b] + lens_h[b]],
                            ops.ctc_greedy(bufs[(copies + 1) % copies][offs[b]:offs[b + 1]]).cpu().numpy())
             for b in range(min(B, 64)))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(calls):
            call(i)
    graph.replay()
    torch.cuda.synchronize()
    ms = []
    for _ in range(replays):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        graph.replay()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1) / calls)
    alg = logit_bytes + 8 * n
    best = min(ms)
    return dict(kernel="hfa_ctc_greedy_batch", batch=name, utts=B, V=V, dtype=str(dtype).replace("torch.", ""),
                sum_T=n, row_blocks=int(sum((t + 63) // 64 for t in T)), logit_copies=copies,
                ms_per_call=[round(x, 5) for x in ms], ms_min=round(best, 5), algorithmic_bytes=alg,
                TB_per_s=round(alg / (best * 1e-3) / 1e12, 3),
                share_of_7p7TBps=round(alg / (best * 1e-3) / HBM_PEAK, 3), matches_single_kernel=ok)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
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
    for name, B, V in (("c2", 256, 63), ("c4", 4096, 74)):
        emit(time_loop_vs_batch(name, B, V, args.reps, synth.SEED0))
        torch.cuda.empty_cache()
        for dt in (torch.float32, torch.bfloat16):
            emit(time_ctc_kernel(name, B, V, dt, synth.SEED0))
            torch.cuda.empty_cache()
    emit({"card_after": card()})


if __name__ == "__main__":
    main()
