"""Timing of AlignmentDecoder.decode on ONE long-form utterance: T = 180 000 frames (an hour at 50 fps),
S = 12 000 phoneme states, V = 63, planted logits already on the device.  CUDA events around each call after a
warm-up; the per-stage times come from the three stage entry points (emission, forward pass, backtrace) on the
same plan.  Prints one JSON line, with the card's name and power limit read in the same run.

    python tools/time_long_form.py [--calls 5] [--T 180000] [--S 12000]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from hubertfa_b200 import _lib, ops, synth  # noqa: E402
from hubertfa_b200.alignment_decoder import AlignmentDecoder  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else "unknown"
    except Exception as e:                       # the measurement still stands; say that the card was not read
        return f"unknown ({e})"


def planted(T, ids, V, seed):
    """[T, V + 2] head output on the device: Gaussian logits, a random monotone alignment planted on top."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    head = torch.randn(T, V + 2, generator=g, device="cuda")
    head[:, 2:] *= 3.0
    head[:, 0] = head[:, 0] * 2.0 - 3.0
    rng = np.random.default_rng(seed)
    cuts = np.sort(rng.choice(np.arange(1, T), size=len(ids) - 1, replace=False))
    state = np.repeat(np.arange(len(ids)), np.diff(np.concatenate([[0], cuts, [T]])))
    head[torch.arange(T, device="cuda"), torch.from_numpy(2 + ids[state]).cuda()] += 6.0
    head[torch.from_numpy(cuts).cuda(), 0] += 8.0
    return head


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--T", type=int, default=180_000)
    ap.add_argument("--S", type=int, default=12_000)
    ap.add_argument("--calls", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_long_form.py measures on a CUDA device; none found")
    V, T, S = 63, a.T, a.S
    vocab = synth.make_vocab(V)
    ph_seq, word_seq, ph2w = synth.make_ph_seq(np.random.default_rng(7), S, V, "dictionary")
    ids = np.array([vocab["vocab"][p] for p in ph_seq], dtype=np.int32)
    head = planted(T, ids, V, seed=11)
    frame, edge = head[None, :, 2:], head[None, :, 0]
    ctc = torch.zeros(1, 16, V, device="cuda")
    dec = AlignmentDecoder(vocab, synth.MELSPEC_50FPS)

    def call():
        return dec.decode(frame, edge, ctc, None, ph_seq, word_seq, ph2w)

    call()                                       # warm-up: module load, workspace, pinned buffers
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    times = []
    for _ in range(a.calls):
        ev[0].record()
        out = call()
        ev[1].record()
        ev[1].synchronize()
        times.append(ev[0].elapsed_time(ev[1]))

    # stages on one plan / workspace, the same kernels decode() launches
    plan = ops.AlignPlan([T], [S], ids, V, dec.frame_length)
    ws, res = plan.new_workspace(head.device), plan.new_result(head.device)
    plan.upload(ws)
    f = head[:, 2:]
    plan.set_inputs(ws, [f.data_ptr()], [f.stride(0)], [f.stride(1)], [head[:, 0].data_ptr()], [head.stride(0)])
    fc = torch.empty(T, device="cuda")
    stages = dict(emission=lambda: ops.emission(ws, plan.handle, _lib.DTYPE_F32),
                  forward=lambda: ops.viterbi_forward(ws, plan.handle, None),
                  backtrace=lambda: ops.backtrace(ws, plan.handle, res, fc, None))
    for fn in stages.values():
        fn()
    torch.cuda.synchronize()
    st = {k: [] for k in stages}
    for _ in range(a.calls):
        for k, fn in stages.items():
            ev[0].record()
            fn()
            ev[1].record()
            ev[1].synchronize()
            st[k].append(ev[0].elapsed_time(ev[1]))
    ms = float(np.median(times))
    print(json.dumps(dict(
        what="AlignmentDecoder.decode, one utterance, logits on the device", T=T, S=S, V=V, cells=T * S,
        calls=a.calls, ms_per_call_median=round(ms, 3), ms_per_call_all=[round(x, 3) for x in times],
        cells_per_s=float(f"{T * S / (ms * 1e-3):.4e}"), workspace_bytes=plan.workspace_bytes,
        peak_device_bytes=torch.cuda.max_memory_allocated(), routing=plan.routing(),
        stage_ms_median={k: round(float(np.median(v)), 3) for k, v in st.items()},
        phonemes=len(out[0]), card=card())))


if __name__ == "__main__":
    main()
