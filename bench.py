#!/usr/bin/env python
"""bench.py -- alignment DP cells/s and audio-hours/s of the B200 forced-alignment decoder.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c1|c3|c4|c4j|c5] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one pass of the whole hot path (emission -> DP -> backtrace/intervals -> compact results on
the host) over one workload of synthetic logits.

N = 1 (default)  BASELINE.json configs[1]: ONE ragged batch of 256 utterances, 5-30 s, 20-150 phonemes, V = 63.
N > 1            BASELINE.json configs[4] ("corpus-scale ... sharded by utterance across 2/4/8 B200"): a FIXED
                 corpus (--corpus utterances, the shapes of configs[1]) sharded over the ranks by cost, every
                 shard streamed in bounded chunks, results gathered on rank 0's host inside the timed region
                 (hubertfa_b200.corpus).  STRONG scaling: the corpus does not grow with N; rank 0 also runs the
                 whole corpus alone in the same process (`n1_same_workload`) and checks that the gathered
                 results are identical to it.  The N = 1 line carries the same corpus as `extra.corpus`.

`value`      device-resident logits -> results in (pinned / shared) host memory, CUDA-event timed, max over
             ranks.  Small batches are launched as ONE CUDA-graph replay per step (ops.GraphedStep).
`e2e`        the same workload from pinned HOST logits through the public API: H2D copies inside the region.
`roofline`   the DP forward stage (the dominant kernels): algorithmic bytes / its CUDA-event time.
`cpu_baseline` / `--impl reference`  the C port of the reference decoder (oracle/hfa_oracle.c; the reference
             itself is Python + numba and cannot travel to the GPU box) on all host cores.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_SETS = 4  # rotating input sets: consecutive steps never touch the same memory (total >> 126 MB L2)

WORKLOADS = {
    #        B     V   (min_s, max_s) (s_lo, s_hi)  description
    "c1": (1, 63, None, None, "configs[0]: single 10 s utterance, T=500, S=40, V=63"),
    "c2": (256, 63, (5, 30), (20, 150), "configs[1]: 256 utterances, 5-30 s, 20-150 phonemes, V=63"),
    "c3": (1, 63, None, None, "configs[2]: one 10 min utterance, T=30000, S=2000, V=63"),
    "c4": (4096, 74, (5, 30), (20, 150), "configs[3]: 4096 mixed-length utterances, jyutping V=74"),
    "c4j": (4096, 39, (5, 30), (20, 150), "configs[3]: 4096 mixed-length utterances, japanese V=39"),
    "c5": (None, 63, (5, 30), (20, 150), "configs[4]: corpus sharded by utterance over the ranks, streamed in chunks, V=63"),
    # sizes between configs[1] and configs[3] (routing threshold experiments)
    "m512": (512, 63, (5, 30), (20, 150), "512 utterances, 5-30 s, 20-150 phonemes, V=63"),
    "m1024": (1024, 63, (5, 30), (20, 150), "1024 utterances, 5-30 s, 20-150 phonemes, V=63"),
    "m2048": (2048, 63, (5, 30), (20, 150), "2048 utterances, 5-30 s, 20-150 phonemes, V=63"),
}
CORPUS_CHUNK_CELLS = 600_000_000     # workspace bound of a corpus chunk (~8000 utterances, ~5.5 GB): measured on
                                     # one B200, 32768 utterances: 9.44 / 8.72 / 8.58 / 8.63 ms per pass with
                                     # chunks of 150M / 300M / 600M / 1200M cells (tools/gpu/r2_chunks2.sh)
DUMP_SAMPLE = 4096                   # corpus utterances whose results --dump-outputs writes


def workload_shapes(name: str, seed: int, corpus: int = 0):
    from hubertfa_b200 import synth
    B, V, dur, srange, desc = WORKLOADS[name]
    if name == "c1":
        T, S = np.array([500], np.int32), np.array([40], np.int32)
    elif name == "c3":
        T, S = np.array([30000], np.int32), np.array([2000], np.int32)
    else:
        if name == "c5":
            B = corpus
        T, S = synth.sample_shapes(B, seed=seed, min_s=dur[0], max_s=dur[1], s_lo=srange[0], s_hi=srange[1])
        if name != "c5":
            # length-bucketed collation (north_star item 4): the batch is packed longest utterance first,
            # the way a length-aware data loader hands it over; both arms see the same batch
            order = np.argsort(-T.astype(np.int64), kind="stable")
            T, S = np.ascontiguousarray(T[order]), np.ascontiguousarray(S[order])
    return T, S, V, desc


def make_config(name, desc, T, S, world, V):
    """The `config` object -- IDENTICAL in our arm and in the reference arm (everything in it follows from the
    workload alone; what only our arm knows -- collation, launch mode, chunking -- goes to `run_config`)."""
    from hubertfa_b200 import synth
    frames = int(T.sum(dtype=np.int64))
    cfg = {"workload": f"{name}: {desc}", "utterances": int(len(T)), "cells": int((T.astype(np.int64) * S).sum()),
           "frames": frames, "frame_seconds": synth.FRAME_SECONDS, "n_ranks": int(world)}
    in_mb = frames * (V + 2) * 4 / 1e6                       # f32 head output [sum T, V+2]
    if name == "c5":
        cfg["l2"] = ("GPU arm: inputs larger than L2 (%.1f GB of logits per rank and pass, 126 MB L2)"
                     % (in_mb / 1e3 / max(int(world), 1)))
    else:
        n_sets = N_SETS if len(T) <= 512 else 2
        cfg["l2"] = ("GPU arm: %d rotating input sets of %.1f MB of logits each, plus their workspaces -- consecutive "
                     "steps touch different memory (inputs alone %.0f MB in rotation, 126 MB L2)"
                     % (n_sets, in_mb, n_sets * in_mb))
    return cfg


def make_head(T, V, seed):
    """Synthetic network-head output [sum T, V+2] f32 on the CPU (col 0 edge, col 1 ctc blank,
    cols 2.. frame logits, networks/task/forced_alignment.py:288-291), SURVEY.md 8d distributions."""
    import torch
    g = torch.Generator().manual_seed(int(seed))
    head = torch.randn(int(np.sum(T)), V + 2, generator=g, dtype=torch.float32)
    head[:, 2:] *= 3.0
    head[:, 0] *= 2.0
    return head


class ClockSampler:
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _once(self):
        nv = self.nv
        try:
            self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
            r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20,
                     "hw_thermal_slowdown": 0x40, "hw_power_brake": 0x80, "sync_boost": 0x10,
                     "applications_clocks": 0x2}
            for k, bit in names.items():
                if r & bit:
                    self.reasons.add(k)
        except Exception:
            pass

    def _loop(self):
        while not self._stop.is_set():
            self._once()
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr is not None:
            self._stop.set()
            self._thr.join()
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ---------------------------------------------------------------------------------------------
# CPU arms (the only place bench.py executes oracle/)
# ---------------------------------------------------------------------------------------------
def cpu_arm(T, S, V, ids_cat, head_np, frame_length, budget_s: float, threads: int = 0):
    """Times the C port of the reference decoder on the host cores; returns (cells/s, sec, reps, threads)."""
    from oracle import c_oracle as oc
    cells = int((T.astype(np.int64) * S).sum())
    nthr = threads or oc.max_threads()
    run = lambda: oc.align_batch(T, S, V, head_np[:, 2:], head_np[:, 0], ids_cat, frame_length, nthr)
    run()  # warm (page faults, thread creation)
    reps, t0 = 0, time.perf_counter()
    while True:
        out = run()
        reps += 1
        dt = time.perf_counter() - t0
        if dt >= budget_s or reps >= 1000:
            break
    assert out["bad"] == 0
    return cells * reps / dt, dt, reps, nthr


def reference_python_note():
    """Throughput of the UNMODIFIED Python + numba reference on a sample of this workload, measured where
    /root/reference exists (the build container; tools/time_reference_python.py) -- it cannot run on the
    GPU box.  Reported beside the C port so the size of the port's head start is visible."""
    p = os.path.join(ROOT, "profiles", "reference_python_cpu.json")
    if os.path.isfile(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def corpus_sample(T, S, ids_list, n):
    """The bounded CPU sample of a corpus workload: its first n utterances."""
    n = min(n, len(T))
    return T[:n], S[:n], ids_list[:n]


def run_reference(args, rank, world):
    """--impl reference: the CPU implementation of the path on this box's host cores (rank 0 only)."""
    if rank != 0:
        return
    from hubertfa_b200 import synth
    from oracle import c_oracle as oc
    name = args.workload or ("c2" if args.gpus <= 1 else "c5")
    T, S, V, desc = workload_shapes(name, synth.SEED0, args.corpus)
    ids_list = (synth.make_ids_corpus(S, V, seed=synth.SEED0) if name == "c5"
                else synth.make_ids_batch(T, S, V, seed=synth.SEED0))
    cfg = make_config(name, desc, T, S, args.gpus, V)
    sample = "the full batch"
    if name == "c5":      # bounded sample of the corpus: its first 2048 utterances
        T, S, ids_list = corpus_sample(T, S, ids_list, 2048)
        sample = f"the first {len(T)} utterances of the corpus"
    ids_cat = np.concatenate(ids_list)
    head = make_head(T, V, synth.SEED0).numpy()
    cells = int((T.astype(np.int64) * S).sum())
    frames = int(T.sum())
    nthr = oc.max_threads()
    run = lambda: oc.align_batch(T, S, V, head[:, 2:], head[:, 0], ids_cat, synth.FRAME_SECONDS, nthr)
    for _ in range(args.warmup):
        run()
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        out = run()
        times.append(time.perf_counter() - t0)
    assert out["bad"] == 0
    if args.dump_outputs:
        seg = segment_slots(out["seg_off"], out["n_seg"])
        write_outputs(args.dump_outputs, {"status": out["status"], "n_seg": out["n_seg"], "total_conf": out["total_conf"],
                                          "ph_idx_seq": out["ph_idx_seq"][seg], "ph_time_int": out["ph_time_int"][seg],
                                          "intervals": out["intervals"].reshape(-1, 2)[seg]})
    k = len(times)
    sec = float(np.sum(times))
    val = cells * k / sec
    line = {
        "impl": "reference", "metric": "dp_cells_per_s", "value": val, "unit": "cells/s",
        "n_gpus": args.gpus, "steps": k, "warmup": args.warmup, "ms_per_step": 1e3 * sec / k,
        "higher_is_better": True, "scaling": "weak" if args.gpus <= 1 else "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "audio_hours_per_s": frames * synth.FRAME_SECONDS / 3600 * k / sec,
        "config": cfg,
        "cpu_baseline": {"value": val, "unit": "cells/s", "cores": nthr, "kind": "port",
                         "sample": f"{k} passes over {sample} ({cells} cells per pass), C port of "
                                   "tools/alignment_decoder.py (oracle/hfa_oracle.c), one utterance per thread",
                         "reference_python": reference_python_note()},
        "e2e": {"value": val, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def verify_against_oracle(T, S, V, ids_list, head_np, row_off, get_result, sample_idx, frame_length):
    """Compares the GPU results of `sample_idx` utterances with the C oracle run on the same logits.
    get_result(b) -> (ph_idx_seq, ph_time_int).  Returns a small report for the JSON line."""
    from oracle import c_oracle as oc
    Ts, Ss = T[sample_idx], S[sample_idx]
    rows = np.concatenate([np.arange(row_off[b], row_off[b] + T[b]) for b in sample_idx])
    sub = np.ascontiguousarray(head_np[rows])
    ref = oc.align_batch(Ts, Ss, V, sub[:, 2:], sub[:, 0], np.concatenate([ids_list[b] for b in sample_idx]), frame_length)
    equal = 0
    for j, b in enumerate(sample_idx):
        o, k = int(ref["seg_off"][j]), int(ref["n_seg"][j])
        idx, tim = get_result(int(b))
        equal += int(len(idx) == k and np.array_equal(idx, ref["ph_idx_seq"][o:o + k])
                     and np.array_equal(tim, ref["ph_time_int"][o:o + k]))
    return {"sample_utterances": int(len(sample_idx)), "paths_equal_to_oracle": int(equal),
            "note": "paths of the last timed step vs oracle/hfa_oracle.c on the same logits; a difference can "
                    "only be a few-ulp near-tie between the two softmax implementations (tests/: tier 2)"}


def segment_slots(seg_off, n_seg):
    """Result-blob slots that hold segments: utterance b owns the slots from seg_off[b] on, and the first n_seg[b]
    of them are written (the rest are not, so they never go into a dump)."""
    return np.concatenate([np.zeros(0, np.int64)] + [np.arange(o, o + k, dtype=np.int64) for o, k in zip(seg_off, n_seg)])


def write_outputs(path, arrays: dict) -> None:
    """--dump-outputs: DIR/<name>.npy per array; integers are stored as float64 (exactly) so that every file is
    float32 or float64."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a if a.dtype.kind == "f" else a.astype(np.float64)))


def corpus_outputs(cp, host, n_utt: int) -> dict:
    """--dump-outputs of the corpus arm: the results of a fixed, seeded sample of DUMP_SAMPLE utterances (all of
    them would be hundreds of MB at the default corpus size)."""
    from hubertfa_b200.corpus import read_results
    utt = np.sort(np.random.default_rng(0).choice(n_utt, size=min(n_utt, DUMP_SAMPLE), replace=False))
    res = read_results(cp, host, utt)
    r = [res[int(b)] for b in utt]
    return {"utterance": utt, "status": [x["status"] for x in r], "n_seg": [len(x["ph_idx_seq"]) for x in r],
            "final_score": np.array([x["final_score"] for x in r], np.float32),
            "total_conf": np.array([x["total_conf"] for x in r], np.float32),
            "ph_idx_seq": np.concatenate([x["ph_idx_seq"] for x in r]),
            "ph_time_int": np.concatenate([x["ph_time_int"] for x in r]),
            "intervals": np.concatenate([x["intervals"] for x in r])}


def kernel_source_stamp():
    h = hashlib.sha1()
    for f in ("hfa_dp.cu", "hfa_dp_skew.cu", "hfa_common.cuh"):
        h.update(open(os.path.join(ROOT, "hubertfa_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:12]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--corpus", type=int, default=100000, help="utterances of the corpus workload (c5)")
    ap.add_argument("--corpus-chunk-cells", type=int, default=0, help="DP cells per corpus chunk (0: automatic)")
    ap.add_argument("--corpus-streams", type=int, default=0, help="streams the corpus chunks alternate over (0: default)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the e2e leg of the corpus arm")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra passes (c4 roofline, corpus, replicas)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-graph", action="store_true", help="launch the kernels eagerly instead of one graph replay")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--e2e-chunks", type=int, default=0,
                    help="equal-sized upload/compute chunks of the e2e leg (0: the library's default shares)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32 / "
                         "float64; the corpus workload: a fixed sample of %d utterances)" % DUMP_SAMPLE)
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.steps is None:
        args.steps = 400 if max(world, args.gpus) <= 1 else 20
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup is None:
        args.warmup = 10 if max(world, args.gpus) <= 1 else 3
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from hubertfa_b200 import ops, synth, _lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: hubertfa_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    try:        # pin this rank to the CPUs next to its GPU (matters for the host-driven e2e leg at N > 1)
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local_rank))
    except Exception:
        pass
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def all_max(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        if world > 1:
            dist.barrier()

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        hbm_peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json (measured copy)"
    else:
        hbm_peak, peak_src = 6650.0, "fallback of B200_PROFILING.md"
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.isfile(tpath):
        traffic = json.load(open(tpath))
    stamp = kernel_source_stamp()

    # -----------------------------------------------------------------------------------------
    # one ragged batch (configs[0..3]): every rank aligns its own batch of the same shape
    # -----------------------------------------------------------------------------------------
    def measure_batch(workload: str, steps: int, warmup: int, do_e2e: bool, seed_rank: int, dump: bool = False):
        seed = synth.SEED0 + 100003 * seed_rank
        T, S, V, desc = workload_shapes(workload, seed)
        ids_list = synth.make_ids_batch(T, S, V, seed=seed)
        ids_cat = np.concatenate(ids_list)
        n_sets = N_SETS if len(T) <= 512 else 2
        heads_host = [make_head(T, V, seed + 17 * i).pin_memory() for i in range(n_sets)]
        heads_dev = [h.to(dev) for h in heads_host]
        plan = ops.AlignPlan(T, S, ids_cat, V, synth.FRAME_SECONDS)
        wss = [plan.new_workspace(dev) for _ in range(n_sets)]
        ress = [plan.new_result(dev) for _ in range(n_sets)]
        host_res = [torch.empty(plan.result_bytes, dtype=torch.uint8, pin_memory=True) for _ in range(n_sets)]
        row0 = plan.frame_off[:-1]
        dt = _lib.DTYPE_F32

        for ws, head in zip(wss, heads_dev):
            base, st = head.data_ptr(), head.stride(0)
            plan.upload(ws)
            plan.set_inputs(ws, base + (row0 * st + 2) * 4, np.full(plan.n_utt, st), np.ones(plan.n_utt),
                            base + row0 * st * 4, np.full(plan.n_utt, st))
        torch.cuda.synchronize()
        rt = plan.routing()

        # --- value: one CUDA-graph replay per step (or the eager launches) ---
        # big batches: launch overhead is nothing there, but their result blob is megabytes -- launched eagerly
        # with the download on a side stream so that it overlaps the next step's kernels
        use_graph = not args.no_graph and len(T) <= 512
        n0 = ops.launch_count()
        ops.align_batch(wss[0], plan.handle, dt, ress[0], None)
        torch.cuda.synchronize()
        launches_per_step = ops.launch_count() - n0
        graphs = None
        if use_graph:
            graphs = [ops.GraphedStep(plan, wss[k], ress[k], host_res[k], dt) for k in range(n_sets)]

        d2h_stream = torch.cuda.Stream()
        d2h_done = [None] * n_sets

        def step(i):
            k = i % n_sets
            if graphs is not None:
                graphs[k].replay()
                return
            cur = torch.cuda.current_stream()
            if d2h_done[k] is not None:          # the last download out of this result buffer
                cur.wait_event(d2h_done[k])
            ops.align_batch(wss[k], plan.handle, dt, ress[k], None)
            ready = torch.cuda.Event()
            ready.record()
            with torch.cuda.stream(d2h_stream):
                d2h_stream.wait_event(ready)
                host_res[k].copy_(ress[k], non_blocking=True)
                d2h_done[k] = torch.cuda.Event()
                d2h_done[k].record()

        for i in range(warmup):
            step(i)
        torch.cuda.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clocks = ClockSampler(local_rank)
        clocks.start()
        torch.cuda.synchronize()
        e0.record()
        for i in range(steps):
            step(i)
        torch.cuda.current_stream().wait_stream(d2h_stream)      # the last download is inside the region
        e1.record()
        if clocks.nv is not None:
            clocks._once()           # the queue is still draining: at least one sample under load even for tiny K
        torch.cuda.synchronize()
        clk = clocks.stop()
        ms = all_max(e0.elapsed_time(e1))
        barrier()

        # --- per-stage times (eager launches, CUDA events between the stages) for the roofline ---
        n_stage = min(steps, 100)
        fused = False
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(n_stage)]
        for i in range(3 + n_stage):
            k = i % n_sets
            ev = evs[i - 3] if i >= 3 else None
            if ev:
                ev[0].record()
            ops.emission(wss[k], plan.handle, dt)
            if ev:
                ev[1].record()
            ops.viterbi_forward(wss[k], plan.handle, None)
            if ev:
                ev[2].record()
            ops.backtrace(wss[k], plan.handle, ress[k], None, None)
            if ev:
                ev[3].record()
        torch.cuda.synchronize()
        st_ms = np.array([[ev[j].elapsed_time(ev[j + 1]) for j in range(3)] for ev in evs]).mean(axis=0)

        # --- results of the last timed step vs the oracle (a sample) ---
        kk = (steps - 1) % n_sets
        v = plan.views(host_res[kk].numpy())
        assert (v["status"] == 0).all() and (v["n_seg"] > 0).all()
        outputs = None
        if dump:
            seg = segment_slots(plan.seg_off[:-1], v["n_seg"])
            outputs = {k: v[k].copy() for k in ("status", "n_seg", "end_state", "final_score", "total_conf")}
            outputs.update({k: v[k][seg] for k in ("ph_idx_seq", "ph_time_int", "intervals")})
        verified = None
        if rank == 0:
            sample = np.unique(np.linspace(0, len(T) - 1, min(16, len(T))).astype(np.int64))

            def get(b):
                o, k = int(plan.seg_off[b]), int(v["n_seg"][b])
                return v["ph_idx_seq"][o:o + k], v["ph_time_int"][o:o + k]

            verified = verify_against_oracle(T, S, V, ids_list, heads_host[kk].numpy(), row0, get, sample,
                                             synth.FRAME_SECONDS)

        e2e = None
        if do_e2e:
            from hubertfa_b200.pipeline import BufferPool, HostBatchAligner
            pool = BufferPool(dev)

            def e2e_step(i):
                # collation (5 plans, longest utterances first) + chunked H2D overlapped with the
                # kernels + D2H of the compact results, from pinned host logits
                al = HostBatchAligner(T, S, ids_cat, V, synth.FRAME_SECONDS, V + 2,
                                      n_chunks=args.e2e_chunks or None, device=dev, pool=pool)
                out = al.run(heads_host[i % n_sets])
                if not out.all_ok():             # the step's results are read on the host, every step
                    raise RuntimeError("e2e: an utterance was not aligned")
                return out

            for i in range(3):
                e2e_step(i)
            torch.cuda.synchronize()
            barrier()
            t0 = time.perf_counter()
            for i in range(steps):
                e2e_step(i)
            torch.cuda.synchronize()
            e2e_s = all_max(time.perf_counter() - t0)
            e2e = {"value": None, "unit": "cells/s", "seconds": e2e_s,
                   "h2d_bytes_per_step": int(heads_host[0].numel() * 4),
                   "d2h_bytes_per_step": int(plan.result_bytes), "ms_per_step": 1e3 * e2e_s / steps,
                   "api": "hubertfa_b200.pipeline.HostBatchAligner.run(pinned host logits): upload cut by rows "
                          "(30/28/22/12/8 % of the bytes), the DMA of piece i+1 overlaps collation and kernels of "
                          "the utterances completed by piece i"}
        alg = plan.algorithmic_bytes(dt)
        words = int((((T + 15) // 16).astype(np.int64) * S).sum())
        alg_8d = int(plan.total_cells * 4 + plan.total_frames * 8 + words * 4)     # SURVEY 8(d): 4.25 B/cell
        # what the kernels are DESIGNED to move: big batches in the pair layout store one emission column per
        # distinct phoneme id (hfa_plan_stored_emission_bytes), fewer than the 4 B per cell of SURVEY 8(d)
        stored = int(rt.get("stored_emission_bytes", plan.total_cells * 4))
        design = {"dp": int(alg["dp"] - plan.total_cells * 4 + stored),
                  "emission": int(alg["emission"] - plan.total_cells * 4 + stored)}
        return dict(fused=fused, T=T, S=S, V=V, desc=desc, ids_cat=ids_cat, head0=heads_host[0], ms=ms, st_ms=st_ms,
                    routing=rt, cells=plan.total_cells, frames=plan.total_frames, clk=clk,
                    launches=launches_per_step * steps,
                    launch_mode=("cuda graph replay, one launch per step" if use_graph
                                 else "eager launches, result download on a side stream"),
                    e2e=e2e, alg=alg, alg_8d=alg_8d, design=design, verified=verified, n_sets=n_sets, outputs=outputs,
                    bytes_per_set=int(heads_host[0].numel() * 4 + plan.workspace_bytes))

    def roofline(m, wl):
        dp_s = m["st_ms"][1] * 1e-3
        ach = m["alg_8d"] / dp_s / 1e9
        ach_kept = m["alg"]["dp"] / dp_s / 1e9
        tr = None
        tr_note = "no ncu figure for this workload in profiles/roofline_traffic.json"
        if traffic and wl in traffic:
            if traffic.get("kernel_source_stamp") == stamp:
                tr = traffic[wl].get("dp_dram_bytes_per_step")
                tr_note = f"ncu dram__bytes of the DP launch, {traffic.get('captured', 'profiles/')}"
            else:
                tr_note = ("profiles/roofline_traffic.json was captured for other kernel sources (stamp "
                           f"{traffic.get('kernel_source_stamp')} != {stamp}): not reported")
        rt = m["routing"]
        names = []
        if rt["band_warps"]:
            names.append((f"hfa_dp_skew_kernel<D={rt['skew_d']}> ({rt['band_warps']} strips, one warp each, several per utterance)"
                          if rt["skew_d"] and rt["band_k"] == 1 else
                          f"hfa_dp_band_kernel<{rt['band_k']}> ({rt['band_warps']} compute warps, several per utterance)"))
        if rt["big_band_warps"]:
            names.append((f"hfa_dp_skew_kernel<D={rt['skew_d']}> ({rt['big_band_warps']} strips, S > 256)"
                          if rt["skew_d"] and rt["big_band_k"] == 1 else
                          f"hfa_dp_band_kernel<{rt['big_band_k']}> ({rt['big_band_warps']} compute warps, S > 256)"))
        if rt["warp_utts"]:
            names.append(f"hfa_dp_warp_any_kernel ({rt['warp_utts']} utterances, one warp each)")
        if rt["cta_utts"]:
            names.append(f"hfa_dp_cta_kernel ({rt['cta_utts']} utterances)")
        em_ms = float(m["st_ms"][0])
        return {"bound": "hbm", "kernel": " + ".join(names) + " = the DP forward stage of one step",
                "keeps_dp": rt["keeps_dp"],
                "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": tr,
                "traffic_note": tr_note, "peak_source": peak_src,
                "algorithmic_bytes_per_step": m["alg_8d"],
                "accounting": "SURVEY 8(d): 4 B/cell emissions read + 8 B/frame edge logs + 2-bit backpointers "
                              "written (4.25 B/cell); `with_kept_dp` adds the 4 B/cell dp store of latency plans",
                "with_kept_dp": {"algorithmic_bytes_per_step": m["alg"]["dp"], "achieved": ach_kept,
                                 "frac": ach_kept / hbm_peak},
                "design_bytes": {"note": "bytes the DP stage is designed to move in this routing: emission rows as "
                                         "stored (one column per distinct phoneme id in the pair layout of big "
                                         "batches, else 4 B/cell) + edge logs + backpointers (+ kept dp)",
                                 "bytes_per_step": m["design"]["dp"],
                                 "achieved": m["design"]["dp"] / dp_s / 1e9,
                                 "frac": m["design"]["dp"] / dp_s / 1e9 / hbm_peak},
                "pair_layout_utterances": rt.get("pair_utts", 0),
                "stage_ms": {"emission": float(m["st_ms"][0]), "dp": float(m["st_ms"][1]),
                             "backtrace": float(m["st_ms"][2])},
                "stage_gbs": {"emission": (m["design"]["emission"] / (em_ms * 1e-3) / 1e9) if em_ms > 1e-4 else None,
                              "dp": ach, "backtrace": m["alg"]["backtrace"] / (m["st_ms"][2] * 1e-3) / 1e9}}

    # -----------------------------------------------------------------------------------------
    # the corpus (configs[4]): sharded by cost, chunked, gathered on rank 0's host
    # -----------------------------------------------------------------------------------------
    def measure_corpus(n_utt: int, steps: int, warmup: int, ranks: int, my_rank: int, do_e2e: bool, tag: str,
                       dump: bool = False):
        """ranks = 1: this process alone runs the whole corpus (the strong-scaling reference)."""
        from hubertfa_b200.corpus import CorpusAligner, CorpusPlan, SharedHostBuffer, all_status_ok, read_results
        T, S, V, desc = workload_shapes("c5", synth.SEED0, n_utt)
        ids_list = synth.make_ids_corpus(S, V, seed=synth.SEED0)
        cp = CorpusPlan(T, S, ids_list, V, synth.FRAME_SECONDS, ranks, args.corpus_chunk_cells or CORPUS_CHUNK_CELLS)
        row_off = np.concatenate([[0], np.cumsum(T.astype(np.int64))])
        # the SAME logits on every rank: the whole corpus from one seeded device generator (3.7 GB at the
        # default size); a rank only ever reads its own utterances' rows
        g = torch.Generator(device=dev).manual_seed(synth.SEED0)
        head = torch.empty(int(row_off[-1]), V + 2, device=dev, dtype=torch.float32)
        rows_per = 4_000_000
        for r0 in range(0, head.shape[0], rows_per):
            head[r0:r0 + rows_per].normal_(generator=g)
        head[:, 2:] *= 3.0
        head[:, 0] *= 2.0
        name = f"hfa_bench_{os.environ.get('MASTER_PORT', '0')}_{os.getppid() if ranks > 1 else os.getpid()}_{tag}"
        multi = ranks > 1
        if multi:
            host = None
            if my_rank == 0:
                host = SharedHostBuffer(name, cp.total_result_bytes, create=True)
            barrier()
            if my_rank != 0:
                host = SharedHostBuffer(name, cp.total_result_bytes, create=False)
        else:
            host = SharedHostBuffer(name, cp.total_result_bytes, create=True)
        al = CorpusAligner(cp, my_rank, dev, head, row_off, host, n_streams=args.corpus_streams or 2)

        def sync_all():
            torch.cuda.synchronize()
            if multi:
                barrier()

        for _ in range(warmup):
            al.run()
            al.join()
        sync_all()
        clocks = ClockSampler(local_rank)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clocks.start()
        e0.record()
        for _ in range(steps):
            al.run()
            al.join()
        e1.record()
        torch.cuda.synchronize()              # this rank's results are in the shared host segment
        clk = clocks.stop()
        ms = e0.elapsed_time(e1)
        if multi:
            ms = all_max(ms)                  # the gather is complete when the slowest rank is done
            barrier()
        out = dict(cp=cp, T=T, S=S, V=V, desc=desc, ms=ms, clk=clk, launches=al.launches_per_pass * steps,
                   chunks=[len(c) for c in cp.chunks], d2h=int(sum(c["plan"].result_bytes for c in al.chunks)))
        torch.cuda.synchronize()
        if my_rank == 0:
            out["ok"] = all_status_ok(cp, host)
            sample = np.unique(np.linspace(0, n_utt - 1, 24).astype(np.int64))
            out["results"] = read_results(cp, host, sample)
            out["sample"] = sample
            if dump:          # before the e2e leg below writes its own passes into the same host segment
                out["outputs"] = corpus_outputs(cp, host, n_utt)
            sub_rows = torch.cat([head[row_off[b]:row_off[b + 1]] for b in sample]).cpu().numpy()
            sub_off = np.concatenate([[0], np.cumsum(T[sample].astype(np.int64))])
            res = out["results"]
            out["verified"] = verify_against_oracle(
                T[sample], S[sample], V, [ids_list[b] for b in sample], sub_rows, sub_off,
                lambda j: (res[int(sample[j])]["ph_idx_seq"], res[int(sample[j])]["ph_time_int"]),
                np.arange(len(sample)), synth.FRAME_SECONDS)
        e2e = None
        al.close()
        del al
        torch.cuda.empty_cache()
        if do_e2e and not args.no_e2e:
            # pinned host copy of this rank's rows -> device staging -> the same pass, every step
            mine = np.sort(cp.shards[my_rank])
            rows = torch.cat([torch.arange(row_off[b], row_off[b + 1]) for b in mine]).to(dev)
            host_rows = head[rows].cpu().pin_memory()
            stage = torch.empty_like(head[rows])
            my_off = np.zeros(n_utt, dtype=np.int64)
            my_off[mine] = np.concatenate([[0], np.cumsum(T[mine].astype(np.int64))])[:-1]
            al2 = CorpusAligner(cp, my_rank, dev, stage, my_off, host, n_streams=args.corpus_streams or 2)
            n_piece = 8
            cuts = [int(x) for x in np.linspace(0, stage.shape[0], n_piece + 1)]

            def e2e_pass():
                for a, b in zip(cuts[:-1], cuts[1:]):
                    stage[a:b].copy_(host_rows[a:b], non_blocking=True)
                al2.run()
                al2.join()

            # ceiling of the box: every rank copies its pinned rows once, all at the same time
            sync_all()
            t0 = time.perf_counter()
            stage.copy_(host_rows, non_blocking=True)
            torch.cuda.synchronize()
            h2d_s = time.perf_counter() - t0
            if multi:
                h2d_s = all_max(h2d_s)
            for _ in range(2):
                e2e_pass()
            sync_all()
            t0 = time.perf_counter()
            for _ in range(steps):
                e2e_pass()
            torch.cuda.synchronize()
            e2e_s = time.perf_counter() - t0
            if multi:
                e2e_s = all_max(e2e_s)
            tot_bytes = float(host_rows.numel() * 4)
            if multi:
                t = torch.tensor([tot_bytes], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.SUM)
                tot_bytes = float(t.item())
            e2e = {"value": cp.cells * steps / e2e_s, "unit": "cells/s", "ms_per_step": 1e3 * e2e_s / steps,
                   "h2d_bytes_per_step": int(tot_bytes), "d2h_bytes_per_step": int(cp.total_result_bytes),
                   "h2d_ceiling": {"aggregate_gbs": tot_bytes / h2d_s / 1e9, "ms": 1e3 * h2d_s,
                                   "how": "every rank copies its pinned logits once, concurrently (one "
                                          "cudaMemcpyAsync each), max over ranks"},
                   "frac_of_h2d_ceiling": (1e3 * h2d_s) / (1e3 * e2e_s / steps),
                   "api": "hubertfa_b200.corpus.CorpusAligner.run() behind 8 H2D pieces of this rank's pinned "
                          "logits per step; results D2H into the shared host segment rank 0 reads"}
            al2.close()
            if multi:
                barrier()
        out["e2e"] = e2e
        out["host"] = host
        return out

    # =========================================================================================
    if world == 1 and (args.workload or "c2") != "c5":
        wl = args.workload or "c2"
        m = measure_batch(wl, args.steps, args.warmup, do_e2e=True, seed_rank=0, dump=bool(args.dump_outputs))
        if args.dump_outputs:
            write_outputs(args.dump_outputs, m["outputs"])
        sec = m["ms"] * 1e-3
        m["e2e"]["value"] = m["cells"] * args.steps / m["e2e"].pop("seconds")
        line = {
            "metric": "dp_cells_per_s", "value": m["cells"] * args.steps / sec, "unit": "cells/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": m["ms"] / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "audio_hours_per_s": m["frames"] * synth.FRAME_SECONDS / 3600 * args.steps / sec,
            "config": make_config(wl, m["desc"], m["T"], m["S"], 1, m["V"]),
            "run_config": {
                "collation": "batch packed longest utterance first",
                "launch_mode": m["launch_mode"],
                "l2": f"{m['n_sets']} rotating input+workspace sets of {m['bytes_per_set'] / 1e6:.0f} MB "
                      "(consecutive steps touch different memory)"},
            "clocks": m["clk"], "e2e": m["e2e"], "gpu_launches": int(m["launches"]),
            "roofline": roofline(m, wl), "verified": m["verified"],
        }
        if not args.no_cpu:
            v, dt_s, reps, nthr = cpu_arm(m["T"], m["S"], m["V"], m["ids_cat"], m["head0"].numpy(),
                                          synth.FRAME_SECONDS, args.cpu_seconds)
            line["cpu_baseline"] = {"value": v, "unit": "cells/s", "cores": nthr, "kind": "port",
                                    "sample": f"{reps} passes over the full {wl} batch in {dt_s:.1f} s, "
                                              "C port of tools/alignment_decoder.py (oracle/hfa_oracle.c), "
                                              "one utterance per thread",
                                    "reference_python": reference_python_note()}
        else:
            line["cpu_baseline"] = None
        if not args.no_extra and wl == "c2":
            del m
            torch.cuda.empty_cache()
            # the machine-filling configuration (configs[3]) for the roofline: same code, 16x the batch
            x = measure_batch("c4", 10, 3, do_e2e=False, seed_rank=0)
            xs = x["ms"] * 1e-3
            line["extra"] = {"c4": {"workload": f"c4: {x['desc']}", "value": x["cells"] * 10 / xs,
                                    "unit": "cells/s", "ms_per_step": x["ms"] / 10,
                                    "audio_hours_per_s": x["frames"] * synth.FRAME_SECONDS / 3600 * 10 / xs,
                                    "roofline": roofline(x, "c4"), "clocks": x["clk"], "verified": x["verified"]}}
            del x
            torch.cuda.empty_cache()
            # the corpus the N > 1 arms shard (configs[4]), on this one GPU: the strong-scaling reference
            c = measure_corpus(args.corpus, 5, 3, 1, 0, do_e2e=False, tag="x")
            cs = c["ms"] * 1e-3
            line["extra"]["corpus"] = {"workload": f"c5: {c['desc']}", "utterances": args.corpus,
                                       "cells": c["cp"].cells, "value": c["cp"].cells * 5 / cs, "unit": "cells/s",
                                       "ms_per_step": c["ms"] / 5, "chunks": c["chunks"][0],
                                       "audio_hours_per_s": c["cp"].frames * synth.FRAME_SECONDS / 3600 * 5 / cs,
                                       "all_status_ok": c["ok"], "verified": c["verified"]}
            c["host"].close()
        print(json.dumps(line), flush=True)
        return

    # ---- the corpus arm: N ranks (or --workload c5 on one GPU) ----
    c = measure_corpus(args.corpus, args.steps, args.warmup, world, rank, do_e2e=True, tag="m",
                       dump=bool(args.dump_outputs))
    cp = c["cp"]
    sec = c["ms"] * 1e-3
    line = None
    if rank == 0:
        line = {
            "metric": "dp_cells_per_s", "value": cp.cells * args.steps / sec, "unit": "cells/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": c["ms"] / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "audio_hours_per_s": cp.frames * synth.FRAME_SECONDS / 3600 * args.steps / sec,
            "config": make_config("c5", c["desc"], c["T"], c["S"], world, c["V"]),
            "run_config": {
                "sharding": "shard_by_cost (LPT over T*S) -> chunks of <= %d cells -> hfa_align_batch per chunk on two "
                            "alternating streams -> D2H into a shared pinned host segment -> barrier: rank 0 holds "
                            "all results; no collective on the data path" % CORPUS_CHUNK_CELLS,
                "chunks_per_rank": [len(x) for x in cp.chunks],
                "cells_per_rank": [cp.cells_of_rank(r) for r in range(world)],
                "logits": "the whole corpus generated on every GPU from one seeded device generator; a rank reads only "
                          "its own utterances (inputs larger than L2: %.1f GB per rank)"
                          % (cp.frames * (c["V"] + 2) * 4 / world / 1e9)},
            "clocks": c["clk"], "e2e": c["e2e"], "gpu_launches": int(c["launches"]),
            "all_status_ok": c["ok"], "verified": c["verified"], "cpu_baseline": None,
        }
    if rank == 0 and args.dump_outputs:
        write_outputs(args.dump_outputs, c["outputs"])
    first = c.get("results")
    sample = c.get("sample")
    c["host"].close()
    del c
    torch.cuda.empty_cache()
    if world > 1 and not args.no_extra:
        # strong-scaling reference inside the same run: rank 0 alone aligns the whole corpus; the other ranks wait
        if rank == 0:
            one = measure_corpus(args.corpus, max(3, args.steps // 4), 2, 1, 0, do_e2e=False, tag="s")
            k1 = max(3, args.steps // 4)
            v1 = one["cp"].cells * k1 / (one["ms"] * 1e-3)
            same = all(np.array_equal(first[int(b)]["ph_idx_seq"], one["results"][int(b)]["ph_idx_seq"]) and
                       np.array_equal(first[int(b)]["ph_time_int"], one["results"][int(b)]["ph_time_int"]) and
                       np.array_equal(first[int(b)]["intervals"], one["results"][int(b)]["intervals"]) and
                       first[int(b)]["final_score"] == one["results"][int(b)]["final_score"] for b in sample)
            line["n1_same_workload"] = {"value": v1, "unit": "cells/s", "ms_per_step": one["ms"] / k1,
                                        "speedup": line["value"] / v1, "efficiency": line["value"] / v1 / world,
                                        "gathered_results_identical_to_1gpu": bool(same),
                                        "compared_utterances": int(len(sample))}
            one["host"].close()
        barrier()
        # weak scaling as before: every rank aligns its own configs[1]-shaped batch (graph replay)
        m = measure_batch("c2", 100, 5, do_e2e=False, seed_rank=rank)
        if rank == 0:
            line["extra"] = {"c2_replicas": {"workload": f"c2: {m['desc']} -- one batch per rank (weak scaling)",
                                             "value": m["cells"] * world * 100 / (m["ms"] * 1e-3), "unit": "cells/s",
                                             "ms_per_step": m["ms"] / 100, "launch_mode": m["launch_mode"]}}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
