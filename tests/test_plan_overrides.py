"""The HFA_* routing overrides (DESIGN.md 4.6) are read once, by hfa_plan_create, and a plan keeps what it read.

CPU: every getenv of the library lies inside hfa_plan_create, and the variables read there are the ones DESIGN.md
4.6 lists.  GPU: a variable no longer read (HFA_HYBRID) changes no routing, and variables set after a plan was made
change nothing the plan's calls compute."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hubertfa_b200", "csrc")


def _code_only(src):
    """src with comments and string / character literals blanked out, offsets and newlines kept."""
    pat = re.compile(r'//[^\n]*|/\*.*?\*/|"(?:\\.|[^"\\\n])*"|\'(?:\\.|[^\'\\\n])*\'', re.S)
    return pat.sub(lambda m: re.sub(r"[^\n]", " ", m.group(0)), src)


def _body_span(code, name):
    """[begin, end) of the brace-delimited body of the function `name` defined in `code`."""
    m = re.search(r"\bint\s+" + name + r"\s*\([^)]*\)\s*\{", code)
    assert m, f"no definition of {name}"
    depth = 0
    for i in range(m.end() - 1, len(code)):
        depth += {"{": 1, "}": -1}.get(code[i], 0)
        if depth == 0:
            return m.end() - 1, i + 1
    raise AssertionError(f"unbalanced braces in {name}")


def _env_reads():
    """Names of the environment variables the library reads, and the getenv calls outside hfa_plan_create."""
    names, outside = [], []
    for fn in sorted(os.listdir(CSRC)):
        path = os.path.join(CSRC, fn)
        if not os.path.isfile(path):
            continue
        with open(path, encoding="utf-8", errors="replace") as f:
            raw = f.read()
        code = _code_only(raw)
        span = _body_span(code, "hfa_plan_create") if fn == "hfa_api.cu" else (0, 0)
        for m in re.finditer(r"\bgetenv\s*\(", code):
            line = raw.count("\n", 0, m.start()) + 1
            if not span[0] <= m.start() < span[1]:
                outside.append(f"{fn}:{line}")
                continue
            arg = re.match(r'\s*"([^"]+)"\s*\)', raw[m.end():])
            assert arg, f"{fn}:{line}: getenv of something other than a string literal"
            names.append(arg.group(1))
    return names, outside


def _design_table_names():
    with open(os.path.join(ROOT, "DESIGN.md"), encoding="utf-8") as f:
        text = f.read()
    sec = re.search(r"^### 4\.6 .*?(?=^##)", text, re.S | re.M)
    assert sec, "DESIGN.md has no section 4.6"
    rows = [ln for ln in sec.group(0).splitlines() if ln.startswith("|") and "HFA_" in ln]
    assert rows, "DESIGN.md 4.6 has no table of variables"
    return {n for ln in rows for n in re.findall(r"\bHFA_[A-Z0-9_]+", ln)}


def test_overrides_are_read_only_by_plan_create_and_match_the_design_table():
    names, outside = _env_reads()
    assert outside == [], f"getenv outside hfa_plan_create: {outside}"
    assert len(names) == len(set(names)), f"a variable is read twice: {sorted(names)}"
    assert set(names) == _design_table_names()


@pytest.fixture
def no_hfa_env(monkeypatch):
    """No HFA_* variable set: the planner's own choices."""
    for k in list(os.environ):
        if k.startswith("HFA_"):
            monkeypatch.delenv(k)
    return monkeypatch


@pytest.mark.gpu
def test_hybrid_variable_is_ignored(no_hfa_env):
    """A config-4-shaped batch (4096 utterances, V = 74) is planned the same with HFA_HYBRID set: its costliest
    utterances stay in the warp-per-utterance kernel.  Plans only, no launch."""
    from hubertfa_b200 import ops, synth
    V = 74
    T, S = synth.sample_shapes(4096, seed=synth.SEED0)
    ids = np.concatenate(synth.make_ids_batch(T, S, V, seed=synth.SEED0))
    plain = ops.AlignPlan(T, S, ids, V, synth.FRAME_SECONDS)
    no_hfa_env.setenv("HFA_HYBRID", "0.26")
    hybrid = ops.AlignPlan(T, S, ids, V, synth.FRAME_SECONDS)
    assert plain.routing()["warp_utts"] == len(T)
    assert hybrid.routing() == plain.routing()
    assert hybrid.workspace_bytes == plain.workspace_bytes


@pytest.mark.gpu
def test_variables_set_after_the_plan_are_ignored(no_hfa_env):
    """A config-2-shaped plan (256 utterances, V = 63) made with no variable set runs in the skewed strips.
    HFA_NO_TENSORMAP=1 and HFA_SKEW_SLOW=1 set afterwards change nothing hfa_align_batch computes with it, while a
    plan made under them takes the halo bands."""
    import torch
    from hubertfa_b200 import _lib, ops, synth
    dev = torch.device("cuda")
    V = 63
    T, S = synth.sample_shapes(256, seed=synth.SEED0, min_s=5, max_s=30, s_lo=20, s_hi=150)
    ids = np.concatenate(synth.make_ids_batch(T, S, V, seed=synth.SEED0))
    plan = ops.AlignPlan(T, S, ids, V, synth.FRAME_SECONDS)
    rt = plan.routing()
    assert rt["skew_d"] == 2 and rt["band_warps"] > 0 and rt["warp_utts"] == 0, rt
    off = np.concatenate([[0], np.cumsum(T, dtype=np.int64)])
    g = torch.Generator(device=dev).manual_seed(2024)
    head = torch.randn(int(off[-1]), V + 2, device=dev, generator=g) * 3.0     # [sum T, V+2]: col 0 edge, 2.. frame
    ws = plan.new_workspace(dev)
    plan.upload(ws)
    n = len(T)
    plan.set_inputs(ws, [head[int(off[b]):int(off[b + 1]), 2:].data_ptr() for b in range(n)], [V + 2] * n, [1] * n,
                    [head[int(off[b]):int(off[b + 1]), 0].data_ptr() for b in range(n)], [V + 2] * n)

    def run():
        res = plan.new_result(dev).zero_()        # segment slots past n_seg are never written
        fc = torch.zeros(plan.total_frames, dtype=torch.float32, device=dev)
        ops.align_batch(ws, plan.handle, _lib.DTYPE_F32, res, fc)
        torch.cuda.synchronize()
        return res.cpu().numpy(), fc.cpu().numpy()

    want_res, want_fc = run()
    no_hfa_env.setenv("HFA_NO_TENSORMAP", "1")
    no_hfa_env.setenv("HFA_SKEW_SLOW", "1")
    got_res, got_fc = run()
    assert np.array_equal(got_res, want_res)
    assert np.array_equal(got_fc.view(np.uint32), want_fc.view(np.uint32))
    assert (plan.views(got_res)["status"] == 0).any()
    rt_new = ops.AlignPlan(T, S, ids, V, synth.FRAME_SECONDS).routing()
    assert rt_new["skew_d"] == 0 and rt_new["band_warps"] > 0, rt_new
