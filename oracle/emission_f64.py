"""float64 restatement of the logits -> emission / edge stage, with per-element error bounds for the
CUDA kernels' f32 arithmetic -- TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Reference: alignment_decoder.py:35-40 (keep mask = ids of ph_seq U {0}), :53 (masked logits pushed down
by 1e9 in f32), :62-65 (log_softmax), :239 (gather by phoneme id), :68-71 (edge sigmoid, rescale, clamp).

Error bound of one emission (hfa_emission.cu, stream / block / wide kernels, and the fused band producer)
-------------------------------------------------------------------------------------------------------
u = 2^-24 (f32 unit round-off); every f32 operation is correctly rounded (no fast-math, explicit _rn
intrinsics), so a rounded result r of an exact value v has |r - v| <= u |v|, and one ulp of v is <= 2u|v|.
The row max m is exact (a max rounds nothing), and so is every conversion of a logit to f32 (bf16 / f16 ->
f32 is exact), so the kernel and this reference start from the same x and the same m.

  d_k = fl(x_k - m)        |d_k - (x_k - m)| <= u |x_k - m|
  e_k = expf(d_k)          expf is within 2 ulp (CUDA C Programming Guide, Appendix "Mathematical
                           Functions"): relative 4u; the error of d_k adds relative |x_k - m| u, and
                           exp(d) |d| <= 1/e for d <= 0, so over the whole sum it adds at most u n / e
                           relative to the sum (the sum is >= 1: the max term is exp(0) = 1)
  Z = sum e_k              positive terms added in a tree of depth D: relative error <= D u.  The stream,
                           block and fused kernels give each row 4 lanes, a lane adds ceil(n/4) terms and
                           two butterfly steps join the lanes: D = ceil(n/4) + 2.  The wide kernel sums all
                           V columns over 32 lanes and 5 steps: D = ceil(V/32) + 5 (masked terms are exactly
                           0 and add nothing).  A sequential sum (the C oracle) has D = n.
  lse = logf(Z)            logf is within 1 ulp: 2u lse absolute; the relative error eta of Z becomes
                           |eta| absolute: (D + 4 + n/e) u
  out = fl(d_id - lse)     d_id carries u |x_id - m| (above), the subtraction rounds by u |out|

  |out - out_f64| <= u (|x_id - m| + |out| + 2 lse + D + 4 + n/e)            (first order)

with n the number of kept ids.  For the 4-lane kernels D + 4 + n/e <= c n + c0 with c = 1/4 + 1/e and
c0 = 3/4 + 2 + 4.  The terms of second order are below (D u)^2 relative, far below the 2^-10 relative
slack the bound carries for them.  Exponentials that underflow to a subnormal or to 0 (x_k - m < -87)
change Z by less than n 2^-126, which Z >= 1 absorbs into its own rounding.

Contract (DESIGN.md 4.1): finite logits with |x| < 5e8 and -inf anywhere.  NaN, +inf and |x| >= 5e8 are
out of contract: the reference then lets masked ids into the max (x - 1e9 no longer stays below every
kept logit).  A row in which every logit is -inf gives NaN here (the reference's value) and -inf in the
kernels, a deliberate divergence.

Error bound of edge_p = clamp((sigmoid(x) - 0.1f) / 0.8f, 0, 1), all f32
--------------------------------------------------------------------------
  e = expf(-x): relative 4u;  a = fl(1 + e): relative 4u + u;  sg = fl(1 / a): relative 6u
  fl(sg - 0.1f): 6u sg + u |sg - 0.1f|;  fl(. / 0.8f): that / 0.8f + u |v|;  the clamp is 1-Lipschitz
  |p - p_f64| <= u (7.5 sg + 1.25 |sg - 0.1f| + |v|)    (first order; same 2^-10 slack)
The f64 reference uses the f32 constants 0.1f and 0.8f, the values the reference's f32 tensors carry.
"""
from __future__ import annotations

import numpy as np

U = 2.0 ** -24
SLACK = 1.0 + 2.0 ** -10          # the second-order terms of the first-order bounds above


def keep_mask(ids, V: int) -> np.ndarray:
    keep = np.zeros(V, dtype=bool)
    keep[np.asarray(ids, dtype=np.int64)] = True
    keep[0] = True                                               # :39 -- id 0 always kept
    return keep


def emission_f64(logits, ids, V: int):
    """logits [T, V] (f32 / f16 / bf16 values as numpy or torch) -> (out f64 [T, S], x - m at the gathered
    ids f64 [T, S], lse f64 [T], n_kept).  Masked logits get the reference's f32 `x - 1e9f` first."""
    if hasattr(logits, "detach"):
        logits = logits.detach().float().cpu().numpy()
    x32 = np.array(logits, dtype=np.float32)                     # exact for bf16 / f16 inputs
    assert x32.ndim == 2 and x32.shape[1] == V
    ids = np.asarray(ids, dtype=np.int64)
    keep = keep_mask(ids, V)
    x32[:, ~keep] = x32[:, ~keep] - np.float32(1e9)              # :53 in f32
    x = x32.astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        m = x.max(axis=1)
        lse = np.log(np.exp(x - m[:, None]).sum(axis=1))
        xm = x[:, ids] - m[:, None]
        out = xm - lse[:, None]
    return out, xm, lse, int(keep.sum())


def sum_depth(n_kept: int, V: int, kernel: str) -> int:
    """Depth D of the kernel's summation tree of one row's exponentials (see the module docstring)."""
    if kernel == "wide":
        return -(-V // 32) + 5
    if kernel == "sequential":
        return n_kept
    return -(-n_kept // 4) + 2


def emission_bound(out, xm, lse, n_kept: int, depth: int) -> np.ndarray:
    """Per-element bound on |kernel - out| for finite `out` (module docstring)."""
    with np.errstate(invalid="ignore"):
        b = np.abs(xm) + np.abs(out) + 2.0 * np.abs(lse)[:, None] + depth + 4 + n_kept / np.e
    return U * b * SLACK


def edge_pred_f64(edge_logits):
    """edge logits (f32 / f16 / bf16 values) -> (p f64, bound on |kernel p - p|)."""
    if hasattr(edge_logits, "detach"):
        edge_logits = edge_logits.detach().float().cpu().numpy()
    x = np.asarray(edge_logits, dtype=np.float32).astype(np.float64)
    with np.errstate(over="ignore"):
        sg = 1.0 / (1.0 + np.exp(-x))
    c, k = float(np.float32(0.1)), float(np.float32(0.8))
    v = (sg - c) / k
    p = np.clip(v, 0.0, 1.0)
    return p, U * (7.5 * sg + 1.25 * np.abs(sg - c) + np.abs(v)) * SLACK


def edge_logs_f64(p32):
    """edge_log / not_edge_log of the kernel's own f32 p, in f64 (:84, :241-242)."""
    p = np.asarray(p32, dtype=np.float32).astype(np.float64)
    ep = p + np.concatenate([[0.0], p[:-1]])
    ep = np.clip(ep, 0.0, 1.0)
    return np.log(ep + 1e-6), np.log((1.0 - ep) + 1e-6)


def f32_ulp(v) -> np.ndarray:
    """One f32 ulp at |v| (v f64)."""
    a = np.abs(np.asarray(v, dtype=np.float64)).astype(np.float32)
    return (np.nextafter(a, np.float32(np.inf)) - a).astype(np.float64)
