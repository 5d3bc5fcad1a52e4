"""CPU: the float64 emission reference and its error bound (oracle/emission_f64.py).  The bound must hold
for the C oracle's libm f32 emissions (a sequential sum), and it must be tight enough to see one kept id
too few or too many in the normaliser."""
import numpy as np
import pytest

from oracle import c_oracle as oc
from oracle import emission_f64 as ef


def _rows(kind, rng, T, V, ids):
    keep = ef.keep_mask(ids, V)
    if kind == "random":
        x = 3.0 * rng.standard_normal((T, V))
    elif kind == "flat":                                   # kept logits within +-1, masked ones anywhere
        x = np.where(keep, rng.uniform(-1.0, 1.0, (T, V)), 5.0 * rng.standard_normal((T, V)))
    elif kind == "range80":                                # exp of the smaller ones underflows in f32
        x = rng.uniform(-80.0, 80.0, (T, V))
    else:                                                  # -inf at kept and at masked ids
        x = 3.0 * rng.standard_normal((T, V))
        x[rng.random((T, V)) < 0.15] = -np.inf
        x[:, 0] = np.where(rng.random(T) < 0.5, -np.inf, x[:, 0])
    return np.ascontiguousarray(x, dtype=np.float32)


@pytest.mark.parametrize("kind", ["random", "flat", "range80", "neginf"])
@pytest.mark.parametrize("V,n_ids", [(2, 1), (39, 20), (63, 48), (200, 199), (300, 120)])
def test_c_oracle_emission_within_the_bound(kind, V, n_ids):
    rng = np.random.default_rng(V * 31 + n_ids + len(kind))
    kept = np.concatenate([[0], rng.choice(np.arange(1, V), n_ids - 1, replace=False)]) if n_ids > 1 else np.array([0])
    ids = rng.choice(kept, 3 * len(kept)).astype(np.int32)
    ids[: len(kept)] = kept
    x = _rows(kind, rng, 257, V, ids)
    got = oc.emission(x, ids).astype(np.float64)
    out, xm, lse, n = ef.emission_f64(x, ids, V)
    assert n == len(kept)
    fin = np.isfinite(out)
    assert np.array_equal(np.isneginf(got), np.isneginf(out))
    err = np.abs(got[fin] - out[fin])
    bound = ef.emission_bound(out, xm, lse, n, ef.sum_depth(n, V, "sequential"))[fin]
    assert (err <= bound).all(), f"worst error / bound = {np.max(err / bound):.3f}"


@pytest.mark.parametrize("n_ids", [8, 33, 64, 200])
def test_bound_sees_one_kept_id_more_or_less(n_ids):
    """Flat rows: leaving one kept id out of the normaliser, or counting it twice, moves every emission of the
    row by |d lse| -- at least 10x the kernels' bound for that row."""
    V = 256
    rng = np.random.default_rng(n_ids)
    kept = np.concatenate([[0], rng.choice(np.arange(1, V), n_ids - 1, replace=False)])
    ids = kept.astype(np.int32)
    x = _rows("flat", rng, 64, V, ids)
    out, xm, lse, n = ef.emission_f64(x, ids, V)
    bound = ef.emission_bound(out, xm, lse, n, ef.sum_depth(n, V, "stream")).max(axis=1)
    x64 = x.astype(np.float64)
    m = x64[:, kept].max(axis=1)
    z = np.exp(x64[:, kept] - m[:, None])
    for k in range(n):
        z_k = z[:, k]
        for lse2 in (np.log(z.sum(axis=1) - z_k), np.log(z.sum(axis=1) + z_k)):
            assert (np.abs(lse2 - lse) >= 10.0 * bound).all(), (k, np.min(np.abs(lse2 - lse) / bound))


def test_edge_bounds_hold_for_the_c_oracle():
    rng = np.random.default_rng(5)
    x = np.concatenate([3.0 * rng.standard_normal(4000), rng.uniform(-100.0, 100.0, 1000),
                        [0.0, -0.0, 2.1972246, -2.1972246, 88.0, -88.0, 104.0, -104.0]]).astype(np.float32)
    p = oc.edge_pred(x).astype(np.float64)
    want, bound = ef.edge_pred_f64(x)
    assert (np.abs(p - want) <= bound).all()
    el, ne = oc.edge_logs(oc.edge_prob(p.astype(np.float32))[1])
    wl, wn = ef.edge_logs_f64(p.astype(np.float32))
    assert (np.abs(el - wl) <= ef.f32_ulp(wl)).all() and (np.abs(ne - wn) <= ef.f32_ulp(wn)).all()
