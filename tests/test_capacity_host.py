"""CPU checks of midaspom_b200.persistence, the reduction of mp_capacity's per-draw capacities: R, R_pre, the posterior summaries,
P(R > 1), the mean patch values and first-order losses against a direct computation, pooling of several calls and chain shards,
and the refusal to pool capacities of different landscapes or patch masks."""
import numpy as np
import pytest

import midaspom_b200 as mb
from midaspom_b200.engine import DRAW_FIELDS, NDRAW


def fake_draws(rng, M, K=None, Ksrc=0.0):
    d = np.zeros((M, NDRAW))
    d[:, DRAW_FIELDS.index("e")] = rng.uniform(0.1, 0.6, M)
    d[:, DRAW_FIELDS.index("c")] = rng.uniform(0.005, 0.2, M)
    d[:, DRAW_FIELDS.index("alpha")] = 1 / 400
    d[:, DRAW_FIELDS.index("b")] = 0.5
    d[:, DRAW_FIELDS.index("K")] = 1.0 if K is None else K
    d[:, DRAW_FIELDS.index("Ksrc")] = Ksrc
    return d


def fake_capacity(rng, M, N, fingerprint="a"):
    V = rng.random((M, N))
    V /= V.sum(axis=1, keepdims=True)
    return dict(lam=rng.uniform(5, 30, M), values=V, fingerprint=fingerprint)


def direct(rows, lam, V):
    e, c, K = rows[:, 0], rows[:, 1], rows[:, 8]
    R = np.array([(1 - e[i]) * (1 + c[i] * lam[i]) for i in range(len(lam))])
    Rp = np.array([(1 - min(1.0, e[i] / K[i])) * (1 + c[i] * K[i] * lam[i]) for i in range(len(lam))])
    loss = np.array([[-2 * lam[i] * V[i, k] for k in range(V.shape[1])] for i in range(len(lam))]).mean(axis=0)
    return R, Rp, loss


def test_against_direct_computation():
    rng = np.random.default_rng(1)
    draws = fake_draws(rng, 200)
    cap = fake_capacity(rng, 200, 30)
    out = mb.persistence(draws, cap)
    R, _, loss = direct(draws, cap["lam"], cap["values"])
    assert np.allclose(out["R"], R, rtol=1e-15)
    assert out["R_pre"] is None and out["P_R_pre_gt_1"] is None
    assert out["P_R_gt_1"] == np.mean(R > 1)
    for key, x in (("lam_summary", cap["lam"]), ("R_summary", R)):
        s = out[key]
        assert np.isclose(s["mean"], x.mean()) and np.isclose(s["q50"], np.median(x))
        assert np.isclose(s["q025"], np.quantile(x, 0.025)) and np.isclose(s["q975"], np.quantile(x, 0.975))
    assert np.allclose(out["value_mean"], cap["values"].mean(axis=0))
    assert np.allclose(out["loss_mean"], loss)
    assert out["n_draws"] == 200


def test_pre_event_regime():
    rng = np.random.default_rng(2)
    draws = fake_draws(rng, 50, K=rng.uniform(0.2, 4.0, 50))
    lam = rng.uniform(5, 30, 50)
    out = mb.persistence(draws, lam)
    R, Rp, _ = direct(draws, lam, np.zeros((50, 1)))
    assert np.allclose(out["R"], R) and np.allclose(out["R_pre"], Rp)
    assert out["P_R_pre_gt_1"] == np.mean(Rp > 1) and out["value_mean"] is None
    src = fake_draws(rng, 50, K=2.0, Ksrc=0.5)                 # an external source: no R_pre
    assert mb.persistence(src, lam)["R_pre"] is None


def test_pooling_calls_and_shards():
    rng = np.random.default_rng(3)
    parts = [(fake_draws(rng, m).reshape(m, 1, NDRAW), fake_capacity(rng, m, 12)) for m in (10, 7, 13)]
    pooled = mb.persistence([d for d, _ in parts], [c for _, c in parts])
    rows = np.concatenate([d.reshape(-1, NDRAW) for d, _ in parts])
    lam = np.concatenate([c["lam"] for _, c in parts])
    V = np.concatenate([c["values"] for _, c in parts])
    one = mb.persistence(rows, dict(lam=lam, values=V, fingerprint="a"))
    for k in ("R", "lam", "value_mean", "loss_mean"):
        assert np.array_equal(pooled[k], one[k]), k
    assert pooled["R_summary"] == one["R_summary"] and pooled["n_draws"] == 30


def test_refuses_mixed_landscapes_and_mismatched_lengths():
    rng = np.random.default_rng(4)
    a, b = fake_capacity(rng, 5, 8, "a"), fake_capacity(rng, 5, 8, "b")
    d = fake_draws(rng, 5)
    with pytest.raises(ValueError, match="different landscapes"):
        mb.persistence([d, d], [a, b])
    with pytest.raises(ValueError, match="capacities"):
        mb.persistence(d, a["lam"][:4])
    with pytest.raises(ValueError, match="one capacity result"):
        mb.persistence([d, d], [a])
