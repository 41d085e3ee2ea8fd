"""CPU tests of the WAIC reduction (midaspom_b200.waic / compare_waic) on sums built from a synthetic matrix of pointwise log
densities: the reduction against a direct computation from the matrix, chain shards reducing to the whole, and the paired
comparison with its standard error."""
import numpy as np
import pytest

import midaspom_b200 as mb


def sums_of(logp, obs):
    """The engine's sums for a (samples, T, N) array of log densities: 0 where obs is -1."""
    m = obs >= 0
    return dict(nsamples=logp.shape[0], lik_sum=np.where(m, np.exp(logp).sum(0), 0.0),
                loglik_sum=np.where(m, logp.sum(0), 0.0), loglik_sq=np.where(m, (logp ** 2).sum(0), 0.0))


def table(seed, T=5, N=40, S=200, miss=0.2):
    rng = np.random.default_rng(seed)
    obs = (rng.random((T, N)) < 0.5).astype(np.int8)
    obs[rng.random((T, N)) < miss] = -1
    # densities in (0, 1): a per-cell level plus per-sample noise, some cells nearly certain
    level = rng.uniform(-4.0, -1e-3, (T, N))
    logp = np.minimum(level[None] + 0.3 * rng.standard_normal((S, T, N)), -1e-9)
    return obs, logp


def direct(logp, obs):
    m = obs >= 0
    lp = logp[:, m]
    lppd = np.log(np.mean(np.exp(lp), axis=0))
    pw = np.var(lp, axis=0, ddof=1)
    return lppd, pw, lppd - pw


def test_waic_matches_a_direct_computation():
    obs, logp = table(1)
    r = mb.waic(obs, sums_of(logp, obs))
    lppd, pw, elpd = direct(logp, obs)
    m = obs >= 0
    assert r["n_obs"] == m.sum() and r["nsamples"] == logp.shape[0]
    assert np.array_equal(r["observed"], m)
    np.testing.assert_allclose(r["lppd"][m], lppd, rtol=1e-12)
    np.testing.assert_allclose(r["p_waic"][m], pw, rtol=1e-8, atol=1e-12)
    np.testing.assert_allclose(r["elpd"][m], elpd, rtol=1e-10)
    assert np.isnan(r["elpd"][~m]).all()
    assert r["elpd_waic"] == pytest.approx(elpd.sum(), rel=1e-10)
    assert r["p_waic_total"] == pytest.approx(pw.sum(), rel=1e-8)
    assert r["waic"] == pytest.approx(-2 * elpd.sum(), rel=1e-10)
    assert r["lppd_total"] == pytest.approx(lppd.sum(), rel=1e-12)


def test_sharded_sums_reduce_to_the_whole():
    obs, logp = table(2, S=300)
    whole = mb.waic(obs, sums_of(logp, obs))
    parts = mb.waic(obs, sums_of(logp[:100], obs), sums_of(logp[100:250], obs), sums_of(logp[250:], obs))
    m = obs >= 0
    assert parts["nsamples"] == whole["nsamples"] == 300
    for k in ("lppd", "p_waic", "elpd"):
        np.testing.assert_allclose(parts[k][m], whole[k][m], rtol=1e-10, atol=1e-13)
    assert parts["elpd_waic"] == pytest.approx(whole["elpd_waic"], rel=1e-12)


def test_identical_samples_have_no_effective_parameters():
    obs, logp = table(3, S=50)
    frozen = np.repeat(logp[:1], 50, axis=0)
    r = mb.waic(obs, sums_of(frozen, obs))
    m = obs >= 0
    assert (r["p_waic"][m] <= 1e-12).all()
    np.testing.assert_allclose(r["lppd"][m], frozen[0][m], rtol=1e-12, atol=1e-14)   # log(L / S) near 0: absolute rounding


def test_one_sample_gives_no_variance_term():
    obs, logp = table(4, S=1)
    r = mb.waic(obs, sums_of(logp, obs))
    assert np.isnan(r["p_waic"][obs >= 0]).all() and np.isnan(r["elpd_waic"])


def test_compare_waic_matches_a_direct_computation():
    obs, la = table(5)
    rng = np.random.default_rng(6)
    lb = np.minimum(la + 0.2 * rng.standard_normal(la.shape[1:])[None] - 0.05, -1e-9)
    a, b = mb.waic(obs, sums_of(la, obs)), mb.waic(obs, sums_of(lb, obs))
    d = direct(la, obs)[2] - direct(lb, obs)[2]
    c = mb.compare_waic(a, b)
    assert c["n_obs"] == d.size
    assert c["delta_elpd"] == pytest.approx(d.sum(), rel=1e-9)
    assert c["se"] == pytest.approx(np.sqrt(d.size * np.var(d, ddof=1)), rel=1e-9)
    back = mb.compare_waic(b, a)
    assert back["delta_elpd"] == pytest.approx(-c["delta_elpd"], rel=1e-12) and back["se"] == pytest.approx(c["se"], rel=1e-12)


def test_compare_waic_refuses_different_observed_cells():
    obs, logp = table(7)
    other = obs.copy()
    other[0, np.argmax(obs[0] >= 0)] = -1
    with pytest.raises(ValueError, match="different observed cells"):
        mb.compare_waic(mb.waic(obs, sums_of(logp, obs)), mb.waic(other, sums_of(logp, other)))


def test_waic_refuses_bad_input():
    obs, logp = table(8)
    with pytest.raises(ValueError):
        mb.waic(obs)
    with pytest.raises(ValueError, match="shape"):
        mb.waic(obs[:, :-1], sums_of(logp, obs))
    with pytest.raises(ValueError, match="no samples"):
        mb.waic(obs, sums_of(logp[:0], obs))
