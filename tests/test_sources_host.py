"""CPU tests of midaspom_b200.colonisation_sources: pooling of calls and chain shards, the refusals, received / net from the
summaries and the distance summaries of the histogram, against a direct computation."""
import numpy as np
import pytest

import midaspom_b200 as mb


def part(rng, T=5, N=7, nbins=6, width=50.0, ns=12, fp="a"):
    ev = rng.integers(5, 20, T - 1).astype(np.uint64)
    un = rng.integers(0, 3, T - 1).astype(np.uint64)
    return dict(nsamples=ns, events=ev, unattributed=un, src_sum=rng.random((T - 1, N)) * 3, ext_sum=rng.random(T - 1),
                dist_hist=rng.random((T - 1, nbins)) if nbins else None, bin_width=width if nbins else 0.0, fingerprint=fp)


def summ(rng, T=5, N=7, ns=12):
    y = rng.integers(0, ns, (T - 1, N)).astype(np.uint32)
    z = np.zeros((T, N), dtype=np.uint32)
    z[1:] = y + rng.integers(0, 3, (T - 1, N)).astype(np.uint32)
    z[0] = rng.integers(0, ns, N)
    return dict(nsamples=ns, z_count=z, y_count=y)


def test_pooling_and_per_sample_quantities():
    rng = np.random.default_rng(1)
    a, b = part(rng, ns=12), part(rng, ns=20)
    r = mb.colonisation_sources([a, b])
    ns = 32
    src = a["src_sum"] + b["src_sum"]
    assert r["nsamples"] == ns
    np.testing.assert_allclose(r["caused_t"], src / ns, rtol=1e-15)
    np.testing.assert_allclose(r["caused"], src.sum(axis=0) / ns, rtol=1e-14)
    ev = a["events"].astype(np.int64) + b["events"]
    un = a["unattributed"].astype(np.int64) + b["unattributed"]
    np.testing.assert_allclose(r["colonisations"], ev / ns)
    np.testing.assert_allclose(r["unattributed"], un / ns)
    np.testing.assert_allclose(r["external"], (a["ext_sum"] + b["ext_sum"]) / ns)
    np.testing.assert_allclose(r["share"], src.sum(axis=0) / (ev - un).sum(), rtol=1e-14)
    np.testing.assert_allclose(r["dist_hist"], (a["dist_hist"] + b["dist_hist"]).sum(axis=0) / ns)
    assert r["received"] is None and r["net"] is None
    one = mb.colonisation_sources(a)                             # a single result needs no list
    np.testing.assert_allclose(one["caused"], a["src_sum"].sum(axis=0) / 12)


def test_received_and_net_from_the_summaries():
    rng = np.random.default_rng(2)
    a, b = part(rng, ns=12), part(rng, ns=20)
    sa, sb = summ(rng, ns=12), summ(rng, ns=20)
    r = mb.colonisation_sources([a, b], [sa, sb])
    z = sa["z_count"].astype(np.int64) + sb["z_count"]
    y = sa["y_count"].astype(np.int64) + sb["y_count"]
    want = np.array([sum(int(z[t + 1, k]) - int(y[t, k]) for t in range(y.shape[0])) for k in range(y.shape[1])]) / 32
    np.testing.assert_allclose(r["received"], want, rtol=1e-15)
    np.testing.assert_allclose(r["net"], r["caused"] - want, rtol=1e-15)
    with pytest.raises(ValueError):
        mb.colonisation_sources([a, b], sa)                      # 12 samples of summaries for 32 of sources
    with pytest.raises(ValueError):
        mb.colonisation_sources(a, summ(rng, T=6, ns=12))


def test_refusals():
    rng = np.random.default_rng(3)
    a = part(rng)
    with pytest.raises(ValueError):
        mb.colonisation_sources([a, part(rng, fp="b")])         # another landscape
    with pytest.raises(ValueError):
        mb.colonisation_sources([a, part(rng, N=8)])
    with pytest.raises(ValueError):
        mb.colonisation_sources([a, part(rng, T=6)])
    with pytest.raises(ValueError):
        mb.colonisation_sources([a, part(rng, nbins=7)])
    with pytest.raises(ValueError):
        mb.colonisation_sources([a, part(rng, width=40.0)])
    with pytest.raises(ValueError):
        mb.colonisation_sources([a, part(rng, nbins=0)])
    with pytest.raises(ValueError):
        mb.colonisation_sources([part(rng, ns=0)])
    with pytest.raises(ValueError):
        mb.colonisation_sources([])


def test_distance_summaries():
    rng = np.random.default_rng(4)
    w = 10.0
    p = part(rng, T=3, nbins=5, width=w)
    p["dist_hist"] = np.array([[1.0, 2.0, 3.0, 2.0, 0.5], [1.0, 2.0, 1.0, 2.0, 0.5]])
    r = mb.colonisation_sources(p)
    H = np.array([2.0, 4.0, 4.0, 4.0, 1.0])
    tot = H.sum()
    np.testing.assert_allclose(r["density"], H[:-1] / (tot * w))
    assert r["beyond"] == pytest.approx(1.0 / 15.0)
    assert r["mean_distance"] == pytest.approx((5 * 2 + 15 * 4 + 25 * 4 + 35 * 4) / 14.0)
    # cdf 2/15, 6/15, 10/15, 14/15, 1: q05 in bin 0, q50 in bin 2, q95 in the open bin
    assert r["quantiles"][0.05] == pytest.approx(0.05 * 15 / 2 * w)
    assert r["quantiles"][0.5] == pytest.approx((2 + (0.5 - 6 / 15) / (4 / 15)) * w)
    assert r["quantiles"][0.95] == float("inf")
    none = mb.colonisation_sources(part(rng, nbins=0))
    assert none["dist_hist"] is None and none["mean_distance"] is None and none["quantiles"] is None
