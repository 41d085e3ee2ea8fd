"""GPU tests of mp_set_sources / mp_get_sources, the attribution of every colonisation to its source patches during sweeps:
the sums against a numpy replay of the state read after every sweep, the conservation of the shares, the sampler left
untouched, determinism, chain and rank sharding, the calls that must not touch the sums, the rejected arguments and the
recovery of the sources of a simulated history."""
import ctypes as C

import numpy as np
import pytest

import midaspom_b200 as mb
import oracle_lib as O
from gpu_util import make_engine, pdict, random_landscape

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_STATE = -1, -3
FIX = 2.0 ** -40                                   # unit of the per-sample fixed-point histogram


def distances(spec):
    """D[k, l]: distance from source l to target k, pair_distance's value in FP64."""
    n = spec["obs"].shape[1]
    geom = spec.get("geom", O.GEOM_LINEAR)
    if geom == O.GEOM_COORDS:
        dx = spec["px"][:, None] - spec["px"][None, :]
        dy = spec["py"][:, None] - spec["py"][None, :]
        return np.sqrt(dx * dx + dy * dy)
    if geom == O.GEOM_DENSE:
        return np.asarray(spec["dist"], dtype=np.float64).T      # dist is [source][target]
    idx = np.arange(n)
    return np.abs(idx[:, None] - idx[None, :]).astype(np.float64) * spec.get("spacing", 100.0)


def sample_sources(spec, D, par, z, y, S, nbins, width):
    """The definitions of DESIGN §2 for one chain in FP64: events, unattributed, src_sum [T-1, N], ext_sum, hist [T-1, nbins],
    the number of pairs and the mass of the pairs within 1e-5 of the landscape's extent of a bin edge (where an FP32 distance
    may fall into the neighbouring bin)."""
    T, n = z.shape
    era = np.zeros(T - 1, dtype=bool) if spec.get("era") is None else np.asarray(spec["era"]) != 0
    area = spec.get("area")
    aw = np.ones(n) if area is None or par["b"] == 0 else np.asarray(area) ** par["b"]
    W = np.exp(-(par["alpha"] * D)) * aw[None, :]
    np.fill_diagonal(W, 0.0)
    unit = spec.get("src_unit")
    unit = np.arange(n) + 1.0 if unit is None else np.asarray(unit)
    out = dict(events=np.zeros(T - 1, np.int64), unattributed=np.zeros(T - 1, np.int64), src_sum=np.zeros((T - 1, n)),
               ext_sum=np.zeros(T - 1), hist=np.zeros((T - 1, max(nbins, 1))), pairs=np.zeros(T - 1), edge=np.zeros(T - 1))
    if nbins:
        q = D / width
        bins = np.minimum(np.floor(q), nbins - 1).astype(np.int64)
        near = np.abs(q - np.round(q)) * width <= 1e-5 * D.max()
    for t in range(T - 1):
        pre = era[t]
        Kt, Ks = (par["K"], par["Ksrc"]) if pre else (1.0, 0.0)
        g = np.exp(-(par["alpha"] * unit) * par["dsrc"]) if pre and par["Ksrc"] != 0 else np.zeros(n)
        ev = (y[t] == 0) & (z[t + 1] == 1)
        P = Kt * S[t] + Ks * g
        att = ev & (P > 0)
        out["events"][t] = ev.sum()
        out["unattributed"][t] = (ev & ~att).sum()
        src = y[t] == 1
        rho = Kt * W[np.ix_(att, src)] / P[att][:, None]
        out["src_sum"][t, src] = rho.sum(axis=0)
        out["ext_sum"][t] = (Ks * g[att] / P[att]).sum()
        out["pairs"][t] = rho.size
        if nbins:
            b = bins[np.ix_(att, src)]
            out["hist"][t] = np.bincount(b.ravel(), weights=rho.ravel(), minlength=nbins)
            out["edge"][t] = rho[near[np.ix_(att, src)]].sum()
    return out


def host_sums(eng, spec, D, nsweeps, first, thin, nbins, width):
    """One sweep at a time; after each qualifying sweep add the definitions evaluated on the state the engine holds."""
    T, N = eng.T, eng.N
    acc = dict(nsamples=0, events=np.zeros(T - 1, np.int64), unattributed=np.zeros(T - 1, np.int64), src_sum=np.zeros((T - 1, N)),
               ext_sum=np.zeros(T - 1), hist=np.zeros((T - 1, max(nbins, 1))), pairs=np.zeros(T - 1), edge=np.zeros(T - 1))
    for _ in range(nsweeps):
        s = eng.lib.mp_sweep_index(eng.h)
        eng.sweep(1)
        if s < first or (s - first) % thin:
            continue
        z, y = eng.get_state()
        S = eng.get_connectivity()
        pars = eng.get_params()
        for c in range(eng.C):
            one = sample_sources(spec, D, pars[c], z[c], y[c], S[c], nbins, width)
            for k in one:
                acc[k] = acc[k] + one[k]
        acc["nsamples"] += eng.C
    return acc


def rel_close(got, want, rtol):
    err = np.abs(got - want) / np.maximum(np.abs(want), 1e-300)
    assert (err <= rtol).all(), err.max()


def conservation(got, rtol):
    lhs = got["src_sum"].sum(axis=1) + got["ext_sum"]
    rhs = (got["events"] - got["unattributed"]).astype(np.float64)
    assert (np.abs(lhs - rhs) <= rtol * np.maximum(rhs, 1.0)).all(), (lhs, rhs)
    if got["dist_hist"] is not None:   # every pair is rounded to 2^-40 once per sample; at most events x N pairs
        bound = got["events"] * got["src_sum"].shape[1] * FIX / 2
        assert (np.abs(got["dist_hist"].sum(axis=1) - got["src_sum"].sum(axis=1)) <= 1e-12 * rhs + bound).all()


def landscape(geom, detect, era, seed, n=300, T=6):
    rng = np.random.default_rng(seed)
    spec, _, _ = random_landscape(rng, n, T, geom, occ=0.5, miss=0.15, areas=True)
    spec["detect"] = detect
    spec["prior_occ"] = 0.3
    if era:
        spec["era"] = np.array([1, 1, 0, 0, 0], dtype=np.uint8)
    return spec


CASES = [  # geom, detect, era, precision, first, thin, nbins
    (O.GEOM_LINEAR, 0, False, mb.FP64, 0, 1, 16),
    (O.GEOM_LINEAR, 1, True, mb.FP64, 3, 2, 0),
    (O.GEOM_COORDS, 0, True, mb.FP64, 2, 3, 32),
    (O.GEOM_COORDS, 1, False, mb.FP32, 1, 1, 24),
    (O.GEOM_DENSE, 1, True, mb.FP64, 0, 2, 20),
    (O.GEOM_DENSE, 0, True, mb.FP32, 4, 1, 12),
    (O.GEOM_LINEAR, 0, True, mb.FP32, 0, 1, 40),
]


@pytest.mark.parametrize("geom,detect,era,precision,first,thin,nbins", CASES)
def test_sums_equal_the_state_read_after_every_sweep(monkeypatch, geom, detect, era, precision, first, thin, nbins):
    spec = landscape(geom, detect, era, 80 + geom * 7 + detect)
    D = distances(spec)
    width = 250.0 if geom != O.GEOM_LINEAR else 300.0     # linear: distances are multiples of 100, some fall on the edges
    par = pdict(e=0.3, c=0.05, alpha=1 / 300, b=0.4, p=0.7, K=2.0, Ksrc=0.3 if era else 0.0, dsrc=40.0)
    sc = mb.engine.sampler_config(sample_alpha=1, sample_p=detect, n_adapt=4)
    sums = {}
    for graph in ("1", "0"):
        monkeypatch.setenv("MP_GRAPH", graph)
        with make_engine(spec, n_chains=3, precision=precision, seed=5) as eng:
            eng.set_params([par] * 3)
            eng.init_chains(sc, disperse=True)
            eng.set_sources(first, thin, nbins, width)
            want = host_sums(eng, spec, D, 12, first, thin, nbins, width)
            got = eng.sources()
        sums[graph] = got
        assert got["nsamples"] == want["nsamples"] == 3 * len(range(first, 12, thin))
        assert np.array_equal(got["events"], want["events"]) and np.array_equal(got["unattributed"], want["unattributed"])
        assert got["events"].sum() > 0
        if era:
            assert (want["ext_sum"] > 0).any()                   # the external source takes a share: the check has content
        if precision == mb.FP64:
            rel_close(got["src_sum"], want["src_sum"], 1e-10)
            rel_close(got["ext_sum"], want["ext_sum"], 1e-10)
            conservation(got, 1e-9)
        else:
            rel_close(got["src_sum"], want["src_sum"], 1e-5)
            rel_close(got["ext_sum"], want["ext_sum"], 1e-5)
            conservation(got, 1e-6)
        if nbins:
            assert got["dist_hist"].shape == (5, nbins) and got["bin_width"] == width
            bound = want["pairs"][:, None] * FIX / 2
            if precision == mb.FP32:
                bound = bound + 1e-5 * want["hist"] + want["edge"][:, None]
            assert (np.abs(got["dist_hist"] - want["hist"]) <= bound + 1e-300).all()
            assert (want["hist"][:, 1:] > 0).any()               # mass beyond the first bin
        else:
            assert got["dist_hist"] is None
    for k in ("events", "unattributed", "src_sum", "ext_sum"):
        assert np.array_equal(sums["1"][k], sums["0"][k]), k    # captured sweeps and eager sweeps add the same numbers
    if nbins:
        assert np.array_equal(sums["1"]["dist_hist"], sums["0"]["dist_hist"])


def test_conservation_on_a_culled_landscape():
    """FP32, 20,000 planar patches: k_conn skips far source tiles, the contraction does not; the shares still sum to the
    attributed events within 1e-6."""
    rng = np.random.default_rng(41)
    spec, z, y = random_landscape(rng, 20000, 4, O.GEOM_COORDS, occ=0.5, miss=0.05, areas=True)
    par = pdict(e=0.35, c=0.05, alpha=1 / 100, b=0.5)
    with make_engine(spec, n_chains=2, precision=mb.FP32, seed=3) as eng:
        eng.set_params([par] * 2)
        eng.init_chains(mb.engine.sampler_config(sample_alpha=1, n_adapt=4), disperse=False)
        eng.set_sources(2, 1, 64, 100.0)
        eng.work_counters(reset=True)
        eng.sweep(5)
        got = eng.sources()
        work = eng.work_counters()
    assert work["conn_exec"] < work["conn_total"]             # the connectivity is culled
    assert got["nsamples"] == 6 and got["events"].sum() > 1000
    conservation(got, 1e-6)


def run_sampler(spec, precision, sources, graph, monkeypatch, nsweeps=12, C=2, **kw):
    monkeypatch.setenv("MP_GRAPH", graph)
    par = pdict(e=0.3, c=0.05, alpha=1 / 300, b=0.4, p=0.7, K=2.0, Ksrc=0.3, dsrc=40.0)
    with make_engine(spec, n_chains=C, precision=precision, seed=9, max_draws=nsweeps, **kw) as eng:
        eng.set_params([par] * C)
        eng.init_chains(mb.engine.sampler_config(sample_alpha=1, sample_b=1, sample_p=1, sample_K=1, n_adapt=6), disperse=True)
        if sources:
            eng.set_sources(1, 1, 32, 200.0)
        eng.sweep(nsweeps)
        z, y = eng.get_state()
        out = dict(draws=eng.get_draws(), z=z, y=y, S=eng.get_connectivity(), scales=eng.get_scales())
        out["sources"] = eng.sources() if sources else None
    return out


@pytest.mark.parametrize("precision", [mb.FP32, mb.FP64])
@pytest.mark.parametrize("graph", ["1", "0"])
def test_sampler_is_untouched(monkeypatch, precision, graph):
    spec = landscape(O.GEOM_COORDS, 1, True, 13)
    a = run_sampler(spec, precision, True, graph, monkeypatch)
    b = run_sampler(spec, precision, False, graph, monkeypatch)
    for key in ("draws", "z", "y", "S", "scales"):
        assert np.array_equal(a[key], b[key]), key
    assert a["sources"]["nsamples"] == 11 * 2


def test_identical_runs_give_identical_sums(monkeypatch):
    spec = landscape(O.GEOM_COORDS, 0, True, 17)
    a = run_sampler(spec, mb.FP32, True, "1", monkeypatch)["sources"]
    b = run_sampler(spec, mb.FP32, True, "1", monkeypatch)["sources"]
    for k in ("events", "unattributed", "src_sum", "ext_sum", "dist_hist"):
        assert np.array_equal(a[k], b[k]), k


def test_chain_sharded_engines_add_up():
    spec = landscape(O.GEOM_COORDS, 1, True, 77)
    C = 4
    pars = [pdict(e=0.3, c=0.04 + 0.01 * c, alpha=1 / 300, b=0.4, p=0.7, K=2.0, Ksrc=0.2, dsrc=40.0) for c in range(C)]
    sc = mb.engine.sampler_config(sample_alpha=1, sample_p=1, n_adapt=4)

    def run(n_chains, offset):
        with make_engine(spec, n_chains=n_chains, precision=mb.FP64, seed=3, chain_offset=offset) as eng:
            eng.set_params(pars[offset:offset + n_chains])
            eng.init_chains(sc, disperse=True)
            eng.set_sources(1, 2, 16, 300.0)
            eng.sweep(9)
            return eng.sources()

    whole = run(C, 0)
    parts = [run(C // 2, 0), run(C // 2, C // 2)]
    assert whole["nsamples"] == parts[0]["nsamples"] + parts[1]["nsamples"] == 4 * C
    for k in ("events", "unattributed"):
        assert np.array_equal(parts[0][k] + parts[1][k], whole[k]), k
    for k in ("src_sum", "ext_sum", "dist_hist"):
        np.testing.assert_allclose(parts[0][k] + parts[1][k], whole[k], rtol=1e-12, atol=0)
    pooled = mb.colonisation_sources(parts)
    np.testing.assert_allclose(pooled["caused"], whole["src_sum"].sum(axis=0) / whole["nsamples"], rtol=1e-12, atol=0)


@pytest.mark.skipif(mb.load_library().mp_device_count() < 2, reason="needs 2 GPUs")
def test_sharded_sweeps_over_two_gpus_hold_identical_sums():
    rng = np.random.default_rng(31)
    n, T, C, nsw = 3000, 6, 2, 6
    spec, _, _ = random_landscape(rng, n, T, O.GEOM_COORDS, occ=0.5, miss=0.05)
    par = pdict(e=0.4, c=0.01, alpha=1 / 400, b=0.5)
    sc = mb.engine.sampler_config(sample_alpha=1, sample_b=1, c_max=0.2, n_adapt=4)

    def fresh(device):
        eng = mb.Engine(n, T, C, precision=mb.FP32, device=device, seed=17, max_draws=nsw)
        eng.set_landscape_coords(spec["px"], spec["py"], spec.get("area")); eng.set_source_units(None)
        eng.set_observations(spec["obs"])
        eng.set_params([par] * C)
        eng.init_chains(sc, disperse=False)
        eng.set_sources(1, 1, 32, 200.0)
        return eng

    engs = [fresh(d) for d in range(2)]
    mb.Engine.comm_init_all(engs)
    mb.Engine.sweep_sharded_all(engs, nsw)
    got = []
    for e in engs:
        e.synchronize()
        got.append(e.sources())
    assert got[0]["nsamples"] == got[1]["nsamples"] == (nsw - 1) * C
    for k in ("events", "unattributed", "src_sum", "ext_sum", "dist_hist"):
        assert np.array_equal(got[0][k], got[1][k]), k
    conservation(got[0], 1e-6)
    for e in engs:
        e.close()


def test_other_calls_leave_the_sums_alone():
    spec = landscape(O.GEOM_COORDS, 0, True, 5)
    C = 2
    with make_engine(spec, n_chains=C, precision=mb.FP64, seed=2) as eng:
        eng.set_params([pdict(e=0.3, c=0.05, alpha=1 / 300, b=0.4, K=2.0, Ksrc=0.2, dsrc=40.0)] * C)
        eng.init_chains(mb.engine.sampler_config(sample_alpha=1, n_adapt=4), disperse=True)
        eng.set_sources(0, 1, 16, 250.0)
        eng.sweep(4)
        before = eng.sources()
        z, y = eng.get_state()
        eng.forecast(3, 4, seed=1)
        eng.ppc(3, seed=2)
        eng.capacity()
        eng.connectivity()
        eng.loglik()
        eng.loglik_host(eng.get_params(), z, y)
        eng.flip_delta(0, 1, 2)
        eng.simulate(pdict(e=0.3, c=0.05), z[0, -1], 3, nsims=2)
        eng.simulate_ensemble([pdict(e=0.3, c=0.05)] * 2, z[:, -1], 3)
        after = eng.sources()
        assert after["nsamples"] == before["nsamples"] == 4 * C
        for k in ("events", "unattributed", "src_sum", "ext_sum", "dist_hist"):
            assert np.array_equal(after[k], before[k]), k
        eng.sweep(2)                                             # and the sweeps go on adding
        assert eng.sources()["nsamples"] == 6 * C
        assert eng.sources(reset=True)["nsamples"] == 6 * C
        again = eng.sources()
        assert again["nsamples"] == 0 and not again["src_sum"].any() and not again["dist_hist"].any()


def test_rejected_calls():
    spec = landscape(O.GEOM_LINEAR, 0, False, 3)
    with make_engine(spec, n_chains=2) as eng:
        lib = eng.lib
        assert lib.mp_get_sources(eng.h, None, None, None, None, None, 0) == ERR_STATE
        assert lib.mp_set_sources(eng.h, -1, 1, 0, 0.0) == ERR_ARG
        assert lib.mp_set_sources(eng.h, 0, -1, 0, 0.0) == ERR_ARG
        assert lib.mp_set_sources(eng.h, 0, 1, -1, 1.0) == ERR_ARG
        assert lib.mp_set_sources(eng.h, 0, 1, 4097, 1.0) == ERR_ARG
        for w in (0.0, -1.0, float("inf"), float("nan")):
            assert lib.mp_set_sources(eng.h, 0, 1, 8, w) == ERR_ARG
        assert lib.mp_get_sources(eng.h, None, None, None, None, None, 0) == ERR_STATE
        assert lib.mp_set_sources(eng.h, 0, 1, 0, float("nan")) == 0        # no histogram: the width is ignored
        assert lib.mp_set_sources(eng.h, 0, 1, 4096, 1.0) == 0
        ns = C.c_int64(-1)
        assert lib.mp_get_sources(eng.h, C.byref(ns), None, None, None, None, 0) == 0 and ns.value == 0
        eng.set_sources(0, 0)                                    # off: freed
        assert lib.mp_get_sources(eng.h, None, None, None, None, None, 0) == ERR_STATE


def simulate_history(rng, n, T, e, alpha, b, target_C=0.3):
    """A cfg2-shaped history (uniform positions in a square of side sqrt(n) 250, lognormal areas), perfect detection; returns
    the spec, the true z, y, S and parameters."""
    side = np.sqrt(n) * 250.0
    px, py = rng.uniform(0, side, n), rng.uniform(0, side, n)
    area = rng.lognormal(0.0, 0.5, n)
    spec = dict(geom=O.GEOM_COORDS, px=px, py=py, area=area)
    D = distances(dict(spec, obs=np.zeros((1, n))))
    W = np.exp(-alpha * D) * (area ** b)[None, :]
    np.fill_diagonal(W, 0.0)
    z = np.zeros((T, n), dtype=np.uint8)
    y = np.zeros((T - 1, n), dtype=np.uint8)
    S = np.zeros((T - 1, n))
    z[0] = rng.random(n) < 0.5
    c = None
    for t in range(T - 1):
        y[t] = z[t] & (rng.random(n) > e)
        S[t] = W @ y[t]
        if c is None:
            c = target_C / S[0].mean()
        z[t + 1] = np.where(y[t] == 1, 1, rng.random(n) < np.minimum(1.0, c * S[t]))
    spec["obs"] = z.astype(np.int8)
    return spec, D, z, y, S, pdict(e=e, c=c, alpha=alpha, b=b)


def test_recovers_the_sources_of_a_simulated_history():
    """Thresholds fixed before the first run: posterior-mean sources correlate with the truth's at r >= 0.8 and the mean
    realised distance is within 10 % of the truth's."""
    rng = np.random.default_rng(2024)
    n, T, C = 1000, 10, 8
    spec, D, z, y, S, truth = simulate_history(rng, n, T, e=0.3, alpha=1 / 400, b=0.5)
    nbins, width = 64, 200.0
    true = sample_sources(spec, D, truth, z, y, S, nbins, width)
    true_caused = true["src_sum"].sum(axis=0)
    true_stats = mb.sources._hist_stats(true["hist"].sum(axis=0), width)
    with make_engine(spec, n_chains=C, precision=mb.FP32, seed=11) as eng:
        eng.set_params([truth] * C)
        eng.init_chains(mb.engine.sampler_config(sample_alpha=1, sample_b=1, n_adapt=100), disperse=True)
        eng.sweep(300)
        eng.set_sources(eng.lib.mp_sweep_index(eng.h), 1, nbins, width)
        eng.set_summaries(eng.lib.mp_sweep_index(eng.h), 1)
        eng.sweep(200)
        res = mb.colonisation_sources(eng.sources(), eng.summaries())
    r = float(np.corrcoef(res["caused"], true_caused)[0, 1])
    dmean, dtrue = res["mean_distance"], true_stats["mean_distance"]
    print(f"sources recovery: r = {r:.3f}, mean distance {dmean:.1f} vs {dtrue:.1f} ({dmean / dtrue - 1:+.3%})")
    assert r >= 0.8
    assert abs(dmean / dtrue - 1.0) <= 0.10
    # z is fixed by the data: every observed 0 -> 1 is a colonisation in every sample (and an occupied patch may be recolonised)
    assert (res["received"] >= ((z[1:] == 1) & (z[:-1] == 0)).sum(axis=0) - 1e-12).all()
