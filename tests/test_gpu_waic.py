"""GPU tests of mp_set_waic / mp_get_waic, the pointwise predictive densities of the observations accumulated during sweeps
for WAIC: exact sums against a numpy evaluation of the state read back after every sweep, the sampler left untouched, a
frozen state, the choice between the die-off hypothesis and no event on synthetic data, chain and rank sharding, the calls
that must not touch the sums and the rejected arguments."""
import numpy as np
import pytest

import midaspom_b200 as mb
import oracle_lib as O
from midaspom_b200 import synth
from gpu_util import make_engine, pdict, random_landscape

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_STATE = -1, -3
KEYS = ("lik_sum", "loglik_sum", "loglik_sq")


def logpred_host(spec, par, z, S):
    """(p, log p) of every cell of one chain in FP64 (DESIGN §2): pi from z of the previous year and S of the previous
    transition, p = q pi for an observed 1, 1 - q pi for an observed 0; NaN where the cell is not an observation."""
    obs = np.asarray(spec["obs"])
    T, n = obs.shape
    era = np.zeros(T - 1, dtype=bool) if spec.get("era") is None else np.asarray(spec["era"]) != 0
    u = np.arange(n) + 1.0 if spec.get("src_unit") is None else np.asarray(spec["src_unit"])
    g = np.exp(-(par["alpha"] * u * par["dsrc"]))
    pi = np.zeros((T, n))
    pi[0] = float(np.float32(spec.get("prior_occ", 0.5)))
    for t in range(1, T):
        pre = era[t - 1]
        Kt, Ks = (par["K"], par["Ksrc"]) if pre else (1.0, 0.0)
        C = par["c"] * (Kt * S[t - 1] + Ks * g) if (pre and (par["Ksrc"] != 0 or Kt != 1)) else par["c"] * S[t - 1]
        C = np.minimum(C, 1.0)
        E = min(1.0, par["e"] / par["K"] if pre else par["e"])
        s = z[t - 1] * (1.0 - E)
        pi[t] = s + (1.0 - s) * C
    qpi = par["p"] * pi if spec.get("detect", 0) else pi
    with np.errstate(divide="ignore"):
        dens = np.where(obs == 1, qpi, np.where(obs == 0, 1.0 - qpi, np.nan))
        logp = np.where(obs == 1, np.log(qpi), np.where(obs == 0, np.log1p(-qpi), np.nan))
    return dens, logp


def host_sums(eng, spec, nsweeps, first, thin):
    """One sweep at a time; after each qualifying sweep add the densities of the state the engine holds."""
    m = np.asarray(spec["obs"]) >= 0
    acc = dict(nsamples=0, **{k: np.zeros((eng.T, eng.N)) for k in KEYS})
    for _ in range(nsweeps):
        s = eng.lib.mp_sweep_index(eng.h)
        eng.sweep(1)
        if s < first or (s - first) % thin:
            continue
        z, _ = eng.get_state()
        S = eng.get_connectivity()
        pars = eng.get_params()
        for c in range(eng.C):
            d, lp = logpred_host(spec, pars[c], z[c], S[c])
            acc["lik_sum"] += np.where(m, d, 0.0)
            acc["loglik_sum"] += np.where(m, lp, 0.0)
            acc["loglik_sq"] += np.where(m, lp * lp, 0.0)
        acc["nsamples"] += eng.C
    return acc


def rel_close(got, want, rtol):
    assert np.isfinite(want).all() and np.isfinite(got).all()
    err = np.abs(got - want) / np.maximum(np.abs(want), 1e-300)
    assert (err <= rtol).all(), err.max()


def landscape(geom, detect, era, seed):
    rng = np.random.default_rng(seed)
    spec, _, _ = random_landscape(rng, 300, 6, geom, occ=0.5, miss=0.15, areas=True)
    spec["detect"] = detect
    spec["prior_occ"] = 0.3
    if era:
        spec["era"] = np.array([1, 1, 0, 0, 0], dtype=np.uint8)
    return spec


CASES = [  # geom, detect, era, precision, first, thin
    (O.GEOM_LINEAR, 0, False, mb.FP64, 0, 1),
    (O.GEOM_LINEAR, 1, True, mb.FP64, 3, 2),
    (O.GEOM_COORDS, 0, True, mb.FP64, 2, 3),
    (O.GEOM_COORDS, 1, False, mb.FP32, 1, 1),
    (O.GEOM_DENSE, 1, True, mb.FP64, 0, 2),
    (O.GEOM_DENSE, 0, False, mb.FP32, 4, 1),
    (O.GEOM_COORDS, 1, True, mb.FP32, 0, 1),
]


@pytest.mark.parametrize("geom,detect,era,precision,first,thin", CASES)
def test_sums_equal_a_replay_of_the_state_after_every_sweep(monkeypatch, geom, detect, era, precision, first, thin):
    spec = landscape(geom, detect, era, 60 + geom * 7 + detect)
    par = pdict(e=0.3, c=0.05, alpha=1 / 300, b=0.4, p=0.7, K=2.0, Ksrc=0.3 if era else 0.0, dsrc=40.0)
    sc = mb.engine.sampler_config(sample_alpha=1, sample_p=detect, n_adapt=4)
    sums = {}
    for graph in ("1", "0"):
        monkeypatch.setenv("MP_GRAPH", graph)
        with make_engine(spec, n_chains=3, precision=precision, seed=5) as eng:
            eng.set_params([par] * 3)
            eng.init_chains(sc, disperse=True)
            eng.set_waic(first, thin)
            want = host_sums(eng, spec, 12, first, thin)
            got = eng.waic_sums()
        sums[graph] = got
        assert got["nsamples"] == want["nsamples"] == 3 * len(range(first, 12, thin))
        # FP64: the same expression, 1e-12; FP32: C in FP32 (MUFU lg2 / ex2 in the source term), 1e-5 per term
        rtol = 1e-12 if precision == mb.FP64 else 1e-5
        rel_close(got["lik_sum"], want["lik_sum"], rtol)
        rel_close(got["loglik_sum"], want["loglik_sum"], rtol)
        rel_close(got["loglik_sq"], want["loglik_sq"], 2 * rtol)
        m = spec["obs"] >= 0
        for k in KEYS:
            assert (got[k][~m] == 0).all(), k                       # cells that are not observations are never written
        # the densities genuinely vary between samples: the check has content
        r = mb.waic(spec["obs"], got)
        assert (r["p_waic"][m] > 1e-6).any()
    for k in KEYS:
        assert np.array_equal(sums["1"][k], sums["0"][k]), k       # captured sweeps and eager sweeps add the same numbers


def grid_landscape(seed, n=6000):
    rng = np.random.default_rng(seed)
    spec, z, y = random_landscape(rng, n, 4, O.GEOM_COORDS, occ=0.5, miss=0.05, areas=True)
    return spec, z, y


@pytest.mark.parametrize("blocks", [False, True])
def test_sampler_is_untouched(blocks):
    """FP32, coordinates, N = 6,000: draws, state, S, scales and work counters are bit-identical with WAIC off and with WAIC
    and the summaries on together."""
    spec, z, y = grid_landscape(12)
    par = pdict(e=0.35, c=0.05, alpha=1 / 100, b=0.5)
    C = 2
    grid = None
    if blocks:
        with make_engine(spec, n_chains=C, precision=mb.FP32, seed=1) as eng:
            eng.set_params([par] * C)
            eng.set_state(np.stack([z] * C), np.stack([y] * C))
            S0 = eng.connectivity()
            grid = eng.set_scan_blocks_auto(spec["px"], spec["py"], par["alpha"], float(S0.min()), float(np.max(spec["area"] ** 0.5)), k=3)
        assert grid[0] * grid[1] > 1, grid
    runs = []
    for on in (True, False):
        with make_engine(spec, n_chains=C, precision=mb.FP32, max_draws=16, seed=9) as eng:
            if grid:
                eng.set_scan_blocks(*grid)
            eng.set_params([par] * C)
            eng.init_chains(mb.engine.sampler_config(sample_alpha=1, sample_b=1, n_adapt=6), disperse=False)
            if on:
                eng.set_waic(2, 1)
                eng.set_summaries(1, 2)
            eng.work_counters(reset=True)
            eng.sweep(16)
            zz, yy = eng.get_state()
            runs.append(dict(draws=eng.get_draws(), z=zz, y=yy, S=eng.get_connectivity(), scales=eng.get_scales(),
                             geo=eng.scan_geometry(), work=eng.work_counters()))
            if on:
                assert eng.waic_sums()["nsamples"] == 14 * C
                assert eng.summaries()["nsamples"] == 8 * C
    a, b = runs
    assert a["geo"]["culled"], a["geo"]
    for key in ("draws", "z", "y", "S", "scales"):
        assert np.array_equal(a[key], b[key]), key
    assert a["work"] == b["work"]


def test_launches_per_sweep():
    """With WAIC on a sweep launches one more MP_K_SMALL kernel; after set_waic(0, 0) exactly what an engine that never turned
    it on launches."""
    spec, _, _ = grid_landscape(13, n=2000)
    par = pdict(e=0.35, c=0.05, alpha=1 / 100, b=0.5)
    sc = mb.engine.sampler_config(sample_alpha=1, sample_b=1, n_adapt=6)
    windows = {}
    for waic in (False, True):
        with make_engine(spec, n_chains=2, precision=mb.FP32, seed=9) as eng:
            eng.set_params([par] * 2)
            eng.init_chains(sc, disperse=False)
            eng.set_timing(True)
            if waic:
                eng.set_waic(0, 1)
            eng.sweep(2)
            eng.get_timing(reset=True)
            eng.sweep(4)
            first = eng.get_timing(reset=True)[1]
            if waic:
                eng.set_waic(0, 0)
            eng.sweep(4)
            windows[waic] = (first, eng.get_timing(reset=True)[1])
    never, toggled = windows[False], windows[True]
    assert toggled[1] == never[1]
    for cat in mb.KERNEL_CATEGORIES:
        assert toggled[0][cat] == never[0][cat] + (4 if cat == "small" else 0), cat


def test_frozen_state_has_no_effective_parameters():
    """Nothing sampled: every sample is the same, p_waic_i vanishes and lppd_i is the one-sample log density."""
    spec = landscape(O.GEOM_COORDS, 1, True, 41)
    rng = np.random.default_rng(41)
    T, n = spec["obs"].shape
    z = np.where(spec["obs"] == 1, 1, (rng.random((T, n)) < 0.4)).astype(np.uint8)
    y = (z[:-1] & z[1:] & (rng.random((T - 1, n)) < 0.6)).astype(np.uint8)
    C = 2
    par = pdict(e=0.3, c=0.05, alpha=1 / 300, b=0.4, p=0.7, K=2.0, Ksrc=0.3, dsrc=40.0)
    frozen = mb.engine.sampler_config(sample_e=0, sample_c=0, sample_alpha=0, sample_b=0, sample_p=0, update_z=0, update_y=0)
    with make_engine(spec, n_chains=C, precision=mb.FP64, seed=4) as eng:
        eng.set_params([par] * C)
        eng.init_chains(frozen, disperse=False)
        eng.set_state(np.stack([z] * C), np.stack([y] * C))
        eng.set_waic(0, 1)
        eng.sweep(10)
        zz, yy = eng.get_state()
        assert np.array_equal(zz[0], z) and np.array_equal(yy[0], y)
        r = mb.waic(spec["obs"], eng.waic_sums())
        _, lp = logpred_host(spec, eng.get_params()[0], z, eng.get_connectivity()[0])
    m = spec["obs"] >= 0
    assert r["nsamples"] == 10 * C
    assert (r["p_waic"][m] <= 1e-12).all()
    np.testing.assert_allclose(r["lppd"][m], lp[m], rtol=1e-12, atol=1e-14)


def fit_waic(wl, era, sample_K, K0, chains=8, burn=300, keep=300):
    """8 FP32 chains on a synthetic workload; WAIC after the burn-in.  era: flags of the fitted model (None: no event)."""
    t = wl["truth"]
    eng = mb.Engine(wl["n"], wl["T"], chains, precision=mb.FP32, seed=2024, detect=wl["detect"], max_draws=4)
    try:
        eng.set_landscape_coords(wl["px"], wl["py"], wl["area"])
        eng.set_source_units(None)
        eng.set_observations(wl["obs"])
        eng.set_era(era)
        eng.set_params([dict(e=t["e"], c=t["c"], alpha=t["alpha"], b=t["b"], p=t["p"], K=K0, Ksrc=0.0, dsrc=0.0)] * chains)
        eng.init_chains(mb.engine.sampler_config(sample_e=1, sample_c=1, sample_alpha=1, sample_b=1, c_max=20.0 * t["c"],
                                                 n_adapt=200, sample_K=sample_K), disperse=False)
        eng.sweep(burn)
        eng.set_waic(eng.lib.mp_sweep_index(eng.h), 1)
        eng.sweep(keep)
        return mb.waic(wl["obs"], eng.waic_sums()), eng.get_params()
    finally:
        eng.close()


@pytest.mark.parametrize("name", ["cfg4", "cfg3"])
def test_waic_picks_the_hypothesis_that_generated_the_data(name):
    """H1 (die-off: era flags on the first 10 transitions, K sampled) against H0 (no event).  Thresholds fixed before the
    first run: on the die-off data (cfg4, K = 3) H1 wins by more than 4 standard errors; on data without an event (cfg3) H1
    is not ahead by more than max(4 se, 5)."""
    wl = synth.make_workload(name)
    era = (np.arange(wl["T"] - 1) < 10).astype(np.uint8)
    h0, _ = fit_waic(wl, None, 0, 1.0)
    h1, p1 = fit_waic(wl, era, 1, 3.0 if name == "cfg4" else 1.0)
    d = mb.compare_waic(h1, h0)
    print(name, d, "K", [round(p["K"], 3) for p in p1], "p_waic", h0["p_waic_total"], h1["p_waic_total"])
    if name == "cfg4":
        assert d["delta_elpd"] > 4 * d["se"], d
    else:
        assert d["delta_elpd"] < max(4 * d["se"], 5.0), d


def test_chain_sharded_engines_add_up():
    spec = landscape(O.GEOM_COORDS, 1, True, 77)
    C = 4
    pars = [pdict(e=0.3, c=0.04 + 0.01 * c, alpha=1 / 300, b=0.4, p=0.7, K=2.0) for c in range(C)]
    sc = mb.engine.sampler_config(sample_alpha=1, sample_p=1, n_adapt=4)

    def run(n_chains, offset):
        with make_engine(spec, n_chains=n_chains, precision=mb.FP64, seed=3, chain_offset=offset) as eng:
            eng.set_params(pars[offset:offset + n_chains])
            eng.init_chains(sc, disperse=True)
            eng.set_waic(1, 2)
            eng.sweep(9)
            return eng.waic_sums()

    whole = run(C, 0)
    parts = [run(C // 2, 0), run(C // 2, C // 2)]
    assert whole["nsamples"] == parts[0]["nsamples"] + parts[1]["nsamples"] == 4 * C
    for k in KEYS:
        np.testing.assert_allclose(parts[0][k] + parts[1][k], whole[k], rtol=1e-12, atol=0)
    a, b = mb.waic(spec["obs"], whole), mb.waic(spec["obs"], *parts)
    m = spec["obs"] >= 0
    for k in ("lppd", "p_waic", "elpd"):
        np.testing.assert_allclose(b[k][m], a[k][m], rtol=1e-12, atol=1e-14)
    assert b["elpd_waic"] == pytest.approx(a["elpd_waic"], rel=1e-12)


@pytest.mark.skipif(mb.load_library().mp_device_count() < 2, reason="needs 2 GPUs")
def test_sharded_sweeps_over_two_gpus_hold_the_single_engine_sums():
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
        eng.set_waic(1, 1)
        return eng

    ref = fresh(0)
    ref.sweep(nsw)
    want = ref.waic_sums()
    ref.close()
    engs = [fresh(d) for d in range(2)]
    mb.Engine.comm_init_all(engs)
    mb.Engine.sweep_sharded_all(engs, nsw)
    for e in engs:
        e.synchronize()
        got = e.waic_sums()
        assert got["nsamples"] == want["nsamples"] == (nsw - 1) * C
        for k in KEYS:
            assert np.array_equal(got[k], want[k]), k
    for e in engs:
        e.close()


def test_other_calls_leave_the_sums_alone():
    spec = landscape(O.GEOM_COORDS, 0, True, 5)
    C = 2
    with make_engine(spec, n_chains=C, precision=mb.FP64, seed=2) as eng:
        eng.set_params([pdict(e=0.3, c=0.05, alpha=1 / 300, b=0.4, K=2.0)] * C)
        eng.init_chains(mb.engine.sampler_config(sample_alpha=1, n_adapt=4), disperse=True)
        eng.set_waic(0, 1)
        eng.sweep(4)
        before = eng.waic_sums()
        z, y = eng.get_state()
        eng.forecast(3, 4, seed=1)
        eng.connectivity()
        eng.loglik()
        eng.loglik_host(eng.get_params(), z, y)
        eng.flip_delta(0, 1, 2)
        eng.simulate(pdict(e=0.3, c=0.05), z[0, -1], 3, nsims=2)
        after = eng.waic_sums()
        assert after["nsamples"] == before["nsamples"] == 4 * C
        for k in KEYS:
            assert np.array_equal(after[k], before[k]), k
        eng.sweep(2)                                             # and the sweeps go on adding
        assert eng.waic_sums()["nsamples"] == 6 * C
        eng.set_observations(spec["obs"])                        # new observations: the sums start again
        s = eng.waic_sums()
        assert s["nsamples"] == 0 and all((s[k] == 0).all() for k in KEYS)
        eng.sweep(1)
        assert eng.waic_sums(reset=True)["nsamples"] == C
        assert eng.waic_sums()["nsamples"] == 0


def test_rejected_calls():
    import ctypes as C
    spec = landscape(O.GEOM_LINEAR, 0, False, 3)
    T, n = spec["obs"].shape
    bare = mb.Engine(n, T, 2)                                   # no observations yet
    try:
        assert bare.lib.mp_set_waic(bare.h, 0, 1) == ERR_STATE
        assert bare.lib.mp_get_waic(bare.h, None, None, None, None, 0) == ERR_STATE
    finally:
        bare.close()
    with make_engine(spec, n_chains=2) as eng:
        lib = eng.lib
        assert lib.mp_get_waic(eng.h, None, None, None, None, 0) == ERR_STATE
        assert lib.mp_set_waic(eng.h, -1, 1) == ERR_ARG
        assert lib.mp_set_waic(eng.h, 0, -1) == ERR_ARG
        assert lib.mp_get_waic(eng.h, None, None, None, None, 0) == ERR_STATE
        eng.set_waic(0, 1)
        ns = C.c_int64(-1)
        assert lib.mp_get_waic(eng.h, C.byref(ns), None, None, None, 0) == 0 and ns.value == 0
        eng.set_waic(0, 0)                                       # off: freed
        assert lib.mp_get_waic(eng.h, None, None, None, None, 0) == ERR_STATE
