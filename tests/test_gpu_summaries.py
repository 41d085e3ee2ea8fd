"""GPU tests of mp_set_summaries / mp_get_summaries, the posterior sums of the latent state accumulated during sweeps: exact
counts and sums against the state read back after every sweep, the Rao-Blackwellised occupancy against a numpy evaluation of
the conditional and against the exact posterior of the bundled example, the sampler left untouched, chain and rank sharding,
the calls that must not touch the sums, the rejected arguments and the driver's -O table."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

import midaspom_b200 as mb
import oracle_lib as O
from gpu_util import make_engine, pdict, random_landscape

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
EXAMPLE = ROOT / "tests" / "golden" / "occupancies_example.txt"
ERR_ARG, ERR_STATE = -1, -3
KEYS = ("z_count", "z_prob", "y_count", "S_sum")


def zprob_host(spec, par, z, y, S):
    """P(z_tk = 1 | y, theta, obs) of one chain in FP64: the log-odds k_update_z forms, the indicator where the data fix z."""
    obs = np.asarray(spec["obs"])
    T, n = obs.shape
    era = np.zeros(T - 1, dtype=bool) if spec.get("era") is None else np.asarray(spec["era"]) != 0
    detect = spec.get("detect", 0)
    p0 = float(np.float32(spec.get("prior_occ", 0.5)))
    g = np.exp(-par["alpha"] * (np.arange(n) + 1.0) * par["dsrc"])
    with np.errstate(all="ignore"):
        lod = np.zeros((T, n))
        for t in range(T):
            if t > 0:
                pre = era[t - 1]
                Kt, Ks = (par["K"], par["Ksrc"]) if pre else (1.0, 0.0)
                C = par["c"] * (Kt * S[t - 1] + Ks * g) if (pre and (par["Ksrc"] != 0 or Kt != 1)) else par["c"] * S[t - 1]
                C = np.minimum(C, 1.0)
                lod[t] += np.log(C) - np.log1p(-C)
            if t < T - 1:
                lod[t] += np.log(min(1.0, par["e"] / par["K"] if era[t] else par["e"]))
        lod[0] += np.log(p0) - np.log(1.0 - p0)
        lod += np.where((obs == 0) & bool(detect), np.log(1.0 - par["p"]), 0.0)
        prob = np.where(np.isnan(lod), 0.0, 1.0 / (1.0 + np.exp(-lod)))
    latent = (obs == -1) | ((obs == 0) & bool(detect))
    forced = np.zeros((T, n), dtype=bool)
    forced[1:] |= y.astype(bool)
    forced[:-1] |= y.astype(bool)
    return np.where(latent, np.where(forced, 1.0, prob), z.astype(np.float64))


def host_sums(eng, spec, nsweeps, first, thin, zprob=True):
    """One sweep at a time; after each qualifying sweep add what the engine holds to host sums."""
    T, N = eng.T, eng.N
    acc = dict(nsamples=0, z_count=np.zeros((T, N), np.int64), z_prob=np.zeros((T, N)), y_count=np.zeros((T - 1, N), np.int64),
               S_sum=np.zeros((T - 1, N)))
    for _ in range(nsweeps):
        s = eng.lib.mp_sweep_index(eng.h)
        eng.sweep(1)
        if s < first or (s - first) % thin:
            continue
        z, y = eng.get_state()
        S = eng.get_connectivity()
        pars = eng.get_params()
        for c in range(eng.C):
            acc["z_count"] += z[c]
            acc["y_count"] += y[c]
            acc["S_sum"] += S[c]
            if zprob:
                acc["z_prob"] += zprob_host(spec, pars[c], z[c], y[c], S[c])
        acc["nsamples"] += eng.C
    return acc


def rel_close(got, want, rtol):
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
]


@pytest.mark.parametrize("geom,detect,era,precision,first,thin", CASES)
def test_sums_equal_the_state_read_after_every_sweep(monkeypatch, geom, detect, era, precision, first, thin):
    spec = landscape(geom, detect, era, 60 + geom * 7 + detect)
    par = pdict(e=0.3, c=0.05, alpha=1 / 300, b=0.4, p=0.7, K=2.0, Ksrc=0.3 if era else 0.0, dsrc=40.0)
    sc = mb.engine.sampler_config(sample_alpha=1, sample_p=detect, n_adapt=4)
    sums = {}
    for graph in ("1", "0"):
        monkeypatch.setenv("MP_GRAPH", graph)
        with make_engine(spec, n_chains=3, precision=precision, seed=5) as eng:
            eng.set_params([par] * 3)
            eng.init_chains(sc, disperse=True)
            eng.set_summaries(first, thin)
            want = host_sums(eng, spec, 12, first, thin)
            got = eng.summaries()
        sums[graph] = got
        assert got["nsamples"] == want["nsamples"] == 3 * len(range(first, 12, thin))
        assert np.array_equal(got["z_count"], want["z_count"]) and np.array_equal(got["y_count"], want["y_count"])
        rel_close(got["S_sum"], want["S_sum"], 1e-12)
        if precision == mb.FP64:
            rel_close(got["z_prob"], want["z_prob"], 1e-12)
        else:
            assert np.abs(got["z_prob"] - want["z_prob"]).max() <= 1e-5 * want["nsamples"]
        latent = (spec["obs"] == -1) | ((spec["obs"] == 0) & bool(detect))
        frac = got["z_prob"][latent] / got["nsamples"]
        assert ((frac > 0.01) & (frac < 0.99)).any()        # some latent cells are genuinely uncertain: the check has content
    for k in KEYS:
        assert np.array_equal(sums["1"][k], sums["0"][k]), k   # captured sweeps and eager sweeps add the same numbers


def grid_landscape(seed, n=6000):
    rng = np.random.default_rng(seed)
    spec, z, y = random_landscape(rng, n, 4, O.GEOM_COORDS, occ=0.5, miss=0.05, areas=True)
    return spec, z, y


@pytest.mark.parametrize("blocks", [False, True])
def test_sampler_is_untouched(blocks):
    """FP32, coordinates, N = 6,000: the culled y scan (by blocks or whole years); draws, state, S and scales are bit-identical
    with the summaries on and off."""
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
                eng.set_summaries(2, 1)
            eng.work_counters(reset=True)
            eng.sweep(16)
            zz, yy = eng.get_state()
            runs.append(dict(draws=eng.get_draws(), z=zz, y=yy, S=eng.get_connectivity(), scales=eng.get_scales(),
                             geo=eng.scan_geometry(), work=eng.work_counters()))
            if on:
                assert eng.summaries()["nsamples"] == 14 * C
    a, b = runs
    assert a["geo"]["culled"], a["geo"]
    for key in ("draws", "z", "y", "S", "scales"):
        assert np.array_equal(a[key], b[key]), key
    assert a["work"] == b["work"]


def example_posterior(obs, cells, prior_occ):
    """P(z_cell = 1 | data) = exp(L(data with the cell := 1) - L(data)), L the oracle's exact marginal likelihood.  An observed
    year-0 cell carries no prior term in L, so a year-0 cell takes the factor p0 of its latent state."""
    par = O.params(e=0.71, c=0.52, alpha=1 / 400)
    l0 = O.marginal_loglik(O.Model(obs, spacing=100.0, prior_occ=prior_occ), par)
    out = []
    for (t, k) in cells:
        o1 = obs.copy()
        o1[t, k] = 1
        p0 = float(np.float32(prior_occ)) if t == 0 else 1.0
        out.append(p0 * np.exp(O.marginal_loglik(O.Model(o1, spacing=100.0, prior_occ=prior_occ), par) - l0))
    return np.array(out)


@pytest.mark.parametrize("year0", [False, True])
def test_occupancy_matches_the_exact_posterior_of_the_example(example_obs, year0):
    obs = example_obs.copy()
    prior_occ = 0.5
    if year0:
        obs[0, 3] = -1
        prior_occ = 0.25
    cells = [tuple(c) for c in np.argwhere(obs == -1)]
    exact = example_posterior(obs, cells, prior_occ)
    if not year0:
        np.testing.assert_allclose(np.sort(exact), [0.3222, 0.3800, 0.6096], atol=6e-5)
    else:
        assert abs(exact[cells.index((0, 3))] - 0.1914) < 6e-5
    C, nbatch, per = 256, 20, 50
    with make_engine(dict(obs=obs, spacing=100.0, prior_occ=prior_occ), n_chains=C, precision=mb.FP64, seed=21) as eng:
        eng.set_params([pdict(e=0.71, c=0.52, alpha=1 / 400)] * C)
        eng.init_chains(mb.engine.sampler_config(sample_e=0, sample_c=0, n_adapt=0), disperse=False)   # keeps c as set
        eng.sweep(50)                                           # burn-in
        eng.set_summaries(eng.lib.mp_sweep_index(eng.h), 1)
        batches = []
        for _ in range(nbatch):
            eng.sweep(per)
            s = eng.summaries(reset=True)
            assert s["nsamples"] == per * C
            batches.append([s["z_prob"][t, k] / s["nsamples"] for (t, k) in cells])
            # the observed cells carry their indicator in every sample
            fixed = obs != -1
            assert np.array_equal(s["z_prob"][fixed], obs[fixed] * float(per * C))
    b = np.array(batches)
    mean, se = b.mean(axis=0), b.std(axis=0, ddof=1) / np.sqrt(nbatch)
    # a cell whose conditional is the same in every sample (the year-0 cell: its y is fixed by the observed 0 that follows) has
    # se = 0 and must equal the exact value to rounding
    assert (np.abs(mean - exact) <= 4 * se + 1e-12).all(), (mean, exact, se)


def test_chain_sharded_engines_add_up():
    spec = landscape(O.GEOM_COORDS, 1, True, 77)
    C = 4
    pars = [pdict(e=0.3, c=0.04 + 0.01 * c, alpha=1 / 300, b=0.4, p=0.7, K=2.0) for c in range(C)]
    sc = mb.engine.sampler_config(sample_alpha=1, sample_p=1, n_adapt=4)

    def run(n_chains, offset):
        with make_engine(spec, n_chains=n_chains, precision=mb.FP64, seed=3, chain_offset=offset) as eng:
            eng.set_params(pars[offset:offset + n_chains])
            eng.init_chains(sc, disperse=True)
            eng.set_summaries(1, 2)
            eng.sweep(9)
            return eng.summaries()

    whole = run(C, 0)
    parts = [run(C // 2, 0), run(C // 2, C // 2)]
    assert whole["nsamples"] == parts[0]["nsamples"] + parts[1]["nsamples"] == 4 * C
    for k in ("z_count", "y_count"):
        assert np.array_equal(parts[0][k].astype(np.int64) + parts[1][k], whole[k]), k
    for k in ("z_prob", "S_sum"):
        np.testing.assert_allclose(parts[0][k] + parts[1][k], whole[k], rtol=1e-12, atol=0)


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
        eng.set_summaries(1, 1)
        return eng

    ref = fresh(0)
    ref.sweep(nsw)
    want = ref.summaries()
    ref.close()
    engs = [fresh(d) for d in range(2)]
    mb.Engine.comm_init_all(engs)
    mb.Engine.sweep_sharded_all(engs, nsw)
    for e in engs:
        e.synchronize()
        got = e.summaries()
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
        eng.set_summaries(0, 1)
        eng.sweep(4)
        before = eng.summaries()
        z, y = eng.get_state()
        eng.forecast(3, 4, seed=1)
        eng.connectivity()
        eng.loglik()
        eng.loglik_host(eng.get_params(), z, y)
        eng.flip_delta(0, 1, 2)
        eng.simulate(pdict(e=0.3, c=0.05), z[0, -1], 3, nsims=2)
        after = eng.summaries()
        assert after["nsamples"] == before["nsamples"] == 4 * C
        for k in KEYS:
            assert np.array_equal(after[k], before[k]), k
        eng.sweep(2)                                             # and the sweeps go on adding
        assert eng.summaries()["nsamples"] == 6 * C


def test_rejected_calls():
    import ctypes as C
    spec = landscape(O.GEOM_LINEAR, 0, False, 3)
    with make_engine(spec, n_chains=2) as eng:
        lib = eng.lib
        assert lib.mp_get_summaries(eng.h, None, None, None, None, None, 0) == ERR_STATE
        assert lib.mp_set_summaries(eng.h, -1, 1) == ERR_ARG
        assert lib.mp_set_summaries(eng.h, 0, -1) == ERR_ARG
        assert lib.mp_get_summaries(eng.h, None, None, None, None, None, 0) == ERR_STATE
        eng.set_summaries(0, 1)
        ns = C.c_int64(-1)
        assert lib.mp_get_summaries(eng.h, C.byref(ns), None, None, None, None, 0) == 0 and ns.value == 0
        eng.set_summaries(0, 0)                                  # off: freed
        assert lib.mp_get_summaries(eng.h, None, None, None, None, None, 0) == ERR_STATE


def test_sweeps_that_would_overflow_the_counts_are_refused():
    """65,535 chains: 65,537 accumulated sweeps make 2^32 - 1 samples, one more is refused before anything is launched."""
    obs = np.array([[1, 0, -1, 1], [0, 1, 1, -1]], dtype=np.int8)
    C = 65535
    with make_engine(dict(obs=obs), n_chains=C, precision=mb.FP64) as eng:
        eng.init_chains(mb.engine.sampler_config(), disperse=False)
        eng.set_summaries(0, 1)
        assert eng.lib.mp_sweep(eng.h, 65538) == ERR_STATE
        assert b"2^32" in eng.lib.mp_last_error(eng.h)
        eng.set_summaries(10, 2)                                 # sweeps 10, 12, ..., 131,084: 65,538 qualifying
        assert eng.lib.mp_sweep(eng.h, 131085) == ERR_STATE
        assert eng.lib.mp_sweep_index(eng.h) == 0
        assert eng.summaries()["nsamples"] == 0


def read_table(path):
    return np.array([[float(v) for v in line.split()] for line in Path(path).read_text().splitlines() if line.strip()])


def test_driver_writes_the_posterior_occupancy(example_obs, tmp_path):
    subprocess.run(["make", "-C", str(ROOT / "driver")], check=True, capture_output=True)
    res = subprocess.run([str(ROOT / "driver" / "midaspom"), "-m", "400", "-d", "100", "-n", "20000", "-c", "16", "-i", str(EXAMPLE),
                          "-o", str(tmp_path / "post.txt"), "-O", str(tmp_path / "occ.txt")], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    occ = read_table(tmp_path / "occ.txt")
    obs = example_obs
    assert occ.shape == obs.shape
    fixed = obs != -1
    assert np.array_equal(occ[fixed], obs[fixed].astype(np.float64))
    _, ltot, _ = mb.engine.exact_posterior(obs)
    for (t, k) in np.argwhere(obs == -1):
        o1 = obs.copy()
        o1[t, k] = 1
        _, l1, _ = mb.engine.exact_posterior(o1)
        assert abs(occ[t, k] - np.exp(l1 - ltot)) < 0.02, (t, k, occ[t, k], np.exp(l1 - ltot))
