"""GPU tests of mp_ppc, the posterior-predictive replicates of the observation table: every statistic against the CPU twin's
spom_simulate with a host replay of the observation step, the occupied counts of mp_simulate_ensemble, culled against
unculled connectivity, the sampler (summaries and WAIC sums included) left untouched, chain sharding, misfit detected on
die-off data and not on data the model generated, and the rejected calls."""
import numpy as np
import pytest

import midaspom_b200 as mb
import oracle_lib as O
from gpu_util import make_engine, make_model, pdict, oparams, random_landscape
from test_gpu_fp32_decisions import rng as philox, u01
from midaspom_b200 import synth

pytestmark = pytest.mark.gpu

RK_PPC_DET = 14
ERR_ARG, ERR_STATE = -1, -3
MIXED = (1, 1, 0, 0, 1, 0, 1)


def chain_params(C):
    return [pdict(e=0.3 + 0.1 * c, c=0.04 + 0.01 * c, alpha=1 / (400 + 100 * c), b=0.4, p=0.7, K=1.2 + 0.1 * c, Ksrc=0.2, dsrc=50.0)
            for c in range(C)]


def chain_state(rng, C, T, n, occ=0.45):
    z = (rng.random((C, T, n)) < occ).astype(np.uint8)
    y = (z[:, :-1] & z[:, 1:]).astype(np.uint8)
    return z, y


def statistics(rep):
    """rep [T, N] (-1 missing, 0, 1) -> [T, 3] detected, colonised, extinct (DESIGN §2)."""
    T = rep.shape[0]
    out = np.zeros((T, 3), dtype=np.int64)
    out[:, 0] = (rep == 1).sum(axis=1)
    both = (rep[1:] >= 0) & (rep[:-1] >= 0)
    out[1:, 1] = (both & (rep[:-1] == 0) & (rep[1:] == 1)).sum(axis=1)
    out[1:, 2] = (both & (rep[:-1] == 1) & (rep[1:] == 0)).sum(axis=1)
    return out


def host_ppc(spec, pars, z, nrep, seed, offset):
    """The CPU twin: spom_simulate from z[c][0] under the model's era flags for simulation (offset + c) nrep + r, then the
    observation step with the host Philox.  Returns stats [C, nrep, T, 3], obs_stats, patch_ge, patch_gt."""
    m = make_model(spec)
    obs = np.asarray(spec["obs"])
    T, n = obs.shape
    detect = spec.get("detect", 0)
    C = len(pars)
    stats = np.zeros((C, nrep, T, 3), dtype=np.int64)
    d_obs = (obs == 1).sum(axis=0)
    ge, gt = np.zeros(n, dtype=np.int64), np.zeros(n, dtype=np.int64)
    tt, kk = np.meshgrid(np.arange(T, dtype=np.uint32), np.arange(n, dtype=np.uint32), indexing="ij")
    for c in range(C):
        for r in range(nrep):
            sim = (offset + c) * nrep + r
            traj = O.simulate(m, oparams(pars[c]), seed, sim, z[c, 0], T - 1).astype(np.int64)
            if detect:
                u = u01(philox(seed, sim, tt, RK_PPC_DET, kk, 0)[0])
                traj = traj & (u < pars[c]["p"])
            rep = np.where(obs >= 0, traj, -1)
            stats[c, r] = statistics(rep)
            d = (rep == 1).sum(axis=0)
            ge += d >= d_obs
            gt += d > d_obs
    return stats, statistics(obs), ge, gt


@pytest.mark.parametrize("geom,n,C,nrep,T,era,detect,offset", [
    (O.GEOM_LINEAR, 50, 2, 3, 8, None, 0, 0),
    (O.GEOM_LINEAR, 60, 3, 5, 6, MIXED[:5], 1, 3),
    (O.GEOM_COORDS, 120, 2, 40, 5, MIXED[:4], 1, 0),     # 40 replicates: two record words per chain
    (O.GEOM_COORDS, 700, 2, 3, 4, None, 1, 1),           # several target tiles
    (O.GEOM_DENSE, 90, 3, 4, 6, MIXED[:5], 0, 0),
])
def test_ppc_follows_the_cpu_twin(geom, n, C, nrep, T, era, detect, offset):
    rng = np.random.default_rng(70 + n)
    spec, _, _ = random_landscape(rng, n, T, geom, occ=0.5, miss=0.15, areas=True)
    spec["detect"] = detect
    if era is not None:
        spec["era"] = np.array(era, dtype=np.uint8)
    assert (spec["obs"][0] == -1).any() and (spec["obs"][1:] == -1).any()
    z, y = chain_state(rng, C, T, n)
    pars = chain_params(C)
    with make_engine(spec, n_chains=C, precision=mb.FP64, chain_offset=offset) as eng:
        eng.set_params(pars)
        eng.set_state(z, y)
        got = eng.ppc(nrep, seed=7)
    stats, obs_stats, ge, gt = host_ppc(spec, pars, z, nrep, 7, offset)
    assert got["nrep_total"] == C * nrep
    assert np.array_equal(got["stats"], stats)
    assert np.array_equal(got["obs_stats"], obs_stats)
    assert np.array_equal(got["patch_ge"], ge) and np.array_equal(got["patch_gt"], gt)
    assert got["stats"][:, :, -1, 0].sum() > 0            # the replicates do not all die out: the comparison has content
    assert (got["stats"][:, :, 1:, 1:] > 0).any(axis=(0, 1, 2)).all()


@pytest.mark.parametrize("precision", [mb.FP64, mb.FP32])
@pytest.mark.parametrize("era_all", [False, True])
def test_detected_counts_equal_simulate_ensemble(monkeypatch, precision, era_all):
    monkeypatch.setenv("MP_CONN_CULL", "0")             # FP32: the culled connectivity is compared in test_culling_is_harmless
    rng = np.random.default_rng(12)
    n, T, C, nrep = 600, 10, 4, 32
    spec, _, _ = random_landscape(rng, n, T, O.GEOM_COORDS, occ=0.5, areas=True)
    if era_all:
        spec["era"] = np.ones(T - 1, dtype=np.uint8)
    with make_engine(spec, n_chains=C, precision=precision, max_draws=8, seed=3) as eng:
        eng.set_params([pdict(e=0.3, c=0.02, alpha=1 / 400, b=0.3, K=1.5)] * C)
        eng.init_chains(mb.engine.sampler_config(sample_alpha=1, n_adapt=4), disperse=True)
        eng.sweep(5)
        got = eng.ppc(nrep, seed=9)
        pars = eng.get_params()
        z, _ = eng.get_state()
        sims = [pars[c] for c in range(C) for _ in range(nrep)]
        _, occ = eng.simulate_ensemble(sims, np.repeat(z[:, 0, :], nrep, axis=0), T - 1, seed=9, era_all=era_all)
    same = (got["stats"][:, :, :, 0] == occ.reshape(C, nrep, T)).all(axis=2)
    if precision == mb.FP64:
        assert same.all()
    else:
        assert same.mean() >= 0.99, same.mean()


def test_culling_is_harmless(monkeypatch):
    rng = np.random.default_rng(6)
    n, T, C, nrep = 20000, 8, 4, 32
    spec, _, _ = random_landscape(rng, n, T, O.GEOM_COORDS, occ=0.4, miss=0.05, areas=True)
    spec["era"] = np.array(MIXED, dtype=np.uint8)
    z, y = chain_state(rng, C, T, n, occ=0.4)
    pars = [pdict(e=0.3, c=0.004 + 0.001 * c, alpha=1 / (400 + 50 * c), b=0.5, K=1.8, Ksrc=0.6, dsrc=80.0) for c in range(C)]
    out = {}
    for cull in ("1", "0"):
        monkeypatch.setenv("MP_CONN_CULL", cull)
        with make_engine(spec, n_chains=C, precision=mb.FP32) as eng:
            eng.set_params(pars)
            eng.set_state(z, y)
            eng.work_counters(reset=True)
            out[cull] = (eng.ppc(nrep, seed=2), eng.work_counters())
    (r1, w1), (r0, w0) = out["1"], out["0"]
    same = (r1["stats"] == r0["stats"]).all(axis=(2, 3))
    assert same.mean() >= 0.99, same.mean()
    assert w1["conn_total"] == w0["conn_total"] > 0
    assert w0["conn_exec"] == w0["conn_total"]
    assert w1["conn_exec"] < w1["conn_total"]             # source tiles out of reach were skipped


@pytest.mark.parametrize("graph", ["1", "0"])
@pytest.mark.parametrize("precision", [mb.FP64, mb.FP32])
def test_sampler_is_untouched(monkeypatch, graph, precision):
    monkeypatch.setenv("MP_GRAPH", graph)
    rng = np.random.default_rng(8)
    n, T, C = 400, 5, 2
    spec, _, _ = random_landscape(rng, n, T, O.GEOM_COORDS, occ=0.5, miss=0.1, areas=True)
    spec["era"] = np.array(MIXED[:T - 1], dtype=np.uint8)
    sc = mb.engine.sampler_config(sample_alpha=1, n_adapt=6)
    runs = []
    for with_ppc in (True, False):
        with make_engine(spec, n_chains=C, precision=precision, max_draws=20, seed=4) as eng:
            eng.set_params([pdict(e=0.3, c=0.02, alpha=1 / 400, b=0.3, K=1.5)] * C)
            eng.init_chains(sc, disperse=True)
            eng.set_summaries(2, 1)
            eng.set_waic(1, 2)
            eng.sweep(10, sync=False)                      # queued sweeps: mp_ppc runs after them
            if with_ppc:
                eng.ppc(8, seed=1)
                before = (eng.summaries(), eng.waic_sums())
            eng.sweep(10)
            zz, yy = eng.get_state()
            runs.append(dict(draws=eng.get_draws(), z=zz, y=yy, scales=eng.get_scales(), S=eng.get_connectivity(),
                             sweep=eng.lib.mp_sweep_index(eng.h), summaries=eng.summaries(), waic=eng.waic_sums()))
            if with_ppc:
                eng.ppc(8, seed=2)
                assert all(np.array_equal(eng.summaries()[k], runs[-1]["summaries"][k]) for k in runs[-1]["summaries"])
                assert all(np.array_equal(eng.waic_sums()[k], runs[-1]["waic"][k]) for k in runs[-1]["waic"])
    a, b = runs
    assert before[0]["nsamples"] == 8 * C and before[1]["nsamples"] == 5 * C
    assert a["sweep"] == b["sweep"] == 20
    for key in ("draws", "z", "y", "scales", "S"):
        assert np.array_equal(a[key], b[key]), key
    for key in ("summaries", "waic"):
        for k in a[key]:
            assert np.array_equal(a[key][k], b[key][k]), (key, k)


@pytest.mark.parametrize("precision", [mb.FP64, mb.FP32])
def test_sharded_chains_give_the_same_replicates(precision):
    rng = np.random.default_rng(9)
    n, T, C, nrep = 900, 6, 4, 6
    spec, _, _ = random_landscape(rng, n, T, O.GEOM_COORDS, miss=0.1, areas=True)
    spec["detect"] = 1
    spec["era"] = np.array(MIXED[:T - 1], dtype=np.uint8)
    z, y = chain_state(rng, C, T, n)
    pars = chain_params(C)
    with make_engine(spec, n_chains=C, precision=precision) as eng:
        eng.set_params(pars)
        eng.set_state(z, y)
        whole = eng.ppc(nrep, seed=3)
    parts = []
    for off in (0, C // 2):
        sl = slice(off, off + C // 2)
        with make_engine(spec, n_chains=C // 2, precision=precision, chain_offset=off) as eng:
            eng.set_params(pars[sl])
            eng.set_state(z[sl], y[sl])
            parts.append(eng.ppc(nrep, seed=3))
    assert np.array_equal(np.concatenate([p["stats"] for p in parts]), whole["stats"])
    for k in ("patch_ge", "patch_gt"):
        assert np.array_equal(parts[0][k].astype(np.int64) + parts[1][k], whole[k]), k
    assert all(np.array_equal(p["obs_stats"], whole["obs_stats"]) for p in parts)
    a, b = mb.ppc_check(whole), mb.ppc_check(*parts)
    for k in ("p_year", "p_omnibus", "p_patch"):
        assert np.array_equal(a[k], b[k]), k


def fit_ppc(wl, era, sample_K, K0, chains=8, burn=300, every=50, calls=6, nrep=32):
    """8 FP32 chains on a synthetic workload; one mp_ppc call every `every` sweeps after the burn-in, pooled."""
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
        res = []
        for i in range(calls):
            eng.sweep(every)
            res.append(eng.ppc(nrep, seed=100 + i))
        return mb.ppc_check(*res)
    finally:
        eng.close()


@pytest.mark.parametrize("name,hyp", [("cfg4", "H0"), ("cfg4", "H1"), ("cfg3", "H0")])
def test_ppc_detects_misfit_and_passes_a_correct_model(name, hyp):
    """Thresholds fixed before the first run: the die-off data (cfg4) fitted without an event fails on `detected` (omnibus
    p < 0.01); fitted as H1 (era flags on the first 10 transitions, K sampled) it passes on all three statistics (p >= 0.01),
    and so does the data without an event (cfg3) fitted as H0."""
    wl = synth.make_workload(name)
    era = (np.arange(wl["T"] - 1) < 10).astype(np.uint8) if hyp == "H1" else None
    r = fit_ppc(wl, era, 1 if hyp == "H1" else 0, 3.0 if hyp == "H1" else 1.0)
    print(name, hyp, "p_omnibus", dict(zip(mb.PPC_STATS, r["p_omnibus"].round(4))), "D_obs", r["D_obs"].round(1),
          "patches p<0.01:", int((r["p_patch"] < 0.01).sum()))
    assert r["nrep_total"] == 8 * 32 * 6
    if hyp == "H0" and name == "cfg4":
        assert r["p_omnibus"][0] < 0.01, r["p_omnibus"]
    else:
        assert (r["p_omnibus"] >= 0.01).all(), r["p_omnibus"]


def test_rejected_calls_leave_the_engine_usable():
    import ctypes as C
    from midaspom_b200.distributed import engine_tensor
    rng = np.random.default_rng(2)
    n, T, nch = 64, 4, 2
    spec, _, _ = random_landscape(rng, n, T, O.GEOM_LINEAR, miss=0.1, areas=False)
    z, y = chain_state(rng, nch, T, n)
    pars = chain_params(nch)

    def call(eng, nrep=2):
        return eng.lib.mp_ppc(eng.h, nrep, 1, None, None, None, None)

    with mb.Engine(n, T, nch, precision=mb.FP64) as bare:      # no landscape, no state, no observations
        assert call(bare) == ERR_STATE
        bare.set_landscape_linear(100.0)
        assert call(bare) == ERR_STATE                             # no chain state
        bare.set_params(pars)
        bare.set_state(z, y)
        assert call(bare) == ERR_STATE                             # no observations
        assert b"observations" in bare.lib.mp_last_error(bare.h)
    with make_engine(spec, n_chains=nch, chain_offset=2 ** 31 - 10) as far:
        far.set_params(pars)
        far.set_state(z, y)
        assert call(far, nrep=3) == ERR_ARG                        # (2^31 - 8) * 3 >= 2^32
        assert call(far, nrep=2) == 0                              # the last simulation number is 2^32 - 17
    with make_engine(spec, n_chains=nch) as eng:
        eng.set_params(pars)
        eng.set_state(z, y)
        assert call(eng, nrep=0) == ERR_ARG
        assert call(eng, nrep=65536) == ERR_ARG
        assert b"nrep" in eng.lib.mp_last_error(eng.h)
        import torch
        par = engine_tensor(eng, 4, (nch, 8), "<f8", "cuda:0")       # MP_BUF_PARAMS; alpha is field 2
        par[1, 2] = 0.0
        torch.cuda.synchronize()
        assert call(eng) == ERR_STATE
        eng.set_params(pars)
        got = eng.ppc(3, seed=1)
    obs = spec["obs"]
    assert got["stats"].shape == (nch, 3, T, 3) and got["obs_stats"].shape == (T, 3)
    # without detection year 0 is the chain's own year 0 seen through the mask
    want0 = ((obs[0] >= 0)[None] & (z[:, 0] == 1)).sum(axis=1)
    assert (got["stats"][:, :, 0, 0] == want0[:, None]).all()
    assert (got["stats"][:, :, 0, 1:] == 0).all()
