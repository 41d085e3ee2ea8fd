"""GPU tests of mp_forecast, the posterior-predictive forecast from the chains' own state: every trajectory against the CPU
twin's spom_simulate, against mp_simulate_ensemble fed the same parameters and start states, culled against unculled, the
sampler left untouched, chain sharding, and the rejected arguments."""
import numpy as np
import pytest

import midaspom_b200 as mb
import oracle_lib as O
from gpu_util import make_engine, make_model, pdict, oparams, random_landscape

pytestmark = pytest.mark.gpu

SCEN = dict(K=1.8, Ksrc=0.6, dsrc=80.0)
ERR_ARG, ERR_STATE = -1, -3


def chain_params(C):
    return [pdict(e=0.3 + 0.1 * c, c=0.04 + 0.01 * c, alpha=1 / (400 + 100 * c), b=0.4, K=1.2 + 0.1 * c, Ksrc=0.2, dsrc=50.0)
            for c in range(C)]


def chain_state(rng, C, T, n, occ=0.45):
    z = (rng.random((C, T, n)) < occ).astype(np.uint8)
    y = (z[:, :-1] & z[:, 1:]).astype(np.uint8)
    return z, y


def with_scenario(par, scenario):
    if scenario is None:
        return dict(par)
    return dict(par, K=scenario["K"], Ksrc=scenario["Ksrc"], dsrc=scenario["dsrc"])


def ensemble_of(eng, nyears, nrep, seed, scenario):
    """The same trajectories through mp_simulate_ensemble: simulation c * nrep + r from chain c's parameters and z[c][T-1]."""
    pars = eng.get_params()
    z, _ = eng.get_state()
    sims = [with_scenario(pars[c], scenario) for c in range(eng.C) for _ in range(nrep)]
    z0 = np.repeat(z[:, -1, :], nrep, axis=0)
    _, occ = eng.simulate_ensemble(sims, z0, nyears, seed=seed, era_all=scenario is not None)
    return occ.reshape(eng.C, nrep, nyears + 1)


@pytest.mark.parametrize("geom,n,C,nrep,years,scenario,offset", [
    (O.GEOM_LINEAR, 50, 2, 3, 8, None, 0),
    (O.GEOM_LINEAR, 60, 2, 5, 6, SCEN, 3),
    (O.GEOM_COORDS, 120, 2, 40, 5, SCEN, 0),       # 40 replicates: two record words per chain
    (O.GEOM_COORDS, 700, 2, 3, 4, None, 1),        # several target tiles
    (O.GEOM_DENSE, 90, 3, 4, 5, SCEN, 0),
])
def test_forecast_follows_the_cpu_twin(geom, n, C, nrep, years, scenario, offset):
    rng = np.random.default_rng(40 + n)
    spec, _, _ = random_landscape(rng, n, 3, geom, areas=True)
    z, y = chain_state(rng, C, 3, n)
    pars = chain_params(C)
    spec_o = dict(spec)
    if scenario is not None:
        spec_o["era"] = np.ones(years, dtype=np.uint8)
    m = make_model(spec_o)
    with make_engine(spec, n_chains=C, precision=mb.FP64, chain_offset=offset) as eng:
        eng.set_params(pars)
        eng.set_state(z, y)
        occ, inc = eng.forecast(years, nrep, seed=7, scenario=scenario)
    want_inc = np.zeros((years + 1, n), dtype=np.int64)
    for c in range(C):
        for r in range(nrep):
            want = O.simulate(m, oparams(with_scenario(pars[c], scenario)), 7, (offset + c) * nrep + r, z[c, -1], years)
            assert (occ[c, r] == want.sum(axis=1)).all(), (c, r)
            want_inc += want
    assert (inc == want_inc).all()
    assert occ[:, :, -1].sum() > 0                  # the trajectories do not all die out: the comparison has content


@pytest.mark.parametrize("precision", [mb.FP64, mb.FP32])
@pytest.mark.parametrize("scenario", [None, SCEN])
def test_forecast_equals_simulate_ensemble(monkeypatch, precision, scenario):
    monkeypatch.setenv("MP_CONN_CULL", "0")         # FP32: the culled forecast is compared in test_culling_is_harmless
    rng = np.random.default_rng(11)
    n, T, C, nrep, years = 600, 6, 4, 32, 12
    spec, z, _ = random_landscape(rng, n, T, O.GEOM_COORDS, occ=0.5, areas=True)
    with make_engine(spec, n_chains=C, precision=precision, max_draws=8, seed=3) as eng:
        eng.set_params([pdict(e=0.3, c=0.02, alpha=1 / 400, b=0.3)] * C)
        eng.init_chains(mb.engine.sampler_config(sample_alpha=1, n_adapt=4), disperse=True)
        eng.sweep(5)
        occ, inc = eng.forecast(years, nrep, seed=9, scenario=scenario)
        ens = ensemble_of(eng, years, nrep, 9, scenario)
    same = (occ == ens).all(axis=2)
    if precision == mb.FP64:
        assert same.all()
    else:
        assert same.mean() >= 0.99, same.mean()
    assert (inc.astype(np.int64).sum(axis=1) == occ.astype(np.int64).sum(axis=(0, 1))).all()


def test_culling_is_harmless(monkeypatch):
    rng = np.random.default_rng(5)
    n, C, nrep, years = 20000, 4, 32, 8
    spec, _, _ = random_landscape(rng, n, 3, O.GEOM_COORDS, areas=True)
    z, y = chain_state(rng, C, 3, n, occ=0.4)
    pars = [pdict(e=0.3, c=0.004 + 0.001 * c, alpha=1 / (400 + 50 * c), b=0.5) for c in range(C)]
    out = {}
    for cull in ("1", "0"):
        monkeypatch.setenv("MP_CONN_CULL", cull)
        with make_engine(spec, n_chains=C, precision=mb.FP32) as eng:
            eng.set_params(pars)
            eng.set_state(z, y)
            eng.work_counters(reset=True)
            occ, inc = eng.forecast(years, nrep, seed=2, scenario=SCEN)
            out[cull] = (occ, inc, eng.work_counters())
    (occ1, _, w1), (occ0, _, w0) = out["1"], out["0"]
    same = (occ1 == occ0).all(axis=2)
    assert same.mean() >= 0.99, same.mean()
    assert w1["conn_total"] == w0["conn_total"] > 0
    assert w0["conn_exec"] == w0["conn_total"]
    assert w1["conn_exec"] < w1["conn_total"]         # source tiles out of reach were skipped


@pytest.mark.parametrize("precision", [mb.FP64, mb.FP32])
def test_sampler_is_untouched(precision):
    rng = np.random.default_rng(8)
    n, T, C = 400, 5, 2
    spec, _, _ = random_landscape(rng, n, T, O.GEOM_COORDS, occ=0.5, areas=True)
    sc = mb.engine.sampler_config(sample_alpha=1, n_adapt=6)
    runs = []
    for with_forecast in (True, False):
        with make_engine(spec, n_chains=C, precision=precision, max_draws=20, seed=4) as eng:
            eng.set_params([pdict(e=0.3, c=0.02, alpha=1 / 400, b=0.3)] * C)
            eng.init_chains(sc, disperse=True)
            eng.sweep(10)
            if with_forecast:
                eng.forecast(6, 8, seed=1, scenario=SCEN)
            eng.sweep(10)
            z, yy = eng.get_state()
            runs.append(dict(draws=eng.get_draws(), z=z, y=yy, scales=eng.get_scales(), S=eng.get_connectivity(),
                             sweep=eng.lib.mp_sweep_index(eng.h)))
    a, b = runs
    assert a["sweep"] == b["sweep"] == 20
    for key in ("draws", "z", "y", "scales", "S"):
        assert np.array_equal(a[key], b[key]), key


@pytest.mark.parametrize("precision", [mb.FP64, mb.FP32])
def test_sharded_chains_give_the_same_forecast(precision):
    rng = np.random.default_rng(9)
    n, T, C, nrep, years = 900, 3, 4, 6, 6
    spec, _, _ = random_landscape(rng, n, T, O.GEOM_COORDS, areas=True)
    z, y = chain_state(rng, C, T, n)
    pars = chain_params(C)
    with make_engine(spec, n_chains=C, precision=precision) as eng:
        eng.set_params(pars)
        eng.set_state(z, y)
        occ, inc = eng.forecast(years, nrep, seed=3, scenario=SCEN)
    parts = []
    for off in (0, C // 2):
        sl = slice(off, off + C // 2)
        with make_engine(spec, n_chains=C // 2, precision=precision, chain_offset=off) as eng:
            eng.set_params(pars[sl])
            eng.set_state(z[sl], y[sl])
            parts.append(eng.forecast(years, nrep, seed=3, scenario=SCEN))
    assert np.array_equal(np.concatenate([p[0] for p in parts]), occ)
    assert np.array_equal(parts[0][1].astype(np.int64) + parts[1][1], inc)


def test_rejected_arguments_leave_the_engine_usable():
    import ctypes as C
    from midaspom_b200.distributed import engine_tensor
    rng = np.random.default_rng(2)
    n, T, nch = 64, 3, 2
    spec, _, _ = random_landscape(rng, n, T, O.GEOM_LINEAR, areas=False)
    z, y = chain_state(rng, nch, T, n)

    def call(eng, nyears=3, nrep=2, scenario=None):
        scen = None if scenario is None else (C.c_double * 3)(*scenario)
        return eng.lib.mp_forecast(eng.h, nyears, nrep, 1, scen, None, None)

    with mb.Engine(n, T, nch, precision=mb.FP64) as bare:      # no landscape
        assert call(bare) == ERR_STATE
        bare.set_landscape_linear(100.0)
        assert call(bare) == ERR_STATE                             # no chain state
    with make_engine(spec, n_chains=nch) as eng:
        pars = chain_params(nch)
        eng.set_params(pars)
        eng.set_state(z, y)
        assert call(eng, nyears=0) == ERR_ARG
        assert call(eng, nrep=0) == ERR_ARG
        assert call(eng, scenario=(0.0, 0.0, 0.0)) == ERR_ARG
        assert call(eng, scenario=(-1.0, 0.0, 0.0)) == ERR_ARG
        assert b"nrep" in eng.lib.mp_last_error(eng.h) or b"K" in eng.lib.mp_last_error(eng.h)
        import torch
        par = engine_tensor(eng, 4, (nch, 8), "<f8", "cuda:0")       # MP_BUF_PARAMS; alpha is field 2
        par[1, 2] = 0.0
        torch.cuda.synchronize()
        assert call(eng) == ERR_STATE
        eng.set_params(pars)
        occ, inc = eng.forecast(3, 2, seed=1)
        assert occ.shape == (nch, 2, 4) and inc.shape == (4, n)
        assert (occ[:, :, 0] == z[:, -1].sum(axis=1)[:, None]).all()
        assert (inc[0] == 2 * z[:, -1].sum(axis=0)).all()
