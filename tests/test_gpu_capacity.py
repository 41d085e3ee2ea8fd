"""GPU tests of mp_capacity, the metapopulation capacity lambda_M and the patch values of the landscape: the FP64 engine against
numpy.linalg.eigh of the matrix built here (linear, planar and dense landscapes, a strongly localised Perron vector), the cfg3
values, FP32 against FP64 and culled against unculled products, patch masks, determinism across batches and engines, the sampler
left untouched, unconverged sets, the rejected calls, and the persistence threshold R = 1 against forecasts of the model itself."""
import numpy as np
import pytest

import midaspom_b200 as mb
import oracle_lib as O
from gpu_util import make_engine, pdict, random_landscape

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_STATE, ERR_UNSUPPORTED = -1, -3, -4


def distances(spec, n):
    if spec["geom"] == O.GEOM_LINEAR:
        i = np.arange(n, dtype=np.float64)
        return np.abs(i[:, None] - i[None, :]) * spec.get("spacing", 100.0)
    if spec["geom"] == O.GEOM_COORDS:
        return np.sqrt((spec["px"][:, None] - spec["px"][None, :]) ** 2 + (spec["py"][:, None] - spec["py"][None, :]) ** 2)
    return np.asarray(spec["dist"], dtype=np.float64)


def mtilde(spec, n, alpha, b, keep=None):
    """M~_kl = sqrt(a_k a_l) exp(-alpha d_kl), zero diagonal, a = A^b (DESIGN.md §2); the principal submatrix of keep."""
    a = np.asarray(spec.get("area", np.ones(n)), dtype=np.float64) ** b
    s = np.sqrt(a)
    M = np.exp(-alpha * distances(spec, n)) * np.outer(s, s)
    np.fill_diagonal(M, 0.0)
    if keep is not None:
        idx = np.flatnonzero(keep)
        M = M[np.ix_(idx, idx)]
    return M


def eig_ref(M):
    w, V = np.linalg.eigh(M)
    return w[-1], w[-1] - w[-2], V[:, -1] ** 2


def spec_of(rng, geom, n):
    spec, _, _ = random_landscape(rng, n, 3, geom, areas=True)
    return spec


def engine_for(spec, n, precision=mb.FP64, n_chains=1, chain_offset=0):
    spec = dict(spec)
    spec["obs"] = np.zeros((3, n), dtype=np.int8)
    return make_engine(spec, n_chains=n_chains, precision=precision, chain_offset=chain_offset)


def check_against_eigh(res, i, M, keep=None, rtol=1e-9, lam_tol=1e-10):
    lam, gap, v = eig_ref(M)
    assert abs(res["lam"][i] - lam) <= lam_tol * lam, (res["lam"][i], lam)
    assert res["residual"][i] <= rtol
    V = res["values"][i]
    if keep is not None:
        assert np.all(V[keep == 0] == 0.0)
        V = V[keep != 0]
    assert abs(V.sum() - 1.0) < 1e-12
    tol = 4.0 * res["residual"][i] * lam / gap + 1e-12       # Davis-Kahan: sin of the vector error <= ||r|| / gap
    assert np.max(np.abs(V - v)) <= tol, (np.max(np.abs(V - v)), tol)


CASES = [(O.GEOM_LINEAR, 300), (O.GEOM_COORDS, 2000), (O.GEOM_DENSE, 500)]
PARAMS = [(1 / 400, 0.5), (1 / 150, 1.0), (1 / 2000, 0.0), (1 / 40, 1.5)]   # the last: a strongly localised Perron vector


@pytest.mark.parametrize("geom,n", CASES)
def test_fp64_against_eigh(geom, n):
    rng = np.random.default_rng(1 + geom)
    spec = spec_of(rng, geom, n)
    with engine_for(spec, n) as eng:
        res = eng.capacity([pdict(alpha=a, b=b) for a, b in PARAMS], rtol=1e-9, values=True)
    for i, (a, b) in enumerate(PARAMS):
        check_against_eigh(res, i, mtilde(spec, n, a, b))
    assert np.all(res["cull_bound"] == 0.0) and np.all(res["iters"] >= 1)
    assert np.allclose(res["value_sum"], res["values"].sum(axis=0), rtol=1e-14, atol=0)
    V = res["values"][3]
    assert np.sort(V)[::-1][: n // 100 + 1].sum() > 0.5          # localised: 1 % of the patches hold most of the value


def cfg3_landscape(n=10000):
    rng = np.random.default_rng(12345)                        # the positions and areas of synth.make_workload("cfg3")
    side = np.sqrt(n) * 250.0
    px, py = rng.uniform(0, side, n), rng.uniform(0, side, n)
    area = np.random.default_rng(12346).lognormal(0.0, 0.5, n)
    return dict(geom=O.GEOM_COORDS, px=px, py=py, area=area)


def test_cfg3_values():
    spec = cfg3_landscape()
    # lambda_M from the FP64 matrix built in numpy; the localised case is alpha = 3/800 (1/266.7)
    want = {1 / 400: 18.07344621, 3 / 800: 8.960987965, 1 / 800: 65.935651}
    with engine_for(spec, 10000) as eng:
        res = eng.capacity([pdict(alpha=a, b=0.5) for a in want], rtol=1e-7, max_iter=5000)
    for i, (a, lam) in enumerate(want.items()):
        assert abs(res["lam"][i] - lam) <= 1e-8 * lam, (a, res["lam"][i], lam)
        assert res["residual"][i] <= 1e-7


def test_fp32_against_fp64():
    rng = np.random.default_rng(3)
    n = 2000
    spec = spec_of(rng, O.GEOM_COORDS, n)
    pars = [pdict(alpha=a, b=b) for a, b in PARAMS[:3]]
    out = {}
    for prec in (mb.FP64, mb.FP32):
        with engine_for(spec, n, precision=prec) as eng:
            out[prec] = eng.capacity(pars, rtol=1e-8)
    extent = np.hypot(np.ptp(spec["px"]), np.ptp(spec["py"]))
    for i, p in enumerate(pars):
        tol = 2 * p["alpha"] * extent * 2.0 ** -24 + 2.0 ** -21     # DESIGN.md §5: coordinate rounding + ex2
        d = abs(out[mb.FP32]["lam"][i] - out[mb.FP64]["lam"][i]) / out[mb.FP64]["lam"][i]
        assert d <= tol, (i, d, tol)


def test_culled_against_unculled(monkeypatch):
    rng = np.random.default_rng(4)
    n = 20000
    spec = spec_of(rng, O.GEOM_COORDS, n)
    pars = [pdict(alpha=1 / 400, b=0.5), pdict(alpha=1 / 200, b=1.0)]
    out = {}
    for cull in ("1", "0"):
        monkeypatch.setenv("MP_CONN_CULL", cull)
        with engine_for(spec, n, precision=mb.FP32) as eng:
            eng.work_counters(reset=True)
            out[cull] = (eng.capacity(pars, rtol=1e-8), eng.work_counters())
    (r1, w1), (r0, w0) = out["1"], out["0"]
    assert w0["conn_exec"] == w0["conn_total"] > 0
    assert w1["conn_exec"] < w1["conn_total"]                 # tiles were skipped
    assert np.all(r0["cull_bound"] == 0.0) and np.all(r1["cull_bound"] > 0.0) and np.all(r1["cull_bound"] <= 2.0 ** -30)
    for i in range(len(pars)):
        d = abs(r1["lam"][i] - r0["lam"][i]) / r0["lam"][i]
        assert d <= r1["cull_bound"][i] + 1e-9, (i, d, r1["cull_bound"][i])


def test_keep_mask():
    rng = np.random.default_rng(5)
    n = 800
    spec = spec_of(rng, O.GEOM_COORDS, n)
    keep = (rng.random(n) < 0.7).astype(np.uint8)
    pars = [pdict(alpha=1 / 400, b=0.5), pdict(alpha=1 / 100, b=1.0)]
    with engine_for(spec, n) as eng:
        res = eng.capacity(pars, keep=keep, rtol=1e-9, values=True)
        full = eng.capacity(pars, rtol=1e-9, values=True)
        ones = eng.capacity(pars, keep=np.ones(n, dtype=np.uint8), rtol=1e-9, values=True)
    for i, p in enumerate(pars):
        check_against_eigh(res, i, mtilde(spec, n, p["alpha"], p["b"], keep), keep=keep)
    for k in ("lam", "residual", "cull_bound", "iters", "values", "value_sum"):
        assert np.array_equal(full[k], ones[k]), k
    assert np.all(res["lam"] < full["lam"])                   # Perron monotonicity


@pytest.mark.parametrize("precision", [mb.FP32, mb.FP64])
def test_determinism(precision):
    rng = np.random.default_rng(6)
    n, C = 1500, 4
    spec = spec_of(rng, O.GEOM_COORDS, n)
    many = [pdict(alpha=1 / rng.uniform(150, 800), b=rng.uniform(0, 1)) for _ in range(64)]
    keep = (rng.random(n) < 0.9).astype(np.uint8)
    with engine_for(spec, n, precision=precision, n_chains=C) as eng:
        all64 = eng.capacity(many, keep=keep, values=True)
        alone = eng.capacity([many[37]], keep=keep, values=True)
        eng.set_params(many[:C])
        resident = eng.capacity(None, keep=keep, values=True)
        given = eng.capacity(eng.get_params(), keep=keep, values=True)
    with engine_for(spec, n, precision=precision, n_chains=1, chain_offset=5) as other:
        shard = other.capacity([many[37]], keep=keep, values=True)
    for k in ("lam", "residual", "cull_bound", "iters", "values"):
        assert np.array_equal(alone[k][0], all64[k][37]), k
        assert np.array_equal(shard[k][0], all64[k][37]), k
        assert np.array_equal(resident[k], given[k]), k
        assert np.array_equal(resident[k], all64[k][:C]), k
    assert np.array_equal(resident["value_sum"], given["value_sum"])


@pytest.mark.parametrize("graph", ["1", "0"])
@pytest.mark.parametrize("precision", [mb.FP64, mb.FP32])
def test_sampler_is_untouched(monkeypatch, graph, precision):
    monkeypatch.setenv("MP_GRAPH", graph)
    rng = np.random.default_rng(8)
    n, T, C = 400, 5, 2
    spec, _, _ = random_landscape(rng, n, T, O.GEOM_COORDS, occ=0.5, miss=0.1, areas=True)
    sc = mb.engine.sampler_config(sample_alpha=1, n_adapt=6)
    runs = []
    for with_cap in (True, False):
        with make_engine(spec, n_chains=C, precision=precision, max_draws=20, seed=4) as eng:
            eng.set_params([pdict(e=0.3, c=0.02, alpha=1 / 400, b=0.3)] * C)
            eng.init_chains(sc, disperse=True)
            eng.set_summaries(2, 1)
            eng.set_waic(1, 2)
            eng.sweep(10, sync=False)                          # queued sweeps: mp_capacity runs after them
            if with_cap:
                eng.capacity(None, values=True)
            eng.sweep(10)
            zz, yy = eng.get_state()
            runs.append(dict(draws=eng.get_draws(), z=zz, y=yy, scales=eng.get_scales(), S=eng.get_connectivity(),
                             sweep=eng.lib.mp_sweep_index(eng.h), summaries=eng.summaries(), waic=eng.waic_sums()))
            if with_cap:
                eng.capacity([pdict(alpha=1 / 300, b=0.5)])
                assert all(np.array_equal(eng.summaries()[k], runs[-1]["summaries"][k]) for k in runs[-1]["summaries"])
                assert all(np.array_equal(eng.waic_sums()[k], runs[-1]["waic"][k]) for k in runs[-1]["waic"])
    a, b = runs
    assert a["sweep"] == b["sweep"] == 20
    for key in ("draws", "z", "y", "scales", "S"):
        assert np.array_equal(a[key], b[key]), key
    for key in ("summaries", "waic"):
        for k in a[key]:
            assert np.array_equal(a[key][k], b[key][k]), (key, k)


def test_unconverged_sets_are_reported():
    rng = np.random.default_rng(9)
    n = 2000
    spec = spec_of(rng, O.GEOM_COORDS, n)
    with engine_for(spec, n) as eng:
        res = eng.capacity([pdict(alpha=1 / 267, b=0.5)], rtol=1e-12, max_iter=2)
    assert res["iters"][0] == 2 and res["residual"][0] > 1e-12 and np.isfinite(res["lam"][0])


def test_rejected_calls():
    rng = np.random.default_rng(10)
    n = 200
    spec = spec_of(rng, O.GEOM_COORDS, n)
    p = [pdict(alpha=1 / 400, b=0.5)]
    with mb.Engine(n, 3, 2, precision=mb.FP64) as eng:
        out3 = np.zeros(3)
        assert eng.lib.mp_capacity(eng.h, 1, eng._params_array([p[0]] * 2), None, 1e-6, 10, out3.ctypes.data_as(mb.engine._dp),
                                   None, None, None) == ERR_STATE          # no landscape
        eng.set_landscape_coords(spec["px"], spec["py"], spec["area"])
        with pytest.raises(mb.MpError, match=r"\(-3\)"):
            eng.capacity(None)                                 # no chain parameters yet
        for kw in (dict(rtol=0.0), dict(rtol=-1.0), dict(max_iter=0)):
            with pytest.raises(mb.MpError, match=r"\(-1\)"):
                eng.capacity(p, **kw)
        with pytest.raises(mb.MpError, match=r"\(-1\)"):
            eng.capacity([pdict(alpha=0.0, b=0.5)])
        with pytest.raises(mb.MpError, match=r"\(-1\)"):
            eng.capacity([pdict(alpha=-1.0, b=0.5)])
        keep = np.zeros(n, dtype=np.uint8)
        keep[3] = 1
        with pytest.raises(mb.MpError, match=r"\(-1\)"):
            eng.capacity(p, keep=keep)
        assert eng.lib.mp_capacity(eng.h, 0, eng._params_array([p[0]] * 2), None, 1e-6, 10, out3.ctypes.data_as(mb.engine._dp),
                                   None, None, None) == ERR_ARG
        keep[4] = 1
        assert eng.capacity(p, keep=keep)["lam"][0] > 0.0       # two kept patches suffice
    d = distances(spec, n)
    d[3, 7] += 1.0                                             # not symmetric
    for prec in (mb.FP64, mb.FP32):
        with mb.Engine(n, 3, 1, precision=prec) as eng:
            eng.set_landscape_dense(d, spec["area"])
            with pytest.raises(mb.MpError, match=r"\(-4\)"):
                eng.capacity(p)
            eng.set_landscape_dense(distances(spec, n), spec["area"])
            assert eng.capacity(p)["lam"][0] > 0.0


def test_growth_factor_predicts_persistence():
    """Thresholds fixed in advance: from a fully occupied cfg2 landscape, R = 0.6 goes extinct (< 1 % of the patches occupied after
    50 years) and R = 1.6 persists (> 20 %)."""
    n = 1000
    rng = np.random.default_rng(12345)                        # the positions and areas of synth.make_workload("cfg2")
    side = np.sqrt(n) * 250.0
    px, py = rng.uniform(0, side, n), rng.uniform(0, side, n)
    area = np.random.default_rng(12346).lognormal(0.0, 0.5, n)
    e, alpha, b = 0.5, 1 / 400, 0.5
    with mb.Engine(n, 2, 2, precision=mb.FP32) as eng:
        eng.set_landscape_coords(px, py, area)
        eng.set_source_units(None)
        lam = eng.capacity([pdict(alpha=alpha, b=b)], rtol=1e-8)["lam"][0]
        assert abs(lam - 17.0868) < 1e-3 * 17.0868
        cs = [(R / (1 - e) - 1) / lam for R in (0.6, 1.6)]
        eng.set_params([pdict(e=e, c=c, alpha=alpha, b=b) for c in cs])
        z = np.ones((2, 2, n), dtype=np.uint8)
        eng.set_state(z, np.ones((2, 1, n), dtype=np.uint8))
        occ, _ = eng.forecast(50, 32, seed=3, want_incidence=False)
        res = mb.persistence(np.array([[e, c, alpha, b, 1, 0, 0, 0, 1, 0, 0] for c in cs]), np.array([lam, lam]))
    assert np.allclose(res["R"], [0.6, 1.6])
    final = occ[:, :, -1].mean(axis=1)
    assert final[0] < 0.01 * n, final
    assert final[1] > 0.20 * n, final
