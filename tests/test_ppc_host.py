"""CPU checks of midaspom_b200.ppc_check, the reduction of mp_ppc's replicate statistics: the per-year, omnibus and per-patch
p-values against a direct loop-by-loop computation, pooling of several calls and chain shards, the years whose statistic does
not vary over the replicates, and the refusal to pool results computed on different observations."""
import numpy as np
import pytest

import midaspom_b200 as mb


def fake_result(rng, C, nrep, T, N, obs_stats, lam=20.0):
    stats = rng.poisson(lam, size=(C, nrep, T, 3)).astype(np.int32)
    stats[:, :, 0, 1:] = 0                                # no transition into year 0
    stats[:, :, 2, 2] = 7                                 # one (year, statistic) that never varies
    ge = rng.integers(0, C * nrep + 1, N).astype(np.uint32)
    gt = np.minimum(ge, rng.integers(0, C * nrep + 1, N)).astype(np.uint32)
    return dict(stats=stats, obs_stats=np.asarray(obs_stats, dtype=np.int32), patch_ge=ge, patch_gt=gt, nrep_total=C * nrep)


def direct(results):
    """Loop-by-loop restatement of the definitions in midaspom_b200/ppc.py."""
    obs = results[0]["obs_stats"].astype(float)
    T = obs.shape[0]
    reps = [r["stats"][c, i].astype(float) for r in results for c in range(r["stats"].shape[0]) for i in range(r["stats"].shape[1])]
    M = len(reps)
    p_year = np.zeros((T, 3))
    for t in range(T):
        for s in range(3):
            ge = sum(x[t, s] >= obs[t, s] for x in reps) / M
            le = sum(x[t, s] <= obs[t, s] for x in reps) / M
            p_year[t, s] = min(1.0, 2.0 * min(ge, le))
    p_omni = np.zeros(3)
    for s in range(3):
        m = [sum(x[t, s] for x in reps) / M for t in range(T)]
        v = [sum((x[t, s] - m[t]) ** 2 for x in reps) / M for t in range(T)]
        years = [t for t in range(1, T) if v[t] > 0]

        def D(x):
            return sum((x[t] - m[t]) ** 2 / v[t] for t in years)
        d_obs = D(obs[:, s])
        p_omni[s] = sum(D(x[:, s]) >= d_obs for x in reps) / M
    ge = sum(r["patch_ge"].astype(float) for r in results)
    gt = sum(r["patch_gt"].astype(float) for r in results)
    p_patch = np.array([min(1.0, 2.0 * min(a / M, 1.0 - b / M)) for a, b in zip(ge, gt)])
    return p_year, p_omni, p_patch, M


def test_matches_a_direct_computation_and_pools_calls():
    rng = np.random.default_rng(3)
    T, N = 6, 40
    obs = rng.poisson(20.0, size=(T, 3))
    obs[0, 1:] = 0
    obs[2, 2] = 9                                          # never reached by a replicate: p = 0 in that year
    parts = [fake_result(rng, 2, 5, T, N, obs), fake_result(rng, 3, 4, T, N, obs), fake_result(rng, 2, 5, T, N, obs)]
    got = mb.ppc_check(*parts)
    p_year, p_omni, p_patch, M = direct(parts)
    assert got["nrep_total"] == M == 32
    np.testing.assert_allclose(got["p_year"], p_year, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(got["p_omnibus"], p_omni, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(got["p_patch"], p_patch, rtol=1e-12, atol=1e-15)
    assert got["p_year"][2, 2] == 0.0
    assert (got["p_year"][0, 1:] == 1.0).all()             # 0 = 0 in every replicate
    assert got["rep_var"][2, 2] == 0.0                     # the year that does not vary is left out of D ...
    assert np.isfinite(got["D_rep"]).all() and np.isfinite(got["D_obs"]).all()
    # ... so changing the observed value there changes no omnibus p-value
    other = [dict(p, obs_stats=p["obs_stats"].copy()) for p in parts]
    for p in other:
        p["obs_stats"][2, 2] = 3
    np.testing.assert_array_equal(mb.ppc_check(*other)["p_omnibus"], got["p_omnibus"])
    # pooling is along the replicate axis only: one result holding all replicates gives the same numbers
    flat = [r["stats"].reshape(-1, T, 3) for r in parts]
    one = dict(stats=np.concatenate(flat)[None], obs_stats=parts[0]["obs_stats"], nrep_total=M,
               patch_ge=sum(r["patch_ge"].astype(np.int64) for r in parts), patch_gt=sum(r["patch_gt"].astype(np.int64) for r in parts))
    single = mb.ppc_check(one)
    for k in ("p_year", "p_omnibus", "p_patch", "D_rep", "D_obs"):
        np.testing.assert_array_equal(single[k], got[k])


def test_data_far_from_the_replicates_is_flagged():
    rng = np.random.default_rng(4)
    T, N = 8, 5
    r = fake_result(rng, 4, 25, T, N, np.zeros((T, 3)))
    m = r["stats"].mean(axis=(0, 1))
    fit = dict(r, obs_stats=np.rint(m).astype(np.int32))
    off = dict(r, obs_stats=np.rint(m + 4 * np.sqrt(m + 1)).astype(np.int32))
    assert (mb.ppc_check(fit)["p_omnibus"][:2] > 0.2).all()
    assert (mb.ppc_check(off)["p_omnibus"][:2] < 0.01).all()
    # per patch: every replicate above the data, every replicate below it, and a patch in the middle
    r2 = dict(r, patch_ge=np.array([100, 0, 50, 100, 100], dtype=np.uint32), patch_gt=np.array([100, 0, 40, 0, 60], dtype=np.uint32))
    np.testing.assert_allclose(mb.ppc_check(r2)["p_patch"], [0.0, 0.0, 1.0, 1.0, 0.8])


def test_refuses_results_on_different_observations():
    rng = np.random.default_rng(5)
    a = fake_result(rng, 2, 3, 4, 6, np.ones((4, 3)))
    b = fake_result(rng, 2, 3, 4, 6, np.ones((4, 3)))
    b["obs_stats"] = b["obs_stats"].copy()
    b["obs_stats"][3, 0] += 1
    with pytest.raises(ValueError, match="different observations"):
        mb.ppc_check(a, b)
    with pytest.raises(ValueError, match="different observations"):
        mb.ppc_check(a, dict(b, obs_stats=np.ones((5, 3), dtype=np.int32)))
    with pytest.raises(ValueError):
        mb.ppc_check()
