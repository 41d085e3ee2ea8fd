"""Host-side logic that needs no GPU: the posterior diagnostics used by bench.py and the drivers, the
reference's row split, the synthetic workload generator."""
import numpy as np

from midaspom_b200 import distributed as D
from midaspom_b200 import synth


def ar1(rng, n, rho):
    x = np.empty(n)
    x[0] = rng.normal()
    e = rng.normal(size=n) * np.sqrt(1 - rho * rho)
    for i in range(1, n):
        x[i] = rho * x[i - 1] + e[i]
    return x


def test_ess_of_an_ar1_chain_matches_theory():
    """ESS of an AR(1) chain is n (1 - rho) / (1 + rho)."""
    rng = np.random.default_rng(3)
    n = 40000
    for rho in (0.0, 0.5, 0.9):
        got = D.ess_geyer(ar1(rng, n, rho))
        want = n * (1 - rho) / (1 + rho)
        assert abs(got - want) < 0.15 * want, (rho, got, want)
    assert D.ess_geyer(np.ones(100)) == 100.0                     # constant chain: defined as n, never NaN
    assert D.ess_geyer(np.arange(5.0)) == 5.0                     # too short to estimate


def test_split_rhat_separates_converged_from_stuck_chains():
    rng = np.random.default_rng(4)
    good = rng.normal(size=(2000, 4))
    assert D.split_rhat(good) < 1.01
    bad = good.copy(); bad[:, 0] += 3.0                           # one chain somewhere else
    assert D.split_rhat(bad) > 1.5
    drift = good + np.linspace(0, 3, 2000)[:, None]               # all chains drifting: caught by the split
    assert D.split_rhat(drift) > 1.2
    assert np.isnan(D.split_rhat(good[:3]))


def test_posterior_summary_fields_and_constant_parameters():
    rng = np.random.default_rng(5)
    d = rng.normal(size=(500, 3, 5)) * np.array([0.1, 0.2, 0.0, 0.3, 0.0]) + np.array([0.3, 0.05, 0.0025, 0.5, 1.0])
    s = D.posterior_summary(d)
    assert set(s) == {"e", "c", "b"}                              # alpha and p never moved: not reported
    assert abs(s["e"]["mean"] - 0.3) < 0.02 and abs(s["b"]["sd"] - 0.3) < 0.03
    assert s["c"]["ess"] > 1000 and s["c"]["rhat"] < 1.02


def test_reference_row_split_and_chain_blocks():
    """main_MIDASPOM_MPI.c:361-372: rank 0 takes the remainder."""
    for total, world in ((101, 4), (101, 1), (7, 8), (64, 8)):
        spans = [D.split_rows(total, world, r) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == total
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        assert spans[0][1] - spans[0][0] == total // world + total % world
    assert [D.chain_block(r, 8, 8) for r in (0, 3, 7)] == [(0, 8), (24, 8), (56, 8)]


def test_synthetic_workloads_are_deterministic_and_feasible():
    a, b = synth.make_workload("tiny"), synth.make_workload("tiny")
    assert (a["obs"] == b["obs"]).all() and (a["px"] == b["px"]).all() and a["truth"] == b["truth"]
    z, obs = a["z_true"], a["obs"]
    assert obs.shape == (a["T"], a["n"]) and set(np.unique(obs)) <= {-1, 0, 1}
    assert (obs[0] != -1).all()                                   # year 0 is never hidden (SURVEY 8c: UB in the reference)
    assert ((obs == z) | (obs == -1)).all()                       # perfect detection: what is seen is the truth
    w = synth.make_workload("cfg2")                               # imperfect detection: misses only, never false presences
    assert w["detect"] == 1 and ((w["obs"] <= w["z_true"]) | (w["obs"] == -1)).all() and (w["obs"][w["z_true"] == 1] == 0).any()
    W = synth.kernel_matrix(a["px"], a["py"], a["area"], 1 / 400, 0.5, dtype=np.float64)
    assert (np.diag(W) == 0).all()
    i, j = 3, 17
    assert np.isclose(W[i, j], np.exp(-np.hypot(a["px"][i] - a["px"][j], a["py"][i] - a["py"][j]) / 400) * a["area"][i] ** 0.5)


def test_bench_roofline_from_work_counters():
    """bench.py's roofline block on the numbers of a real cfg3 line (profiles/r02_bench_cfg3.json): fractions of the MUFU peak
    (scan) and of the FP64 peak (k_conn) come from executed work and stay below 1; the culled and the unculled scan both work."""
    import importlib.util
    import json
    from pathlib import Path
    root = Path(__file__).resolve().parents[1]
    spec = importlib.util.spec_from_file_location("bench_mod", root / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    wl = dict(n=10000, T=20)
    kms = dict(conn=149.574, col=6.58, sweep_y=1197.05, sweep_z=6.65, small=18.79, sim=0.0)
    klaunch = dict(conn=20, col=60, sweep_y=20, sweep_z=20, small=280, sim=0)
    # engine counters of 20 sweeps of 64 chains (groups of 32 targets; tiles of 32 x 32 pairs)
    work = dict(scan_trips=78_600_000, scan_exec=12_600_000_000, scan_retired=11_000_000_000, scan_commit=4_300_000_000, scan_dense=0,
                conn_exec=55_000_000, conn_total=137_900_000, gemm_tiles=0, scan_blocks=0)
    geo = dict(threads_per_task=512, cluster=1, candidates_per_trip=2, culled=True, blocks=False)
    probe = dict(mufu_gops=4613.8, ffma_gfma=31600.0, dadd_gops=18000.0, copy_gbs=6400.0)
    roof = bench.roofline("cfg3", wl, 64, 102752.0, kms, klaunch, work, geo, probe, 6650.0, True, sum(kms.values()))
    assert roof["kernel"] == "k_sweep_y_cull" and 0.05 < roof["frac"] < 1.0 and roof["executed"]["frac"] >= roof["frac"]
    conn = roof["conn"]
    assert 0.0 < conn["frac"] < 1.0
    assert conn["fp64"]["dfma_per_pair"] == 20 and 0.1 < conn["fp64"]["frac"] < 1.0
    assert abs(conn["fp64"]["frac"] - conn["pairs_executed_per_launch"] * 20 / (conn["ms_per_launch"] * 1e-3) * 1e-9 / 18000.0) < 1e-12
    json.dumps(roof)                                              # the block goes into the bench's JSON line
    # unculled scan (cfg2: k_sweep_y_fast), more than 32 years: 32 accumulators per pass
    geo2 = dict(threads_per_task=256, cluster=1, candidates_per_trip=1, culled=False, blocks=False)
    work2 = dict(work, scan_dense=3_000_000_000, scan_exec=0, scan_retired=0, scan_commit=0, scan_trips=0)
    roof2 = bench.roofline("cfg2", dict(n=1000, T=41), 8, 3000.0, kms, klaunch, work2, geo2, probe, 6650.0, False, sum(kms.values()))
    assert roof2["kernel"] == "k_sweep_y_fast" and roof2["conn"]["fp64"]["dfma_per_pair"] == 32
    # no probe figure for the FP64 peak: the block is simply absent
    roof3 = bench.roofline("cfg3", wl, 64, 102752.0, kms, klaunch, work, geo, dict(probe, dadd_gops=0.0), 6650.0, True, sum(kms.values()))
    assert "fp64" not in roof3["conn"]


def test_bench_dump_outputs_types_and_sample(tmp_path):
    """bench.py --dump-outputs: float64 stays float64, 0/1 states become float32, an array above the size limit becomes the same
    seeded sample of its elements in every run."""
    import importlib.util
    from pathlib import Path
    spec = importlib.util.spec_from_file_location("bench_mod", Path(__file__).resolve().parents[1] / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rng = np.random.default_rng(4)
    big = rng.random(bench.DUMP_SAMPLE + 1000)
    z = (rng.random((3, 5, 7)) < 0.5).astype(np.uint8)
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, dict(S=big, z=z))
    S, zd = np.load(tmp_path / "a" / "S.npy"), np.load(tmp_path / "a" / "z.npy")
    assert S.dtype == np.float64 and S.shape == (bench.DUMP_SAMPLE,) and np.isin(S, big).all()
    assert (S == np.load(tmp_path / "b" / "S.npy")).all()
    assert zd.dtype == np.float32 and (zd == z).all()
