"""The culled y scan's branch sum (how every 512-thread task runs): one trip also decides candidate i+1 given that candidate i
was accepted, from the weights the trip already evaluated.  The reference without the branch is the culled scan at 1,024
threads per task (MP_FAST_TPT=1024), which takes the same two-candidate trips and evaluates the same 32-target groups.  The
decisions must be the reference's up to FP32 ties, S must stay consistent, and the cancellation guard must defer i+1 where the
shortcut would lose accuracy."""
import numpy as np
import pytest

import midaspom_b200 as mb
import oracle_lib as O
from gpu_util import make_engine, pdict, random_landscape
from test_gpu_blocks import auto_grid, wide_landscape, ALPHA

pytestmark = pytest.mark.gpu

FIXED = dict(sample_e=0, sample_c=0, update_z=0, n_adapt=0)


def one_sweep(monkeypatch, spec, z, y, par, C, prec=mb.FP32, branch=True, seed=13, grid=None):
    """One fixed-parameter sweep from (z, y): new y, incremental S, recomputed S, scan geometry, work counters.
    branch=False: the reference scan without the branch, 1,024 threads per task."""
    if branch:
        monkeypatch.delenv("MP_FAST_TPT", raising=False)
    else:
        monkeypatch.setenv("MP_FAST_TPT", "1024")
    with make_engine(spec, n_chains=C, precision=prec, seed=seed, max_draws=1) as eng:
        if grid is not None:
            eng.set_scan_blocks(*grid)
        eng.set_params([par] * C)
        eng.set_state(np.stack([z] * C), np.stack([y] * C))
        eng.set_sampler(mb.engine.sampler_config(**FIXED))
        eng.connectivity(fetch=False)
        eng.work_counters(reset=True)
        eng.sweep(1)
        work, geo = eng.work_counters(), eng.scan_geometry()
        yy, S_inc = eng.get_state()[1], eng.get_connectivity()
        return dict(y=yy, S=S_inc, S_new=eng.connectivity(), geo=geo, work=work)


def trips_per_candidate(r, cand):
    return r["work"]["scan_trips"] / (r["geo"]["threads_per_task"] // 32) / cand     # scan_trips counts warp-trips


def max_rel(a, b, floor=1e-9):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))


def test_branch_agrees_with_the_1024_thread_scan_at_the_cfg3_shape(monkeypatch):
    """N = 10,000, 20 years, 64 chains (clusters of 4 x 128 threads): the 512-thread scan with the branch and the 1,024-thread
    scan without it decide the same cells in the same sweep up to FP32 ties; with the branch a trip retires two candidates
    (about 0.5 trips per candidate), without it one after an accepted flip (1 / (2 - p) trips per candidate at acceptance
    rate p)."""
    monkeypatch.delenv("MP_FAST_TPT", raising=False); monkeypatch.delenv("MP_FAST_CS", raising=False)
    rng = np.random.default_rng(515)
    n, T, C = 10000, 20, 64
    spec, z, y = random_landscape(rng, n, T, O.GEOM_COORDS, occ=0.5, miss=0.03)
    par = pdict(e=0.35, c=0.004, alpha=1 / 400, b=0.5)
    on = one_sweep(monkeypatch, spec, z, y, par, C, branch=True)
    off = one_sweep(monkeypatch, spec, z, y, par, C, branch=False)
    assert on["geo"]["threads_per_task"] == 512 and on["geo"]["cluster"] == 4 and on["geo"]["culled"], on["geo"]
    assert off["geo"]["threads_per_task"] == 1024 and off["geo"]["culled"], off["geo"]
    for r in (on, off):
        assert max_rel(r["S"], r["S_new"]) <= 1e-6
    cand = int(((z[:-1] & z[1:]) == 1).sum()) * C
    differ = int((on["y"] != off["y"]).sum())
    print(f"y cells differing with / without the branch: {differ} of {cand} candidates")
    assert differ <= max(10, 1e-5 * cand), differ
    p = float((off["y"] != np.stack([y] * C)).sum()) / cand                   # accepted flips per candidate
    t_on, t_off = trips_per_candidate(on, cand), trips_per_candidate(off, cand)
    print(f"trips per candidate: {t_on:.4f} with the branch, {t_off:.4f} without (1 / (2 - p) = {1 / (2 - p):.4f}, p = {p:.3f})")
    assert 0.5 <= t_on <= 0.51, t_on
    assert abs(t_off - 1 / (2 - p)) <= 0.02, (t_off, p)
    # every trip but the deferred ones retires both candidates it evaluated
    w = on["work"]
    assert w["scan_retired"] <= w["scan_exec"] <= 1.01 * w["scan_retired"], w


def test_guard_defers_on_isolated_targets(monkeypatch):
    """Pairs of patches 50 m apart, 4 km from any other pair (1/alpha = 400 m): the removal of one member takes nearly all of
    the other's S, the case where fl(S_hi - w) + S_lo is not accurate enough for the branch.  The guard must fire (trips whose
    second candidate is deferred: executed > retired evaluations), the decisions still agree with the FP64 path, and y and S
    are those of the scan without the branch (1,024 threads per task: the same groups, so the same commits).  (The
    incremental S of the most isolated targets, ~1e-14 here, differs from a recomputation by more than the 1e-6 the other
    landscapes meet, identically with and without the branch.)"""
    rng = np.random.default_rng(77)
    npair, T, C = 2200, 4, 2
    n = 2 * npair
    spec, z, y = random_landscape(rng, n, T, O.GEOM_COORDS, occ=0.5, miss=0.03)
    side = int(np.ceil(np.sqrt(npair)))
    cx, cy = (np.arange(npair) % side) * 4000.0, (np.arange(npair) // side) * 4000.0
    ang = rng.uniform(0, 2 * np.pi, npair)
    spec["px"] = np.concatenate([cx, cx + 50 * np.cos(ang)])
    spec["py"] = np.concatenate([cy, cy + 50 * np.sin(ang)])
    m = O.Model(spec["obs"], geom=O.GEOM_COORDS, px=spec["px"], py=spec["py"], area=spec.get("area"))
    S0 = O.connectivity(m, 1 / 400, 0.5, y[0])
    par = pdict(e=0.35, c=float(0.3 / np.median(S0[S0 > 0])), alpha=1 / 400, b=0.5)
    r64 = one_sweep(monkeypatch, spec, z, y, par, C, prec=mb.FP64)
    r32 = one_sweep(monkeypatch, spec, z, y, par, C)
    off = one_sweep(monkeypatch, spec, z, y, par, C, branch=False)
    assert r32["geo"]["threads_per_task"] == 512 and r32["geo"]["culled"], r32["geo"]
    assert off["geo"]["threads_per_task"] == 1024 and off["geo"]["culled"], off["geo"]
    cand = int(((z[:-1] & z[1:]) == 1).sum()) * C
    w = r32["work"]
    print(f"evaluations executed {w['scan_exec']}, retired {w['scan_retired']}")
    assert w["scan_exec"] > w["scan_retired"], w                              # deferrals happened
    assert (r64["y"] != r32["y"]).sum() <= max(2, 2e-3 * cand), (r64["y"] != r32["y"]).sum()
    differ = int((off["y"] != r32["y"]).sum())
    assert differ <= 2, differ
    if differ == 0:                                                           # same decisions: the same commits, bit for bit
        assert np.array_equal(r32["S"], off["S"])


def test_branch_on_a_linear_landscape(monkeypatch):
    """The linear geometry's culled scan with the branch against the FP64 path."""
    rng = np.random.default_rng(88)
    n, T, C = 6000, 5, 3
    spec, z, y = random_landscape(rng, n, T, O.GEOM_LINEAR, occ=0.5, miss=0.03)
    par = pdict(e=0.35, c=0.1, alpha=1 / 400, b=0.5)
    r64 = one_sweep(monkeypatch, spec, z, y, par, C, prec=mb.FP64)
    r32 = one_sweep(monkeypatch, spec, z, y, par, C)
    assert r32["geo"]["threads_per_task"] == 512 and r32["geo"]["culled"], r32["geo"]
    cand = int(((z[:-1] & z[1:]) == 1).sum()) * C
    assert trips_per_candidate(r32, cand) <= 0.52
    assert (r32["y"] != np.stack([y] * C)).sum() > 0.05 * cand                 # the scan moved
    assert (r64["y"] != r32["y"]).sum() <= max(2, 2e-3 * cand), (r64["y"] != r32["y"]).sum()
    assert max_rel(r32["S"], r32["S_new"]) <= 1e-6


def test_branch_in_block_launches(monkeypatch):
    """Block tasks of 512 threads (MP_BLK_TPT=512) with the branch: the same decisions as the FP64 path in the block order."""
    monkeypatch.setenv("MP_BLK_TPT", "512")
    rng = np.random.default_rng(1234)
    nside, T, C = 145, 3, 2
    spec, z, y = wide_landscape(rng, nside, T)
    par = pdict(e=0.35, c=0.05, alpha=ALPHA, b=0.5)
    grid = auto_grid(spec, z, y, par, 3)
    r64 = one_sweep(monkeypatch, spec, z, y, par, C, prec=mb.FP64, grid=grid)
    r32 = one_sweep(monkeypatch, spec, z, y, par, C, grid=grid)
    assert r32["geo"]["blocks"] and r32["geo"]["threads_per_task"] == 512, r32["geo"]
    assert r32["work"]["scan_blocks"] > 0
    cand = int(((z[:-1] & z[1:]) == 1).sum()) * C
    assert (r64["y"] != r32["y"]).sum() <= max(2, 2e-3 * cand), (r64["y"] != r32["y"]).sum()
    assert max_rel(r32["S"], r32["S_new"]) <= 1e-6
