#!/usr/bin/env python
"""The culled y scan (k_sweep_y_cull) in each launch geometry on the same chains: cfg3 (N = 10,000, T = 20, 64 chains unless --chains), every
engine started from one sampler state (parameters, latent states, proposal scales, seed).  After warm-up the geometries
alternate over the repeats; each repeat reports the scan's ms per launch (the engine's per-kernel CUDA events) and the step
ms (host wall time around K synchronous sweeps, per-kernel timing off).  One sweep from an identical state with fixed
parameters gives the y cells that differ from the first geometry and the largest relative |S_inc - S_recomputed|.
    python scripts/scan_micro.py [--steps 10] [--warmup 5] [--repeats 3] [--geometries 512x1,512x2,512x4] [--chains 64] [--out FILE]
A geometry is TPTxCS, set through MP_FAST_TPT / MP_FAST_CS before its engine is created."""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import midaspom_b200 as mb  # noqa: E402
from midaspom_b200 import synth  # noqa: E402

def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [v.strip() for v in out.split(",")]
        return dict(name=name, power_limit=power, sm_clock_max=clock)
    except Exception as ex:  # the numbers below still stand; say why the card is not named
        return dict(error=f"{type(ex).__name__}: {ex}")


def bench_module():
    """bench.py's start parameters and sampler settings, so that the chains are the benchmark's."""
    spec = importlib.util.spec_from_file_location("bench_mod", ROOT / "bench.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def make_engine(wl, geom, chains, max_draws):
    tpt, cs = geom
    os.environ["MP_FAST_TPT"], os.environ["MP_FAST_CS"] = str(tpt), str(cs)
    try:
        eng = mb.Engine(wl["n"], wl["T"], chains, precision=mb.FP32, seed=1000, detect=wl["detect"], max_draws=max_draws)
    finally:
        del os.environ["MP_FAST_TPT"], os.environ["MP_FAST_CS"]
    eng.set_landscape_coords(wl["px"], wl["py"], wl["area"])
    eng.set_source_units(wl.get("src_unit"))
    eng.set_observations(wl["obs"])
    eng.set_era(wl.get("era"))
    return eng


def start(eng, st, sc):
    eng.set_params(st["par"])
    eng.set_state(st["z"], st["y"])
    eng.set_scales(st["lsig"])
    eng.set_sampler(sc)
    eng.reset_draws()


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--geometries", default="512x1,512x2,512x4")
    ap.add_argument("--chains", type=int, default=64)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "scan_micro.json"))
    args = ap.parse_args()
    if mb.engine.load_library().mp_device_count() < 1:
        raise SystemExit("scan_micro.py: no CUDA device; there is nothing to measure without a B200")
    geoms = [tuple(int(v) for v in g.split("x")) for g in args.geometries.split(",")]
    bench = bench_module()
    wl = synth.make_workload("cfg3")
    sc = mb.engine.sampler_config(**bench.sampler_kwargs(wl))
    K, C = args.steps, args.chains
    max_draws = 4 + args.warmup + 2 * K * args.repeats

    # one sampler state for every engine: the bench's start, 20 sweeps into the adaptation
    with make_engine(wl, geoms[0], C, 32) as eng:
        eng.set_params([bench.start_params(wl)] * C)
        eng.init_chains(sc, disperse=False)
        eng.sweep(20)
        z, y = eng.get_state()
        st = dict(par=eng.get_params(), z=z, y=y, lsig=eng.get_scales())

    engines = {g: make_engine(wl, g, C, max_draws) for g in geoms}
    # ---- one sweep from the identical state, parameters fixed: what each geometry decides
    fixed = mb.engine.sampler_config(sample_e=0, sample_c=0, update_z=0, n_adapt=0)
    agree = {}
    for g, eng in engines.items():
        start(eng, st, fixed)
        eng.connectivity(fetch=False)
        eng.work_counters(reset=True)
        eng.sweep(1)
        work = eng.work_counters()
        yy = eng.get_state()[1]
        S_inc = eng.get_connectivity()
        S_new = eng.connectivity()
        scan = eng.scan_geometry()
        agree[g] = (yy, float(np.max(np.abs(S_inc - S_new) / np.maximum(np.abs(S_new), 1e-9))), scan, work)
    y_ref = agree[geoms[0]][0]
    cand = int(((st["z"][:, :-1] & st["z"][:, 1:]) == 1).sum())

    # ---- timing: the bench's sampler from the common state, geometries alternating
    for eng in engines.values():
        start(eng, st, sc)
        eng.sweep(args.warmup)
    runs = {g: dict(sweep_y_ms=[], step_ms=[]) for g in geoms}
    for _ in range(args.repeats):
        for g, eng in engines.items():
            eng.set_timing(False)
            t0 = time.perf_counter()
            eng.sweep(K)
            runs[g]["step_ms"].append((time.perf_counter() - t0) * 1e3 / K)
            eng.set_timing(True)
            eng.get_timing(reset=True)
            eng.sweep(K)
            kms, klaunch = eng.get_timing(reset=True)
            eng.set_timing(False)
            runs[g]["sweep_y_ms"].append(kms["sweep_y"] / max(1, klaunch["sweep_y"]))
    results = []
    for g, eng in engines.items():
        yy, srel, scan, work = agree[g]
        r = runs[g]
        results.append(dict(geometry=dict(threads_per_task=g[0], cluster=g[1]), scan=scan,
                            sweep_y_ms_per_launch=dict(median=float(np.median(r["sweep_y_ms"])), runs=[round(v, 3) for v in r["sweep_y_ms"]]),
                            step_ms=dict(median=float(np.median(r["step_ms"])), runs=[round(v, 3) for v in r["step_ms"]]),
                            one_sweep=dict(y_cells_differing=int((yy != y_ref).sum()), candidates=cand, max_rel_S_inc_vs_recomputed=srel,
                                           trips_per_candidate=work["scan_trips"] / (g[0] // 32) / cand,
                                           evaluations_executed=work["scan_exec"], evaluations_retired=work["scan_retired"])))
        print(json.dumps(results[-1]), flush=True)
        eng.close()
    out = dict(gpu=gpu_info(), workload="cfg3", desc=wl["desc"], n_patches=wl["n"], years=wl["T"], chains=C, steps=K,
               warmup=args.warmup, repeats=args.repeats,
               method="engines built per geometry (MP_FAST_TPT / MP_FAST_CS), all from one sampler state; after warm-up the geometries "
                      "alternate; sweep_y = per-kernel CUDA events (ms per launch), step = host wall time around K synchronous sweeps "
                      "with the per-kernel timing off; one_sweep compares y with the first geometry after one fixed-parameter sweep",
               results=results)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
