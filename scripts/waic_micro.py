#!/usr/bin/env python
"""Step time with the WAIC sums (mp_set_waic) off and on, thin = 1: two engines per workload with bench.py's chains, start
parameters and sampler settings, the same seed and start state (so both run the same chain), one without and one with the
sums.  Device time of every step from CUDA events on the engine stream, L2 flushed between steps, captured sweeps (warm-up
long enough for both kinds of captured sweep); the two engines alternate over the repeats.  A separate pass with per-kernel
timing gives k_waic's own time (the added MP_K_SMALL ms per sweep).
Workloads: cfg3 (64 chains), cfg5 (one chain, block grid of the y scan), cfg2 (8 chains, imperfect detection).
    python scripts/waic_micro.py [--steps 10] [--warmup 40] [--repeats 3] [--workloads cfg3,cfg5,cfg2] [--out FILE]"""
import argparse
import importlib.util
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import midaspom_b200 as mb  # noqa: E402
from midaspom_b200 import synth  # noqa: E402

CHAINS = dict(cfg3=64, cfg5=1, cfg2=8)


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


def make_engine(bench, wl, chains, waic, grid):
    eng = mb.Engine(wl["n"], wl["T"], chains, precision=mb.FP32, seed=1000, detect=wl["detect"], max_draws=4)
    eng.set_landscape_coords(wl["px"], wl["py"], wl["area"])
    eng.set_source_units(wl.get("src_unit"))
    eng.set_observations(wl["obs"])
    eng.set_era(wl.get("era"))
    eng.set_params([bench.start_params(wl)] * chains)
    eng.init_chains(mb.engine.sampler_config(**bench.sampler_kwargs(wl)), disperse=False)
    if grid == "auto":
        p0 = bench.start_params(wl)
        grid = eng.set_scan_blocks_auto(wl["px"], wl["py"], p0["alpha"], float(eng.get_connectivity().min()),
                                        float(np.max(np.asarray(wl["area"]) ** p0["b"])), k=4)
    elif grid:
        eng.set_scan_blocks(*grid)
    if waic:
        eng.set_waic(0, 1)
    return eng, grid


def timed_steps(torch, eng, stream, nsteps, flush):
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nsteps)]
    with torch.cuda.stream(stream):
        for a, b in evs:
            flush.fill_(1)
            a.record(stream)
            eng.sweep(1, sync=False)
            b.record(stream)
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in evs]


def run(torch, bench, name, steps, warmup, repeats):
    chains = CHAINS[name]
    wl = synth.make_workload_large(name) if name == "cfg5" else synth.make_workload(name)
    off, grid = make_engine(bench, wl, chains, False, "auto" if name == "cfg5" else None)
    on, _ = make_engine(bench, wl, chains, True, grid)
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    arms = dict(off=(off, torch.cuda.ExternalStream(off.stream(), device=dev)), on=(on, torch.cuda.ExternalStream(on.stream(), device=dev)))
    for eng, _ in arms.values():
        eng.sweep(warmup)
    times = dict(off=[], on=[])
    for _ in range(repeats):
        for key in ("off", "on"):
            eng, st = arms[key]
            times[key].append(float(np.median(timed_steps(torch, eng, st, steps, flush))))
    swept = warmup + repeats * steps
    same = all(np.array_equal(a, b) for a, b in zip(off.get_state(), on.get_state())) and np.array_equal(off.get_draws(), on.get_draws())
    s = on.waic_sums()
    assert s["nsamples"] == swept * chains, (s["nsamples"], swept, chains)
    # the kernel's own time: per-kernel CUDA events (captured sweeps off), MP_K_SMALL ms per sweep with and without it
    small = {}
    for key in ("off", "on"):
        eng = arms[key][0]
        eng.set_timing(True)
        eng.sweep(2)
        eng.get_timing(reset=True)
        eng.sweep(steps)
        ms, launches = eng.get_timing(reset=True)
        small[key] = dict(ms_per_sweep=ms["small"] / steps, launches_per_sweep=launches["small"] / steps)
        eng.set_timing(False)
    T, n = wl["T"], wl["n"]
    nobs = int((np.asarray(wl["obs"]) >= 0).sum())
    # z of the previous year and S per chain, obs, and the three sums of every observed cell read and written
    read_bytes = chains * ((T - 1) * n + (T - 1) * n * 8) + T * n + 2 * nobs * 24
    med_off, med_on = float(np.median(times["off"])), float(np.median(times["on"]))
    res = dict(workload=name, desc=wl["desc"], n_patches=n, years=T, chains=chains, precision="fp32", scan_blocks=grid,
               step_ms=dict(off=times["off"], on=times["on"], median_off=med_off, median_on=med_on),
               overhead_pct=100.0 * (med_on - med_off) / med_off,
               waic_kernel_ms=small["on"]["ms_per_sweep"] - small["off"]["ms_per_sweep"], small_category=small,
               bytes_per_accumulation=read_bytes, same_chain_on_and_off=bool(same), nsamples=int(s["nsamples"]))
    off.close(); on.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=40)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--workloads", default="cfg3,cfg5,cfg2")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "waic_micro.json"))
    args = ap.parse_args()
    if mb.engine.load_library().mp_device_count() < 1:
        raise SystemExit("waic_micro.py: no CUDA device; there is nothing to measure without a B200")
    import torch
    bench = bench_module()
    out = dict(gpu=gpu_info(), method="device time per step (CUDA events on the engine stream around each mp_sweep(1), 256 MB "
               "L2 flush between steps, captured sweeps), median over the steps of a repeat; the engines without and with "
               "the WAIC sums alternate over the repeats.  waic_kernel_ms: added MP_K_SMALL ms per sweep under per-kernel "
               "timing.  bytes_per_accumulation: z of the previous year and S read per chain, obs, and the sums of the "
               "observed cells read and written", results=[])
    for name in args.workloads.split(","):
        res = run(torch, bench, name, args.steps, args.warmup, args.repeats)
        print(json.dumps(res), flush=True)
        out["results"].append(res)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
