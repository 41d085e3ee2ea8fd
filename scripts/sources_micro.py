#!/usr/bin/env python
"""Extra step time of the colonisation sources (mp_set_sources): four engines per workload with bench.py's chains, start
parameters and sampler settings, the same seed and start state (so all run the same chain): sources off; on with thin = 1 and
no histogram; on with thin = 1 and 64 bins of 100 m; on but never due (first_sweep beyond the run: only the gated launches
run).  Device time of every step from CUDA events on the engine stream, L2 flushed between steps, captured sweeps; the engines
alternate over the repeats.  Also records the events and sources per (chain, transition) of the final state, so the pairs the
contraction evaluates per sample are known.
Workloads: cfg3 (64 chains), cfg4 (8 chains, die-off era flags), cfg5 (one chain, block grid of the y scan).
    python scripts/sources_micro.py [--steps 10] [--warmup 40] [--repeats 3] [--workloads cfg3,cfg4,cfg5] [--out FILE]"""
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

CHAINS = dict(cfg3=64, cfg4=8, cfg5=1)
ARMS = dict(off=None, on_nohist=(0, 1, 0, 0.0), on_hist64=(0, 1, 64, 100.0), gated=(1 << 30, 1, 64, 100.0))


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


def make_engine(bench, wl, chains, arm, grid):
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
    if ARMS[arm] is not None:
        eng.set_sources(*ARMS[arm])
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
    engs, grid = {}, "auto" if name == "cfg5" else None
    for arm in ARMS:
        engs[arm], grid = make_engine(bench, wl, chains, arm, grid)
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    streams = {arm: torch.cuda.ExternalStream(e.stream(), device=dev) for arm, e in engs.items()}
    for e in engs.values():
        e.sweep(warmup)
    times = {arm: [] for arm in ARMS}
    for _ in range(repeats):
        for arm, e in engs.items():
            times[arm].append(float(np.median(timed_steps(torch, e, streams[arm], steps, flush))))
    swept = warmup + repeats * steps
    ref = engs["off"]
    same = all(all(np.array_equal(a, b) for a, b in zip(ref.get_state(), e.get_state())) and np.array_equal(ref.get_draws(), e.get_draws())
               for e in engs.values())
    src = {arm: engs[arm].sources() for arm in ARMS if arm != "off"}
    assert src["on_hist64"]["nsamples"] == swept * chains and src["gated"]["nsamples"] == 0
    got = src["on_hist64"]
    lhs = got["src_sum"].sum(axis=1) + got["ext_sum"]
    rhs = (got["events"] - got["unattributed"]).astype(np.float64)
    z, y = ref.get_state()
    ev = ((y == 0) & (z[:, 1:] == 1)).sum(axis=2)           # [chain, transition] of the final state
    nsrc = (y == 1).sum(axis=2)
    pairs = int((ev.astype(np.int64) * nsrc).sum())
    med = {arm: float(np.median(v)) for arm, v in times.items()}
    res = dict(workload=name, desc=wl["desc"], n_patches=wl["n"], years=wl["T"], chains=chains, precision="fp32", scan_blocks=grid,
               step_ms=dict(times, **{f"median_{a}": m for a, m in med.items()}),
               extra_ms=dict(qualifying_nohist=med["on_nohist"] - med["off"], qualifying_hist64=med["on_hist64"] - med["off"],
                             not_due=med["gated"] - med["off"]),
               events_per_chain_transition=dict(mean=float(ev.mean()), max=int(ev.max())),
               sources_per_chain_transition=dict(mean=float(nsrc.mean()), max=int(nsrc.max())),
               pairs_per_sample_sweep=pairs, pair_rate_per_s=pairs / max(1e-9, (med["on_nohist"] - med["off"]) * 1e-3),
               conservation_max_rel=float(np.max(np.abs(lhs - rhs) / np.maximum(rhs, 1.0))),
               same_chain_in_every_arm=bool(same), nsamples=int(got["nsamples"]))
    for e in engs.values():
        e.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=40)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--workloads", default="cfg3,cfg4,cfg5")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "sources_micro.json"))
    args = ap.parse_args()
    if mb.engine.load_library().mp_device_count() < 1:
        raise SystemExit("sources_micro.py: no CUDA device; there is nothing to measure without a B200")
    import torch
    bench = bench_module()
    out = dict(gpu=gpu_info(), method="device time per step (CUDA events on the engine stream around each mp_sweep(1), 256 MB "
               "L2 flush between steps, captured sweeps), median over the steps of a repeat; the four engines (off, on without "
               "histogram, on with 64 bins, on but never due) alternate over the repeats.  extra_ms: median step time of an arm "
               "minus that of the engine without sources.  pairs_per_sample_sweep: sum over (chain, transition) of events x "
               "sources of the final state; pair_rate_per_s: that over the extra time without histogram", results=[])
    for name in args.workloads.split(","):
        res = run(torch, bench, name, args.steps, args.warmup, args.repeats)
        print(json.dumps(res), flush=True)
        out["results"].append(res)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
