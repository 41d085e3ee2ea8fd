#!/usr/bin/env python
"""Cost of one posterior-predictive check (mp_ppc, nrep replicates per chain) against one sweep on the same engine: bench.py's
chains, start parameters, sampler settings and era flags, FP32, captured sweeps.  The sweep time comes from CUDA events on the
engine stream around each mp_sweep(1) (median over the steps, 256 MB L2 flush between steps); the check time is the host wall
time around one synchronous mp_ppc call (median of the repeats, after a warm-up call), the way a user calls it between sweeps.
Workloads: cfg3 (64 chains), cfg4 (8 chains, die-off era flags, K sampled), cfg5 (one chain, block grid of the y scan).
    python scripts/ppc_micro.py [--nrep 32] [--steps 10] [--warmup 40] [--repeats 3] [--workloads cfg3,cfg4,cfg5] [--out FILE]"""
import argparse
import importlib.util
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import midaspom_b200 as mb  # noqa: E402
from midaspom_b200 import synth  # noqa: E402

CHAINS = dict(cfg3=64, cfg4=8, cfg5=1)


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


def make_engine(bench, wl, chains, blocks):
    eng = mb.Engine(wl["n"], wl["T"], chains, precision=mb.FP32, seed=1000, detect=wl["detect"], max_draws=4)
    eng.set_landscape_coords(wl["px"], wl["py"], wl["area"])
    eng.set_source_units(wl.get("src_unit"))
    eng.set_observations(wl["obs"])
    eng.set_era(wl.get("era"))
    eng.set_params([bench.start_params(wl)] * chains)
    eng.init_chains(mb.engine.sampler_config(**bench.sampler_kwargs(wl)), disperse=False)
    grid = None
    if blocks:
        p0 = bench.start_params(wl)
        grid = eng.set_scan_blocks_auto(wl["px"], wl["py"], p0["alpha"], float(eng.get_connectivity().min()),
                                        float(np.max(np.asarray(wl["area"]) ** p0["b"])), k=4)
    return eng, grid


def run(torch, bench, name, nrep, steps, warmup, repeats):
    chains = CHAINS[name]
    wl = synth.make_workload_large(name) if name == "cfg5" else synth.make_workload(name)
    eng, grid = make_engine(bench, wl, chains, name == "cfg5")
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)
    eng.sweep(warmup)
    eng.ppc(nrep, seed=1)                                      # warm-up: module load, first launches
    sweep_ms, ppc_ms = [], []
    for i in range(repeats):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        with torch.cuda.stream(stream):
            for a, b in evs:
                flush.fill_(1)
                a.record(stream)
                eng.sweep(1, sync=False)
                b.record(stream)
        torch.cuda.synchronize()
        sweep_ms.append(float(np.median([a.elapsed_time(b) for a, b in evs])))
        eng.work_counters(reset=True)
        t0 = time.perf_counter()
        r = eng.ppc(nrep, seed=2 + i)
        ppc_ms.append((time.perf_counter() - t0) * 1e3)
        work = eng.work_counters(reset=True)
    p = mb.ppc_check(r)
    med_sweep, med_ppc = float(np.median(sweep_ms)), float(np.median(ppc_ms))
    res = dict(workload=name, desc=wl["desc"], n_patches=wl["n"], years=wl["T"], chains=chains, nrep=nrep, precision="fp32",
               scan_blocks=grid, sweep_ms=sweep_ms, ppc_ms=ppc_ms, median_sweep_ms=med_sweep, median_ppc_ms=med_ppc,
               ppc_in_sweeps=med_ppc / med_sweep, ppc_ms_per_transition=med_ppc / (wl["T"] - 1),
               conn_tiles_executed=work["conn_exec"] / max(1, work["conn_total"]),
               p_omnibus=dict(zip(mb.PPC_STATS, [float(v) for v in p["p_omnibus"]])))
    eng.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--nrep", type=int, default=32)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=40)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--workloads", default="cfg3,cfg4,cfg5")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "ppc_micro.json"))
    args = ap.parse_args()
    if mb.engine.load_library().mp_device_count() < 1:
        raise SystemExit("ppc_micro.py: no CUDA device; there is nothing to measure without a B200")
    import torch
    bench = bench_module()
    out = dict(gpu=gpu_info(), method="sweep_ms: device time of mp_sweep(1) from CUDA events on the engine stream, 256 MB L2 flush "
               "between steps, captured sweeps, median over the steps of a repeat.  ppc_ms: host wall time around one synchronous "
               "mp_ppc call (nrep replicates per chain, arena allocation and copies included) after a warm-up call, one per "
               "repeat, alternating with the sweeps.  ppc_in_sweeps = median ppc_ms / median sweep_ms", results=[])
    for name in args.workloads.split(","):
        res = run(torch, bench, name, args.nrep, args.steps, args.warmup, args.repeats)
        print(json.dumps(res), flush=True)
        out["results"].append(res)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
