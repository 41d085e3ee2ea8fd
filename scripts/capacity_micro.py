#!/usr/bin/env python
"""Cost of mp_capacity (the metapopulation capacity of every set, LOBPCG to rtol) on FP32 engines: cfg3 with the 64 chains of
bench.py after a burn-in (par = NULL: one set per chain), and cfg5 with one set (the generating alpha, b).  The call time is the
host wall time around one synchronous call (median of the repeats, after a warm-up call).  The work counters give the executed
fraction of (32 x 32) tiles and the executed pairs; the pair rate is compared with the MUFU.EX2 rate mp_probe_peaks measures on the
same card (two MUFU operations per pair: the square root of the distance and ex2).  Card name and power limit are read in the
same call.
    python scripts/capacity_micro.py [--burnin 40] [--repeats 3] [--rtol 1e-6] [--workloads cfg3,cfg5] [--out FILE]"""
import argparse
import importlib.util
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import midaspom_b200 as mb  # noqa: E402
from midaspom_b200 import synth  # noqa: E402

_spec = importlib.util.spec_from_file_location("ppc_micro", ROOT / "scripts" / "ppc_micro.py")
ppc_micro = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(ppc_micro)


def timed_calls(eng, params, rtol, repeats):
    eng.capacity(params, rtol=rtol)                                        # warm-up
    times, res = [], None
    eng.work_counters(reset=True)
    for _ in range(repeats):
        t0 = time.perf_counter()
        res = eng.capacity(params, rtol=rtol)
        times.append(time.perf_counter() - t0)
    w = eng.work_counters()
    return float(np.median(times)) * 1e3, times, res, w


def run(bench, name, burnin, repeats, rtol, mufu_gops):
    wl = synth.make_workload(name)
    if name == "cfg5":
        eng = mb.Engine(wl["n"], wl["T"], 1, precision=mb.FP32)
        eng.set_landscape_coords(wl["px"], wl["py"], wl["area"])
        params = [dict(alpha=wl["truth"]["alpha"], b=wl["truth"]["b"])]
        setup = "one set: the generating alpha, b"
    else:
        eng, _ = ppc_micro.make_engine(bench, wl, 64, False)
        eng.sweep(burnin)
        params = None
        setup = f"bench.py's 64 chains after {burnin} sweeps (par = NULL)"
    ms, times, res, w = timed_calls(eng, params, rtol, repeats)
    eng.close()
    iters = res["iters"]
    pairs = w["conn_exec"] / repeats * 1024.0
    out = dict(workload=name, n=wl["n"], sets=int(len(iters)), setup=setup, rtol=rtol, ms_per_call=ms,
               ms_all=[t * 1e3 for t in times], iters_mean=float(iters.mean()), iters_max=int(iters.max()),
               ms_per_iteration=ms / float(iters.max() + 3),     # + the start (two products) and the final product
               tile_exec_fraction=w["conn_exec"] / max(1, w["conn_total"]), pairs_per_call=pairs,
               pair_rate_gpairs=pairs / (ms * 1e-3) * 1e-9, mufu_gops=mufu_gops,
               mufu_fraction=2.0 * pairs / (ms * 1e-3) * 1e-9 / mufu_gops if mufu_gops else None,
               lam=dict(min=float(res["lam"].min()), max=float(res["lam"].max())),
               residual_max=float(res["residual"].max()), cull_bound_max=float(res["cull_bound"].max()))
    print(json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--burnin", type=int, default=40)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--rtol", type=float, default=1e-6)
    ap.add_argument("--workloads", default="cfg3,cfg5")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "capacity_micro.json"))
    args = ap.parse_args()
    bench = ppc_micro.bench_module()
    with mb.Engine(1024, 2, 1, precision=mb.FP32) as probe:
        mufu = probe.probe_peaks()["mufu_gops"]
    rows = [run(bench, name, args.burnin, args.repeats, args.rtol, mufu) for name in args.workloads.split(",")]
    rec = dict(gpu=ppc_micro.gpu_info(), what="mp_capacity host wall time per synchronous call, FP32 engines", results=rows)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(rec, indent=1) + "\n")
    print(json.dumps(rec["gpu"]))


if __name__ == "__main__":
    main()
