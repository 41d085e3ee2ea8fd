#!/usr/bin/env python
"""Forecast two ways on the same chains and seeds: mp_forecast (one weight per (target, source) pair and chain, shared by the
chain's replicates through k_conn) and mp_simulate_ensemble fed the same parameters and start states (every weight again per
trajectory).  Both calls are synchronous; the time is host wall time around the call, after one warm-up call of each, with
the two methods alternating over the repeats.  FP32 engines (the throughput path), N x N above the 126 MB of L2 at cfg5 only.
    python scripts/forecast_micro.py [--years 50] [--nrep 32] [--repeats 3] [--workloads cfg3,cfg5] [--out FILE]"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import midaspom_b200 as mb  # noqa: E402
from midaspom_b200 import synth  # noqa: E402

CHAINS = dict(cfg3=64, cfg5=1)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [v.strip() for v in out.split(",")]
        return dict(name=name, power_limit=power, sm_clock_max=clock)
    except Exception as ex:  # the numbers below still stand; say why the card is not named
        return dict(error=f"{type(ex).__name__}: {ex}")


def engine_for(wl, chains):
    eng = mb.Engine(wl["n"], wl["T"], chains, precision=mb.FP32, seed=5)
    eng.set_landscape_coords(wl["px"], wl["py"], wl["area"])
    eng.set_source_units(None)
    eng.set_observations(wl["obs"])
    t = wl["truth"]
    eng.set_params([dict(e=t["e"], c=t["c"], alpha=t["alpha"] * (1.0 + 0.01 * c), b=t["b"]) for c in range(chains)])
    eng.init_chains(mb.engine.sampler_config(n_adapt=2), disperse=False)
    eng.sweep(2)                                            # a sampler state: the latent completion of the last survey
    return eng


def run(name, years, nrep, repeats, seed=11):
    chains = CHAINS[name]
    wl = synth.make_workload(name)
    eng = engine_for(wl, chains)
    pars = eng.get_params()
    z, _ = eng.get_state()
    sims = [pars[c] for c in range(chains) for _ in range(nrep)]
    z0 = np.repeat(z[:, -1, :], nrep, axis=0)

    def forecast(ny):
        eng.work_counters(reset=True)
        t0 = time.perf_counter()
        occ, _ = eng.forecast(ny, nrep, seed=seed)
        dt = time.perf_counter() - t0
        w = eng.work_counters()
        return dt, occ.reshape(chains * nrep, ny + 1), w

    def ensemble(ny):
        t0 = time.perf_counter()
        _, occ = eng.simulate_ensemble(sims, z0, ny, seed=seed)
        return time.perf_counter() - t0, occ

    forecast(2); ensemble(2)                                # warm-up: module load, arenas, every kernel shape
    tf, te = [], []
    for _ in range(repeats):
        dt, occ_f, w = forecast(years); tf.append(dt)
        dt, occ_e = ensemble(years); te.append(dt)
    eng.close()
    same = (occ_f == occ_e).all(axis=1)
    traj_years = chains * nrep * years

    def summary(ts):
        med = float(np.median(ts))
        return dict(seconds=[round(v, 4) for v in ts], ms_per_year=med * 1e3 / years, trajectory_years_per_s=traj_years / med)

    return dict(workload=name, desc=wl["desc"], n_patches=wl["n"], chains=chains, nrep=nrep, years=years, precision="fp32",
                forecast=summary(tf), ensemble=summary(te), speedup=float(np.median(te) / np.median(tf)),
                conn_exec_fraction=w["conn_exec"] / max(1, w["conn_total"]), conn_tiles=dict(exec=w["conn_exec"], total=w["conn_total"]),
                occupied_agree_fraction=float(same.mean()), final_year_mean_occupied=dict(forecast=float(occ_f[:, -1].mean()),
                                                                                         ensemble=float(occ_e[:, -1].mean())))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--years", type=int, default=50)
    ap.add_argument("--nrep", type=int, default=32)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--workloads", default="cfg3,cfg5")
    ap.add_argument("--out", default=str(Path(__file__).resolve().parent.parent / "profiles" / "forecast_micro.json"))
    args = ap.parse_args()
    if mb.engine.load_library().mp_device_count() < 1:
        raise SystemExit("forecast_micro.py: no CUDA device; there is nothing to measure without a B200")
    out = dict(gpu=gpu_info(), method="host wall time around each synchronous call (device work and the result copies), "
               "one warm-up call of each method, then the two methods alternating; median over the repeats", results=[])
    for name in args.workloads.split(","):
        res = run(name, args.years, args.nrep, args.repeats)
        print(json.dumps(res), flush=True)
        out["results"].append(res)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
