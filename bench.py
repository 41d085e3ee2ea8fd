#!/usr/bin/env python
"""bench.py -- MCMC iterations/s of the SPOM engine on the shapes BASELINE.json names.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg3|cfg2|cfg4|cfg4l|cfg5|cfg1|tiny]
                    [--impl ours|reference] [--chains C] [--weak] [--dump-outputs DIR]

A "step" is one MCMC iteration (sweep) of every chain resident on the GPU: refresh of the
connectivity S, Metropolis steps on (alpha, b) and c, Gibbs updates of the latent z cells and of
every free intermediate-state cell y (rank-1 updates of S), Metropolis steps on e (and p).
metric = chain-iterations per second = (chains on all ranks) x K / (max over ranks of the device
time of the K steps).

Default workload: cfg3 as BASELINE.json states it -- synthetic N=10,000 patches x T=20 years, 64
independent chains IN TOTAL, sharded over the N GPUs (64/N chains each): "scaling": "strong".  Under
torchrun each rank owns its own block of chains (no data-path collective); NCCL only gathers the
draws for R-hat.  The 8-chains-per-GPU figure of round 1 is reported as extra.weak_8_chains_per_gpu
(--weak makes it the headline), and extra.cfg5_sharded carries a short run of BASELINE config 5 (one chain
at N=100,000 x T=30) on the same N GPUs, patch-sharded for N>1.

--impl reference times the CPU side.  The reference's own algorithm enumerates 2^N states and cannot
run at N >= 32, so this is the FP64 C restatement of its per-cell terms in oracle/ ("port"), one chain
per host thread on ALL host threads (explicit thread count from the affinity mask, immune to
OMP_NUM_THREADS=1 under torchrun).  Each step is a bounded sample of a sweep: the fixed part in full and
the y scan on at least 25 % of the candidate cells, extrapolated to all of them; ms_per_step is the
measured time of the sample, value the extrapolated whole-job throughput.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "mcmc_chain_iterations_per_sec"
UNIT = "chain-iterations/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="cfg3")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chains", type=int, default=0, help="total chains of the job (default: the workload's)")
    ap.add_argument("--weak", action="store_true", help="fixed chains per GPU (round-1 behaviour) instead of a fixed total")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline leg of the GPU arm")
    ap.add_argument("--ref-seconds", type=float, default=170.0, help="budget of the whole --impl reference run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra.* runs (weak figure, cfg5)")
    ap.add_argument("--no-blocks", action="store_true", help="cfg5: scan every year as a whole (no block grid)")
    ap.add_argument("--blocks-k", type=int, default=4, help="cfg5: colours per axis of the block grid")
    ap.add_argument("--torch-collectives", action="store_true", help="cfg5 on several GPUs: round-1 exchange (torch.distributed all-reduce) instead of NCCL inside the library")
    ap.add_argument("--ess-sweeps", type=int, default=1000, help="extra sweeps after the timed regions for the ESS/s figure (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed steps computed in the last one to DIR/<name>.npy "
                                                          "(rank 0's chains under torchrun), for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU arm's outputs: it needs --impl ours")
    return args


DUMP_SAMPLE = 1 << 20       # elements kept of a larger array: 3 such arrays in float64 stay below 64 MB


def dump_outputs(dirname, arrays):
    """--dump-outputs: every array as DIR/<name>.npy, in float64 if it is float64 and in float32 otherwise (0/1 states).  An
    array of more than DUMP_SAMPLE elements becomes a sample of its flattened elements drawn with a fixed seed, so that two
    runs with the same arguments store the same elements."""
    out = Path(dirname)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        if a.size > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))
            a = a.ravel()[idx]
        np.save(out / f"{name}.npy", a)


def sweep_outputs(eng):
    """What a caller of mp_sweep receives after a sweep: its draws (chains x NDRAW: e, c, alpha, b, p, loglik, n_y1, n_z1, K,
    Ksrc, dsrc), the latent states z and y, and the resident connectivity S (chains x years-1 x patches)."""
    z, y = eng.get_state()
    return dict(draws=eng.get_draws(eng.num_draws() - 1, 1)[0], z=z, y=y, S=eng.get_connectivity())


def sampler_kwargs(wl):
    c0 = wl["truth"]["c"]
    return dict(sample_e=1, sample_c=1, sample_alpha=1, sample_b=1, sample_p=int(wl["detect"]),
                e_min=0.0, e_max=1.0, c_min=0.0, c_max=20.0 * c0, alpha_min=1e-4, alpha_max=1e-1, b_min=0.0, b_max=2.0,
                p_min=0.0, p_max=1.0, n_e_steps=4, n_c_steps=1, n_adapt=200, update_z=1, update_y=1,
                sample_K=int("era" in wl and "src_unit" not in wl), K_min=0.1, K_max=100.0, n_v_steps=2,   # die-off variant: K on the reference's range (dieoff.c:113-114)
                sample_Ksrc=int("src_unit" in wl), sample_dsrc=int("src_unit" in wl),                       # patch-loss variant: K_L, d_L (loss.c:93-101)
                Ksrc_min=0.1, Ksrc_max=100.0, dsrc_min=100.0, dsrc_max=4000.0)


def start_params(wl):
    t = wl["truth"]
    return dict(e=0.5 if "era" not in wl else t["e"], c=t["c"], alpha=t["alpha"], b=t["b"], p=t["p"], K=t.get("K", 1.0), Ksrc=t.get("Ksrc", 0.0), dsrc=t.get("dsrc", 0.0))


def job_chains(wl, world, args):
    """(chains per GPU, chains of the whole job, "strong" | "weak")."""
    if args.chains:
        total = args.chains
    elif "chains_total" in wl and not args.weak:
        total = wl["chains_total"]
    else:
        return wl["chains_per_gpu"], wl["chains_per_gpu"] * world, "weak"
    if total % world:
        raise SystemExit(f"bench.py: {total} chains do not divide over {world} GPUs")
    return total // world, total, "strong"


def host_threads():
    """Threads this process may run on (the affinity mask, not OMP_NUM_THREADS: torchrun exports OMP_NUM_THREADS=1)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([v.strip() for v in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(sm))


# ----------------------------------------------------------------------------- CPU side (oracle port)
def cpu_sample(wl, job, budget_s, steps=1, warmup=0, min_frac=0.25):
    """Time the oracle's sweep (FP64 C restatement) with one chain on EVERY host thread.  Each step is a bounded sample
    of a sweep: the fixed part (two full connectivity evaluations + parameter and z updates) in full, the y scan on a
    fraction >= min_frac of the candidate cells of every year, extrapolated linearly to all candidates.  A job of `job`
    chains is ceil(job / threads) such rounds.  Returns the whole-job throughput and the measured sample times."""
    sys.path.insert(0, str(ROOT / "tests"))
    import oracle_lib as O
    m = O.Model(wl["obs"], geom=O.GEOM_COORDS, px=wl["px"], py=wl["py"], area=wl["area"], detect=wl["detect"], era=wl.get("era"),
                src_unit=wl.get("src_unit"))
    cfg = O.sampler_cfg(**sampler_kwargs(wl))
    sp = start_params(wl)
    threads = host_threads()
    nch = threads                                                    # one chain per thread: every core busy
    ch = O.Chains(m, cfg, nch, seed=1000, par0=O.params(**sp), disperse=False)
    ncand = int(((ch.z[0][:-1] & ch.z[0][1:]) == 1).sum())          # candidate cells per chain-sweep
    ntrans = wl["T"] - 1
    # probe: the fixed part + a 1 % y scan sizes the sample
    probe_limit = max(1, ncand // ntrans // 100)
    ch.run(1, y_flip_limit=probe_limit, nthreads=threads)
    t_fixed0 = float(ch.phase_s[:, 0].max())
    per_cand = max(float(ch.phase_s[:, 1].max()) / max(1.0, ch.visited / nch), 1e-8)   # s per candidate (one chain on one thread, all threads busy)
    # warm-up steps scan 1 % of the candidates (the fixed part dominates them); the timed steps share the rest of the budget,
    # each scanning at least 5 % and together at least min_frac of a sweep's candidates
    per_step = (budget_s - warmup * (t_fixed0 + 0.01 * per_cand * ncand)) / max(1, steps)
    frac = (per_step - t_fixed0) / max(per_cand * ncand, 1e-9)
    frac = float(min(1.0, max(0.05, min_frac / max(1, steps), frac)))
    per_year = max(1, int(math.ceil(frac * ncand / ntrans)))
    fixed, yscan, visited, wall = [], [], [], []
    for s in range(warmup + steps):
        t0 = time.perf_counter()
        ch.run(1, y_flip_limit=per_year if s >= warmup else probe_limit, nthreads=threads)
        dt = time.perf_counter() - t0
        if s >= warmup:
            fixed.append(float(ch.phase_s[:, 0].max())); yscan.append(float(ch.phase_s[:, 1].max()))
            visited.append(ch.visited / nch); wall.append(dt)
    t_fixed, t_y, vis = float(np.mean(fixed)), float(np.mean(yscan)), float(np.mean(visited))
    t_full = t_fixed + t_y * (ncand / max(vis, 1.0))                  # one sweep of `threads` chains, one per thread
    J = max(job, threads)                                             # the job keeps every thread busy
    rounds = math.ceil(J / threads)
    value = J / (rounds * t_full)
    sample = (f"{nch} chains on {threads} host threads (one per thread; a job of {J} chains = {rounds} such rounds), FP64 oracle port "
              f"(CPU restatement of the reference's per-cell terms, not MIDASPOM_MPI.out: the reference enumerates 2^N states); "
              f"every step: full connectivity refresh + proposal + parameter and z updates ({t_fixed:.2f} s), y scan timed on "
              f"{int(vis)} of {ncand} candidate cells per chain ({100.0 * vis / max(ncand, 1):.0f} % per step, {t_y:.2f} s; "
              f"{len(fixed)} timed steps = {100.0 * len(fixed) * vis / max(ncand, 1):.0f} % of a sweep's candidates in all) and extrapolated linearly to all")
    return dict(value=value, unit=UNIT, cores=threads, kind="port", sample=sample, t_fixed_s=t_fixed, t_y_sample_s=t_y,
                sample_fraction=vis / max(ncand, 1), ms_per_sample_step=float(np.mean(wall)) * 1e3, ms_per_full_step=rounds * t_full * 1e3,
                job_chains=J, measured_steps=len(fixed))


def run_reference(args, rank, world):
    if rank != 0:
        return
    if args.workload.startswith("cfg5"):
        emit(json.dumps(dict(impl="reference", unavailable="N=100,000: one connectivity evaluation is 1e10 pair terms (minutes per "
                              "sweep on the host); no CPU arm for this workload")), flush=True)
        return
    from midaspom_b200 import synth
    wl = synth.make_workload(args.workload)
    world_cfg = max(1, args.gpus)
    cpg, chains, scaling = job_chains(wl, world_cfg, args)
    r = cpu_sample(wl, chains, args.ref_seconds, steps=args.steps, warmup=args.warmup)
    line = dict(metric=METRIC, value=r["value"], unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=r["ms_per_sample_step"], higher_is_better=True, scaling=scaling, vs_baseline=None, dtype="f64",
                data="synthetic", impl="reference",
                config=workload_config(args, wl, chains, cpg, world_cfg),
                cpu_baseline=dict(value=r["value"], unit=UNIT, cores=r["cores"], kind=r["kind"], sample=r["sample"]),
                e2e=dict(value=r["value"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0,
                ms_per_full_step_extrapolated=r["ms_per_full_step"], sample_fraction_of_y_scan=r["sample_fraction"])
    emit(json.dumps(line), flush=True)


def workload_config(args, wl, chains, cpg, world):
    """`config` of the JSON line: identical keys and values in both arms."""
    return dict(workload=f"{args.workload}: {wl['desc']}", n_patches=wl["n"], n_years=wl["T"], chains=chains,
                geometry="planar coordinates + areas", l2="GPU arm: flushed between timed steps (256 MiB write)")


# ----------------------------------------------------------------------------- profile look-ups
def ncu_entry(workload, kernel):
    """Newest tracked ncu summary (profiles/*_ncu_full*.json) of this kernel ON THIS WORKLOAD, or None."""
    for f in sorted((ROOT / "profiles").glob("*_ncu_full*.json"), reverse=True):
        try:
            entries = json.loads(f.read_text())
        except Exception:
            continue
        for kd in entries:
            if kd.get("workload") == workload and kernel in kd.get("kernel", ""):
                return kd, f"profiles/{f.name}"
    return None, None


def ncu_counters(workload, kernel):
    kd, src = ncu_entry(workload, kernel)
    if kd is None:
        return None, None
    pick = {"pipe_xu_pct": "sm__inst_executed_pipe_xu.avg.pct_of_peak_sustained_active",
            "pipe_fma_pct": "sm__inst_executed_pipe_fma.avg.pct_of_peak_sustained_active",
            "pipe_fp64_pct": "sm__inst_executed_pipe_fp64.avg.pct_of_peak_sustained_active",
            "pipe_lsu_pct": "sm__inst_executed_pipe_lsu.avg.pct_of_peak_sustained_active",
            "issue_active_pct": "smsp__issue_active.avg.pct_of_peak_sustained_active",
            "warps_active_pct": "sm__warps_active.avg.pct_of_peak_sustained_active",
            "dram_pct": "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
            "tensor_pct": "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"}
    c = {}
    for k, name in pick.items():
        if name in kd:
            try:
                c[k] = float(str(kd[name]).replace(",", ""))
            except ValueError:
                pass
    c["source"] = src
    traffic = kd.get("dram_traffic_bytes_per_launch")
    return c, (dict(bytes_per_launch=traffic, source=src, note="dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this kernel on this workload") if traffic is not None else None)


# ----------------------------------------------------------------------------- our arm
class Arm:
    """One engine with the bench's workload resident, and the timed loops over it."""

    def __init__(self, torch, mb, wl, cpg, first, local_rank, max_draws):
        self.torch, self.mb, self.wl, self.cpg, self.dev = torch, mb, wl, cpg, local_rank
        n, T = wl["n"], wl["T"]
        self.eng = eng = mb.Engine(n, T, cpg, precision=mb.FP32, device=local_rank, seed=1000, detect=wl["detect"], chain_offset=first,
                                   max_draws=max_draws)
        eng.set_landscape_coords(wl["px"], wl["py"], wl["area"])
        eng.set_source_units(wl.get("src_unit"))
        self.obs_pinned = torch.from_numpy(wl["obs"].copy()).pin_memory()
        self.obs_host = self.obs_pinned.numpy()
        eng.set_observations(self.obs_host)
        eng.set_era(wl.get("era"))
        eng.set_params([start_params(wl)] * cpg)
        eng.init_chains(mb.engine.sampler_config(**sampler_kwargs(wl)), disperse=False)
        self.stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", local_rank))

    def timed_steps(self, nsteps, flush, e2e=False):
        """CUDA events on the engine's stream around every step; the chain state is evicted from L2 between steps."""
        torch, eng = self.torch, self.eng
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nsteps)]
        with torch.cuda.stream(self.stream):
            for a, b in evs:
                flush.fill_(1)
                a.record(self.stream)
                if e2e:
                    eng.set_observations(self.obs_host)               # H2D from pinned memory, every step
                    eng.sweep(1, sync=False)
                    eng.get_draws(eng.num_draws() - 1, 1)             # D2H of the step's result (syncs)
                else:
                    eng.sweep(1, sync=False)
                b.record(self.stream)
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in evs]


def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import midaspom_b200 as mb
    from midaspom_b200 import synth, distributed as D

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    wl = synth.make_workload(args.workload)
    if args.workload.startswith("cfg5"):
        line = run_cfg5(args, rank, local_rank, world, wl, args.steps, args.warmup, dump=args.dump_outputs)
        if rank == 0:
            emit(json.dumps(line), flush=True)
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return
    cpg, chains_total, scaling = job_chains(wl, world, args)
    first, _ = D.chain_block(rank, world, cpg)
    K, W = args.steps, args.warmup
    n, T = wl["n"], wl["T"]
    dev = f"cuda:{local_rank}"
    arm = Arm(torch, mb, wl, cpg, first, local_rank, max_draws=3 * K + W + 8 + max(0, args.ess_sweeps))
    eng = arm.eng
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    # ---- the timed region: K steps, engine-internal per-kernel timing OFF
    eng.sweep(W)                                                 # warm-up (untimed)
    eng.set_timing(False)
    barrier()
    with ClockSampler(local_rank) as clk:
        barrier()
        t_wall0 = time.perf_counter()
        step_ms = arm.timed_steps(K, flush)
        barrier()
        t_wall = time.perf_counter() - t_wall0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sweep_outputs(eng))      # before the other arms sweep the same chains further
    launches0 = sum(eng.get_timing(reset=True)[1].values())      # launch counters run with timing off too
    total_ms = float(sum(step_ms))
    # ---- end-to-end arm: host buffers in and out every step
    barrier()
    e2e_ms = arm.timed_steps(K, flush, e2e=True)
    barrier()
    e2e_total = float(sum(e2e_ms))
    eng.get_timing(reset=True)
    # ---- kernel split and work counters: a separate pass of K steps with per-kernel CUDA events ON (not part of `value`)
    eng.set_timing(True)
    eng.work_counters(reset=True)
    eng.get_timing(reset=True)
    split_ms = arm.timed_steps(K, flush)
    kms, klaunch = eng.get_timing(reset=True)
    work = eng.work_counters(reset=True)
    scan_geo = eng.scan_geometry()
    eng.set_timing(False)
    split_total = float(sum(split_ms))
    total_ms, e2e_total = max_over_ranks([total_ms, e2e_total])
    value = chains_total * K / (total_ms * 1e-3)
    e2e_value = chains_total * K / (e2e_total * 1e-3)

    # ---- ESS/s (third part of BASELINE's metric): a longer run after the timed regions, wall clock, second half of its draws
    ess_run = None
    n_ess = min(args.ess_sweeps, int(15000.0 / max(total_ms / K, 1e-3)))      # at most ~15 s of extra sweeps
    if n_ess >= 100:
        barrier()
        t0 = time.perf_counter()
        eng.sweep(n_ess)
        barrier()
        ess_run = time.perf_counter() - t0
    # ---- likelihood evaluations/s (second part of BASELINE's metric): 1 evaluation = full connectivity S of the resident
    # state + the summed log-terms of one chain (SURVEY 8d) = one chain's share of one mp_loglik call (the call recomputes S
    # from scratch every time; it is not preceded by mp_connectivity, which would compute the same S a second time)
    barrier()
    n_ll = 10
    eng.loglik()
    t0 = time.perf_counter()
    for _ in range(n_ll):
        eng.loglik()
    barrier()
    (t_ll,) = max_over_ranks([time.perf_counter() - t0])
    lik_evals = chains_total * n_ll / t_ll
    # the same through host buffers: parameters, z and y of every chain go in with the call (mp_loglik_host), per-chain sums come back
    par_h = eng.get_params()
    z_h, y_h = eng.get_state()
    eng.loglik_host(par_h, z_h, y_h)
    barrier()
    t0 = time.perf_counter()
    for _ in range(n_ll):
        eng.loglik_host(par_h, z_h, y_h)
    barrier()
    (t_ll_h,) = max_over_ranks([time.perf_counter() - t0])
    lik_evals_host = dict(value=chains_total * n_ll / t_ll_h, h2d_bytes_per_call=int(z_h.nbytes + y_h.nbytes),
                          note="mp_loglik_host: z and y of every chain copied from (pageable) host arrays inside the timed call")
    # posterior diagnostics on everything recorded so far (gathered over ranks with NCCL)
    nd = eng.num_draws()
    d_local = torch.from_numpy(eng.get_draws(0, nd)).to(dev)
    d_all = D.gather_draws(d_local).cpu().numpy()
    if ess_run is not None:
        half = n_ess // 2
        summ = D.posterior_summary(d_all[nd - half:])
        run_s = ess_run * half / n_ess
    else:
        summ = D.posterior_summary(d_all[W:])
        run_s = (total_ms + e2e_total) * 1e-3
    ess_min = min((v["ess"] for v in summ.values()), default=float("nan"))
    z, y = eng.get_state()
    ncand = float(((z[:, :-1] & z[:, 1:]) == 1).sum()) / cpg             # candidate cells per chain-sweep
    # the same evaluation for a batch of chains that share (alpha, b): the connectivity is one dense contraction and runs on the
    # tensor cores (k_conn_gemm: tcgen05.mma + TMEM + TMA); every chain gets chain 0's current parameters
    p0 = eng.get_params()[0]
    eng.set_params([p0] * cpg)
    eng.loglik()
    barrier()
    t0 = time.perf_counter()
    for _ in range(n_ll):
        eng.loglik()
    barrier()
    (t_ll_g,) = max_over_ranks([time.perf_counter() - t0])
    lik_evals_shared = dict(value=chains_total * n_ll / t_ll_g, connectivity_kernel=eng.conn_path(),
                            note="all chains of a GPU hold the same (alpha, b): fixed-parameter batch evaluation")
    probe = eng.probe_peaks() if rank == 0 else None
    eng.close()
    del arm

    # ---- extras (after the headline's timed regions; every rank takes part, rank 0 reports)
    extra = {}
    if not args.no_extra:
        if args.workload == "cfg3" and scaling == "strong":
            if cpg == 8:
                extra["weak_8_chains_per_gpu"] = dict(value=value, unit=UNIT, ms_per_step=total_ms / K, chains=chains_total,
                                                      note="identical to the headline at this GPU count (64 / 8 = 8 chains per GPU)")
            else:
                arm8 = Arm(torch, mb, wl, 8, rank * 8, local_rank, max_draws=K + W + 4)
                arm8.eng.sweep(W)
                barrier()
                ms8 = arm8.timed_steps(K, flush)
                (t8,) = max_over_ranks([float(sum(ms8))])
                extra["weak_8_chains_per_gpu"] = dict(value=8 * world * K / (t8 * 1e-3), unit=UNIT, ms_per_step=t8 / K, chains=8 * world,
                                                      note="round-1 configuration: 8 chains on every GPU (152 year tasks on 148 SMs)")
                arm8.eng.close()
                del arm8
        if args.workload == "cfg3":
            try:
                wl5 = synth.make_workload("cfg5", device=local_rank)
                l5 = run_cfg5(args, rank, local_rank, world, wl5, steps=4, warmup=2)
                if rank == 0:
                    extra["cfg5_sharded"] = {k: l5[k] for k in ("value", "unit", "ms_per_step", "n_gpus", "scaling", "config", "phase_ms_per_sweep",
                                                                 "collective_bytes_per_sweep", "ranks_hold_identical_draws", "steps", "warmup") if k in l5}
            except Exception as ex:      # an extra must never cost the headline
                extra["cfg5_sharded"] = dict(error=f"{type(ex).__name__}: {ex}")

    if rank == 0:
        peaks_meas = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()) if (ROOT / "MEASURED_PEAKS.json").exists() else {}
        hbm_peak = float(peaks_meas.get("hbm_gbs", 6650.0))
        roof = roofline(args.workload, wl, cpg, ncand, kms, klaunch, work, scan_geo, probe, hbm_peak, bool(peaks_meas), split_total)
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=K, warmup=W, ms_per_step=total_ms / K,
                    higher_is_better=True, scaling=scaling, vs_baseline=None, dtype="f32", data="synthetic",
                    config=workload_config(args, wl, chains_total, cpg, world),
                    run=dict(chains_per_gpu=cpg, weights="evaluated on the fly from the coordinates",
                             connectivity=dict(sampler="k_conn, year contraction in FP64 (DFMA): rank-1 removals by the y scan cancel exactly",
                                               likelihood_calls="k_conn, year contraction in FP32 (FFMA2, partial sums per 32 sources joined in FP64); "
                                                                "k_conn_gemm (tcgen05) when every chain holds the same (alpha, b)"),
                             sampled=["e", "c", "alpha", "b"] + (["p"] if wl["detect"] else []) + (["Ksrc", "dsrc"] if "src_unit" in wl else ["K"] if "era" in wl else []),
                             parallelism=f"chains x{world}", scan=scan_geo),
                    clocks=clk.summary(),
                    e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=int(arm_bytes(wl)),
                             d2h_bytes_per_step=int(cpg * mb.NDRAW * 8), ms_per_step=e2e_total / K),
                    gpu_launches=int(launches0),
                    kernel_ms={k: round(v, 4) for k, v in kms.items()}, kernel_launches=klaunch,
                    kernel_split_note=f"separate pass of {K} steps with per-kernel CUDA events on ({split_total / K:.3f} ms per step); `value` is timed with them off",
                    wall_s_timed_region=t_wall,
                    likelihood_evals_per_sec=lik_evals, likelihood_evals_per_sec_host_buffers=lik_evals_host,
                    likelihood_evals_per_sec_shared_params=lik_evals_shared,
                    ess_per_sec=ess_min / run_s if run_s > 0 else None,
                    ess=dict(min_ess=ess_min, seconds=run_s, sweeps=(n_ess // 2 if ess_run is not None else nd - W),
                             note="min over sampled parameters of the summed per-chain ESS (Geyer), second half of a separate "
                                  f"{n_ess}-sweep run, wall clock" if ess_run is not None else "timed draws only"),
                    posterior=summ, candidates_per_chain_sweep=ncand, roofline=roof, extra=extra,
                    parity_note="cfg2-cfg5 use extensions the reference has no code for (planar coordinates, areas, sampled alpha and b): "
                                "checked against the CPU restatement only (parity unpinned except at the reference's degenerate point)")
        if not args.no_cpu_baseline and world == 1:
            try:
                r = cpu_sample(wl, chains_total, args.cpu_seconds, steps=1, warmup=0, min_frac=0.5)
                line["cpu_baseline"] = dict(value=r["value"], unit=UNIT, cores=r["cores"], kind=r["kind"], sample=r["sample"])
            except Exception as ex:  # the oracle is test infrastructure: never let it break the GPU line
                line["cpu_baseline"] = dict(value=None, unit=UNIT, cores=0, kind="port", sample=f"failed: {ex}")
        emit(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def arm_bytes(wl):
    return wl["obs"].nbytes


def roofline(workload, wl, cpg, ncand, kms, klaunch, work, geo, probe, hbm_peak, have_peaks, split_total_ms):
    """Roofline of the dominant kernel (the y scan) from EXECUTED work: the always-on work counters of the engine
    (mp_get_work_counters) give the (candidate, 32-target group) evaluations and rank-1 updates the kernel really ran."""
    n, T = wl["n"], wl["T"]
    n_scan = max(1, klaunch["sweep_y"])
    t_scan = kms["sweep_y"] / n_scan * 1e-3                               # s per launch (CUDA events on the engine stream)
    sp = max(1, geo["candidates_per_trip"])
    lg2_share = (sp + 1) / (4.0 * sp)                                     # one MUFU.LG2 per product of <= 4 factors, sp numerators + 1 denominator
    dense_pairs = cpg * ncand * (n - 1)                                   # per launch, the dense algorithm's count
    if geo["culled"]:
        kernel = "k_sweep_y_cull"
        retired = work["scan_retired"] * 32.0 / n_scan                    # (candidate, target) evaluations of candidates decided in their trip
        executed = work["scan_exec"] * 32.0 / n_scan                      # the same plus re-evaluated speculative ones
        commit = work["scan_commit"] * 32.0 / n_scan                      # rank-1 updates of S
        bounds = work["scan_trips"] * 32.0 * sp / n_scan                  # per trip every lane bounds one group against sp candidates
        mufu_required = retired * (2.0 + lg2_share) + commit * 2.0
        mufu_executed = executed * (2.0 + lg2_share) + commit * 2.0 + bounds * 2.0
    else:
        kernel = "k_sweep_y_fast"
        retired = executed = work["scan_dense"] / n_scan
        commit = retired / 3.0                                            # about one flip in three is accepted; the commit pass covers all targets
        mufu_required = mufu_executed = retired * 2.2 + commit * 2.2
    peak = probe["mufu_gops"]
    counters, traffic = ncu_counters(workload, kernel)
    alg_bytes = cpg * (T - 1) * n * (8 + 1 + 1 + 1 + 8 + 1) + cpg * ncand * 32   # S,y,z_t,z_t+1 in; S,y out; candidate records
    frac = mufu_required / t_scan * 1e-9 / peak
    roof = dict(bound="sfu", kernel=kernel, achieved=mufu_required / t_scan * 1e-9, peak=peak, unit="Gop/s (MUFU)",
                frac=frac, traffic=(traffic or {}).get("bytes_per_launch"), traffic_detail=traffic, counters=counters,
                share_of_step=kms["sweep_y"] / max(split_total_ms, 1e-9), ms_per_launch=t_scan * 1e3,
                executed=dict(achieved=mufu_executed / t_scan * 1e-9, frac=mufu_executed / t_scan * 1e-9 / peak,
                              note="every MUFU the kernel issued for weights: speculative re-evaluations and the per-trip group bounds included "
                                   "(comparable with ncu's XU-pipe utilisation)"),
                effective_vs_dense=dict(value=dense_pairs * 2.2 / t_scan * 1e-9 / peak,
                                        note="dense-equivalent: counts the (candidate, target) pairs the exact culling skips as if they had "
                                             "been evaluated; may exceed 1 and is NOT a roofline fraction"),
                algorithmic=dict(pairs_required_per_launch=retired, pairs_executed_per_launch=executed, commit_pairs_per_launch=commit,
                                 dense_pairs_per_launch=dense_pairs, evaluated_fraction_of_dense=retired / max(dense_pairs, 1.0),
                                 mufu_per_eval_pair=2.0 + lg2_share, mufu_per_commit_pair=2.0, bytes_per_launch=alg_bytes,
                                 note="frac = MUFU operations of the algorithmically required pair evaluations (candidates decided in their trip, "
                                      "targets within FP32 reach) and rank-1 updates / launch time / MUFU peak; counts come from the engine's "
                                      "work counters, not from a model"),
                peak_source="builder-measured: mp_probe_peaks micro-benchmark on this GPU in this run (MEASURED_PEAKS.json has no MUFU figure)",
                hbm=dict(achieved=alg_bytes / t_scan * 1e-9, peak=hbm_peak, unit="GB/s", frac=alg_bytes / t_scan * 1e-9 / hbm_peak,
                         peak_source="MEASURED_PEAKS.json" if have_peaks else "fallback"),
                probe=probe)
    n_conn = max(1, klaunch["conn"])
    t_conn = kms["conn"] / n_conn * 1e-3
    conn_pairs = work["conn_exec"] * 1024.0 / n_conn                      # executed (target, source) pairs per launch
    conn_total = work["conn_total"] * 1024.0 / n_conn
    c_counters, c_traffic = ncu_counters(workload, "k_conn")
    roof["conn"] = dict(kernel="k_conn", ms_per_launch=t_conn * 1e3, achieved=conn_pairs * 2.0 / t_conn * 1e-9, unit="Gop/s (MUFU)",
                        frac=conn_pairs * 2.0 / t_conn * 1e-9 / peak, pairs_executed_per_launch=conn_pairs,
                        pairs_dense_per_launch=conn_total, share_of_step=kms["conn"] / max(split_total_ms, 1e-9),
                        counters=c_counters, traffic=(c_traffic or {}).get("bytes_per_launch"), traffic_detail=c_traffic)
    # the sampler's k_conn contracts every executed pair over the years in FP64: the FP64 pipe, not the MUFU, bounds it
    nyb = min(32, (T - 1 + 3) // 4 * 4)                                   # year accumulators per target and pass (k_conn's NYB)
    fp64_peak = float(probe.get("dadd_gops", 0.0)) if probe else 0.0
    if fp64_peak > 0:
        dfma = conn_pairs * nyb                                           # conn_exec counts every pass (32 years each) over the sources
        roof["conn"]["fp64"] = dict(achieved=dfma / t_conn * 1e-9, peak=fp64_peak, unit="Gop/s (DFMA)", frac=dfma / t_conn * 1e-9 / fp64_peak,
                                    dfma_per_pair=nyb, note="executed (target, source) pairs x year accumulators / launch time / FP64 peak "
                                                            "(mp_probe_peaks, builder-measured); compare with counters.pipe_fp64_pct")
    return roof


# ----------------------------------------------------------------------------- cfg5: one chain, patch-sharded over the GPUs
def run_cfg5(args, rank, local_rank, world, wl, steps, warmup, dump=None):
    """BASELINE config 5: one chain at N=100,000 x T=30 on the `world` GPUs of the box.  N=1: a single engine.  N>1:
    midaspom_b200/distributed.py ShardedChain (connectivity by target patches, y scan by years, collectives per sweep).
    Total work is fixed: "scaling": "strong".  `dump`: directory of --dump-outputs.  Returns the JSON line (rank 0) or None."""
    if dump and world > 1:
        raise SystemExit("bench.py: --dump-outputs does not support a chain sharded over several GPUs (cfg5 with --gpus > 1)")
    import torch
    import torch.distributed as dist
    import midaspom_b200 as mb
    from midaspom_b200 import distributed as D
    K, W = steps, warmup
    n, T, C = wl["n"], wl["T"], wl["chains_per_gpu"]
    dev = torch.device("cuda", local_rank)
    eng = mb.Engine(n, T, C, precision=mb.FP32, device=local_rank, seed=1000, detect=wl["detect"], chain_offset=0, max_draws=K + W + 4)
    eng.set_landscape_coords(wl["px"], wl["py"], wl["area"]); eng.set_source_units(None)
    eng.set_observations(wl["obs"])
    eng.set_params([start_params(wl)] * C)
    eng.init_chains(mb.engine.sampler_config(**sampler_kwargs(wl)), disperse=False)
    # block grid of the y scan: blocks of one colour are scanned concurrently (mp_set_scan_blocks); the halo comes from the
    # start parameters and the smallest connectivity of the start state, with a margin for what the sampler does to them
    grid = None
    if not getattr(args, "no_blocks", False):
        p0 = start_params(wl)
        grid = eng.set_scan_blocks_auto(wl["px"], wl["py"], p0["alpha"], float(eng.get_connectivity().min()),
                                        float(np.max(np.asarray(wl["area"]) ** p0["b"])), k=getattr(args, "blocks_k", 4))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    sc = None
    if world > 1:
        sc = D.ShardedChain(eng, rank, world, dev) if getattr(args, "torch_collectives", False) else D.NativeShardedChain(eng)
    run = (lambda k: sc.sweep(k)) if sc else (lambda k: eng.sweep(k))
    run(W)
    if sc and hasattr(sc, "phase_s"):
        sc.phase_s = dict.fromkeys(sc.phase_s, 0.0)
    eng.get_timing(reset=True)
    eng.work_counters(reset=True)
    times = []
    with ClockSampler(local_rank) as clk:
        for _ in range(K):
            flush.fill_(1)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(1)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
    if dump:
        dump_outputs(dump, sweep_outputs(eng))
    t = torch.tensor([sum(times)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_s = float(t[0])
    identical = True
    if world > 1:
        draws = eng.get_draws()
        same = torch.tensor(draws[-1, 0, :6], device=dev)
        ref = same.clone(); dist.broadcast(ref, 0)
        ok = torch.tensor([1.0 if bool((same == ref).all()) else 0.0], device=dev); dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        identical = bool(ok.item() == 1.0)
    line = None
    if rank == 0:
        _, klaunch = eng.get_timing(reset=False)
        line = dict(metric=METRIC, value=C * K / total_s, unit=UNIT, n_gpus=world, steps=K, warmup=W, ms_per_step=total_s / K * 1e3,
                    higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f32", data="synthetic",
                    config=dict(workload=f"cfg5: {wl['desc']}", n_patches=n, n_years=T, chains=C,
                                parallelism=(sc.describe() if sc else "one engine on one GPU"),
                                l2="flushed between timed steps (256 MiB write)", scan=eng.scan_geometry(),
                                scan_blocks=(dict(nx=grid[0], ny=grid[1], colours=grid[2] ** 2, halo_m=round(grid[3], 1),
                                                  block_tasks_per_sweep=eng.work_counters()["scan_blocks"] / K) if grid else None),
                                timing="host clock between device synchronisations, max over ranks"),
                    clocks=clk.summary(), gpu_launches=int(sum(klaunch.values())),
                    ranks_hold_identical_draws=identical,
                    e2e=dict(value=C * K / total_s, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0,
                             note="state resident; the sharded loop has no per-step host buffers"))
        if sc:
            line["collective_bytes_per_sweep"] = int(sc.bytes_per_sweep())
            if hasattr(sc, "phase_s"):
                line["phase_ms_per_sweep"] = {k: round(v / K * 1e3, 3) for k, v in sc.phase_s.items()}
    eng.close()
    return line


# ----------------------------------------------------------------------------- cfg1: the bundled example, exact grid posterior
def run_cfg1(args, rank):
    """BASELINE config[0]: `MIDASPOM.out -m 400 -d 100` on the bundled 8 x 7 example = 101 x 101 = 10,201 exact
    likelihood evaluations (run_examples.sh:8).  ours: mp_exact_posterior (host buffers in and out);
    reference: the reference binary itself, compiled from its sources into oracle/_ref (kind "reference"), one copy per
    host thread running concurrently (MIDASPOM_MPI.out is a static row split of the same loop, main_MIDASPOM_MPI.c:361-372;
    no MPI runtime exists in the image, so N concurrent serial copies stand in for it)."""
    if rank != 0:
        return
    import tempfile
    example = ROOT / "tests" / "golden" / "occupancies_example.txt"
    nev = 101 * 101
    cfgd = dict(workload="cfg1: bundled example (8 patches x 7 years), 101 x 101 grid of (e, c), exact likelihood", grid=101)
    if args.impl == "reference":
        exe = ROOT / "oracle" / "_ref" / "MIDASPOM.out"
        if not exe.exists():
            emit(json.dumps(dict(impl="reference", unavailable="oracle/_ref/MIDASPOM.out not built (make -C oracle ref REF=<reference checkout>)")))
            return
        tmp = tempfile.mkdtemp()
        threads = host_threads()

        def one(i):
            subprocess.run([str(exe), "-m", "400", "-d", "100", "-i", str(example), "-o", f"{tmp}/p{i}.txt"], check=True, capture_output=True)

        def timed(copies):
            ts = []
            for s in range(args.warmup + args.steps):
                t0 = time.perf_counter()
                th = [threading.Thread(target=one, args=(i,)) for i in range(copies)]
                [t.start() for t in th]; [t.join() for t in th]
                if s >= args.warmup:
                    ts.append(time.perf_counter() - t0)
            return float(np.mean(ts))
        t1 = timed(1)
        tall = timed(threads)
        v1, vall = nev / t1, nev * threads / tall
        emit(json.dumps(dict(metric="likelihood_evals_per_sec", value=vall, unit="likelihood evaluations/s", n_gpus=args.gpus, steps=args.steps,
                              warmup=args.warmup, ms_per_step=tall * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64",
                              data="bundled example", impl="reference", config=cfgd,
                              cpu_baseline=dict(value=vall, unit="likelihood evaluations/s", cores=threads, kind="reference",
                                                sample=f"{threads} concurrent copies of MIDASPOM.out (reference sources, gcc -O3, naive cblas_dgemm), whole "
                                                       f"program incl. file I/O, one per host thread; a single copy on one thread: {v1:.0f} evaluations/s"),
                              single_thread=dict(value=v1, ms_per_run=t1 * 1e3),
                              e2e=dict(value=vall, unit="likelihood evaluations/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)))
        return
    import torch
    import midaspom_b200 as mb
    raw = example.read_bytes()
    n = 1 + sum(1 for ch in raw.split(b"\n", 1)[0] if ch in b" \t")
    tmax = raw.count(b"\n")
    obs = np.array([int(v) for v in raw.split()][: n * tmax], dtype=np.int8).reshape(tmax, n)
    times = []
    for s in range(args.warmup + args.steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ll, ltot, info = mb.exact_posterior(obs, a=1 / 400, d=100.0, prior_occ=0.5, nstep=101)
        if s >= args.warmup:
            times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(loglik=ll, ltot=np.array([ltot])))
    t = float(np.mean(times))
    v = nev / t
    emit(json.dumps(dict(metric="likelihood_evals_per_sec", value=v, unit="likelihood evaluations/s", n_gpus=1, steps=args.steps, warmup=args.warmup,
                          ms_per_step=t * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="bundled example",
                          config=dict(cfgd, states=info["nstates"], short_states=info["nextid"], total_loglik=ltot),
                          ms_per_step_min=float(np.min(times)) * 1e3, ms_per_step_median=float(np.median(times)) * 1e3,
                          e2e=dict(value=v, unit="likelihood evaluations/s", h2d_bytes_per_step=int(obs.nbytes), d2h_bytes_per_step=nev * 8),
                          gpu_launches=2 * args.steps)))


_REAL_STDOUT = None


def emit(line, flush=True):
    """The ONE JSON line of the contract goes to the process's real stdout; everything else any library writes to
    file descriptor 1 (NCCL prints its version there under torchrun) has been redirected to stderr by main()."""
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(line + "\n")
    if flush:
        out.flush()


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    args = parse_args()
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.workload == "cfg1":
        run_cfg1(args, rank)
    elif args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
