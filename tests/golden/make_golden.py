"""Generate tests/golden/golden.npz from THE REFERENCE ITSELF (run in the build container only).

Needs a checkout of the reference and oracle/_ref built from it (make -C oracle ref REF=<dir>).  The
tests read the committed golden.npz and need neither.

    REF=<dir> python tests/golden/make_golden.py

What is recorded (all produced by reference code, none by our oracle):
  example_obs        the bundled example as the reference's stream-order parser reads it
                     (main_MIDASPOM.c:138-167), taken from the program's own "Year i:" echo (:293-298)
  post_default       101x101 posterior table of `MIDASPOM.out -m 400 -d 100` (run_examples.sh:8)
  post_s11           11x11 table of `-s 11` (includes the e=0 / c=0 edges where the likelihood is 0)
  post_s3            3x3 table of `-s 3 -l 0.3 -u 0.7`; loglik_s3_survey: the log-likelihoods of the
                     same grid recorded in SURVEY.md section 8c
  ltot_*             the "Total log-likelihood" line (5 decimals, :425)
  dieoff_s151        `MIDASPOM_dieoff.out -a 10 -e 0.71 -c 0.52 -m 400 -d 100 -s 151` (run_examples.sh:11)
  loss_s7v3          `MIDASPOM_loss.out   -a 10 -e 0.71 -c 0.52 -m 400 -d 100 -s 7 -v 3`
  cpp_*              compPePc (serial product form and MPI log form) on the example's state tables
  var_*              pije / pijc / pijcsource / dieoff variants on random 6-patch state triples
  simpij_*           10,000 draws of simpij from one state (libc rand(), srand(12345))
  future_*_runs      6 runs of `MIDASPOM_future.out -a 50 -m 400 -d 100 -q posterior.txt` (run_examples.sh:17,20): extinct counts per year
"""
import ctypes as C
import os
import re
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent))
import oracle_lib as O  # noqa: E402

if not os.environ.get("REF"):
    sys.exit("make_golden.py needs REF=<directory of a reference checkout>")
EXAMPLE = str(Path(os.environ["REF"]) / "examples" / "input" / "occupancies.txt")


def run(prog, args):
    out = subprocess.run([str(O.REF_BIN / prog)] + args, check=True, capture_output=True, text=True).stdout
    return out


def table(path):
    return np.array([[float(v) for v in line.split()] for line in Path(path).read_text().splitlines() if line.strip()])


def main():
    O.build_oracle()
    assert O.have_ref(), "oracle/_ref missing: run make -C oracle ref"
    g = {}
    tmp = Path(tempfile.mkdtemp())
    out = run("MIDASPOM.out", ["-m", "400", "-d", "100", "-i", EXAMPLE, "-o", str(tmp / "p.txt")])
    rows = re.findall(r"Year \d+: ([-\d ]+)\n", out.split("Input occupancy data:")[1].split("Number of possible")[0])
    g["example_obs"] = np.array([[int(v) for v in r.split()] for r in rows], dtype=np.int8)
    g["post_default"] = table(tmp / "p.txt")
    g["ltot_default"] = float(re.search(r"Total log-likelihood=([-\d.]+)", out).group(1))
    out = run("MIDASPOM.out", ["-m", "400", "-d", "100", "-s", "11", "-i", EXAMPLE, "-o", str(tmp / "p11.txt")])
    g["post_s11"] = table(tmp / "p11.txt")
    g["ltot_s11"] = float(re.search(r"Total log-likelihood=([-\d.]+)", out).group(1))
    out = run("MIDASPOM.out", ["-m", "400", "-d", "100", "-s", "3", "-l", "0.3", "-u", "0.7", "-i", EXAMPLE, "-o", str(tmp / "p3.txt")])
    g["post_s3"] = table(tmp / "p3.txt")
    g["ltot_s3"] = float(re.search(r"Total log-likelihood=([-\d.]+)", out).group(1))
    g["loglik_s3_survey"] = np.array([[-42.264661832917, -44.586856259586, -48.386656788855],
                                      [-38.506491291687, -38.903129146384, -40.977489281515],
                                      [-38.335574831701, -37.064899913015, -37.732493912103]])
    # prior 0.25 (exact in float) to pin the year-0 prior; missing cell moved into year 0
    obs2 = g["example_obs"].copy(); obs2[0, 1] = -1; obs2[0, 4] = -1
    f2 = tmp / "obs2.txt"
    f2.write_text("\n".join(" ".join(str(int(v)) for v in r) for r in obs2) + "\n")
    g["obs_prior"] = obs2
    # NB year-0 missing cells leave part of Pold uninitialised in the serial program (SURVEY 5);
    # with 2 missing cells npstates[0]=4 and only Pold[0..3] are set while 4*npstates[j-1] are read.
    # => not recorded as an absolute golden.  Kept only as an input for oracle-vs-oracle tests.
    run("MIDASPOM_dieoff.out", ["-a", "10", "-e", "0.71", "-c", "0.52", "-m", "400", "-d", "100", "-s", "151", "-i", EXAMPLE, "-o", str(tmp / "d.txt")])
    g["dieoff_s151"] = table(tmp / "d.txt")[0]
    run("MIDASPOM_loss.out", ["-a", "10", "-e", "0.71", "-c", "0.52", "-m", "400", "-d", "100", "-s", "7", "-v", "3", "-i", EXAMPLE, "-o", str(tmp / "l.txt")])
    g["loss_s7v3"] = table(tmp / "l.txt")

    # ---- compPePc on the example's own state tables (built here exactly as main_MIDASPOM.c:198-287 does)
    obs = g["example_obs"].astype(int)
    T, n = obs.shape
    var = (obs != 0).any(axis=0)
    nvar = int(var.sum())
    nstates = 2 ** nvar
    piall = np.zeros((nstates, n), dtype=np.uint32)
    for i in range(nstates):
        jt = 0
        for j in range(n):
            if var[j]:
                piall[i, j] = (i // (2 ** (nvar - jt - 1))) % 2
                jt += 1
    # short list of states compatible with the observations, in the reference's discovery order
    short = []
    for t in range(T):
        miss = [j for j in range(n) if obs[t, j] == -1]
        for k in range(2 ** len(miss)):
            row = obs[t].copy()
            for m_i, j in enumerate(miss):
                st1 = (2 ** len(miss)) // (2 ** (m_i + 1))
                row[j] = (k // st1) % 2
            jt, sid = 0, 0
            for j in range(n):
                if var[j]:
                    sid += int(row[j]) * 2 ** (nvar - jt - 1); jt += 1
            if sid not in short:
                short.append(sid)
    all2short = np.array(short, dtype=np.uint32)
    nextid = len(short)
    a, d, e, c = 1.0 / 400, 100.0, 0.71, 0.52
    M = O.ref_kernel_matrix(n, a, d)
    R = O.ref()
    u32p, dp = C.POINTER(C.c_uint32), C.POINTER(C.c_double)
    for name, fn in (("base", R.ref_base_compPePc), ("mpi", R.ref_mpi_compPePc)):
        Pe = np.zeros((nextid, nstates)); Pc = np.zeros((nstates, nextid))
        for j in range(nstates):
            pC = np.minimum(1.0, c * (M.T @ piall[j].astype(float)))   # main_MIDASPOM.c:351-358 (diag of M is 0)
            # reproduce the reference's accumulation order exactly instead of the BLAS dot product
            for k in range(n):
                s1 = 0.0
                for l in range(n):
                    if l != k:
                        s1 += M[l, k] * float(piall[j, l])
                pC[k] = min(1.0, c * s1)
            fn(Pe.ctypes.data_as(dp), Pc.ctypes.data_as(dp), piall.ctypes.data_as(u32p), all2short.ctypes.data_as(u32p),
               e, pC.ctypes.data_as(dp), M.ctypes.data_as(dp), n, nextid, nstates, j)
        g[f"cpp_{name}_Pe"], g[f"cpp_{name}_Pc"] = Pe, Pc
    g["cpp_piall"], g["cpp_all2short"] = piall, all2short
    g["cpp_params"] = np.array([a, d, e, c])

    # ---- variant functions on random 6-patch triples
    rng = np.random.default_rng(20261018)
    n6, ntri = 6, 300
    zo = rng.integers(0, 2, (ntri, n6)).astype(np.int32)
    ym = (zo * rng.integers(0, 2, (ntri, n6))).astype(np.int32)          # y <= z_old mostly
    zn = np.maximum(ym, rng.integers(0, 2, (ntri, n6))).astype(np.int32)  # z_new >= y mostly
    flipmask = rng.random(ntri) < 0.15                                    # some impossible triples
    ym[flipmask, 0] = 1 - ym[flipmask, 0]
    pars = np.column_stack([rng.uniform(0.05, 1.3, ntri), rng.uniform(0.05, 2.0, ntri), rng.uniform(0.2, 8.0, ntri),
                            rng.uniform(0.1, 5.0, ntri), rng.uniform(150, 900, ntri)])   # e, c, K, Ksrc, dL
    a6, d6 = 1.0 / 400, 200.0
    ip = C.POINTER(C.c_int)
    res = np.zeros((ntri, 5))
    for i in range(ntri):
        e_, c_, K_, Ks_, dL_ = pars[i]
        M6 = O.ref_kernel_matrix(n6, a6, d6, source_d=dL_)
        Msq = np.ascontiguousarray(M6[:n6])
        A = [np.ascontiguousarray(v) for v in (zo[i], ym[i], zn[i])]
        res[i, 0] = R.ref_dieoff_pije(A[0].ctypes.data_as(ip), A[1].ctypes.data_as(ip), e_, K_, n6)
        res[i, 1] = R.ref_dieoff_pijc(A[1].ctypes.data_as(ip), A[2].ctypes.data_as(ip), c_, K_, Msq.ctypes.data_as(dp), n6)
        res[i, 2] = R.ref_loss_pije(A[0].ctypes.data_as(ip), A[1].ctypes.data_as(ip), e_, n6)
        res[i, 3] = R.ref_loss_pijc(A[1].ctypes.data_as(ip), A[2].ctypes.data_as(ip), c_, Msq.ctypes.data_as(dp), n6)
        res[i, 4] = R.ref_loss_pijcsource(A[1].ctypes.data_as(ip), A[2].ctypes.data_as(ip), c_, Ks_, M6.ctypes.data_as(dp), n6)
    g["var_zo"], g["var_y"], g["var_zn"], g["var_pars"], g["var_res"] = zo, ym, zn, pars, res
    g["var_geom"] = np.array([a6, d6])

    # ---- simpij: empirical one-step distribution from a fixed state (libc rand, fixed seed)
    n8 = 8
    z0 = np.array([0, 1, 1, 1, 1, 0, 1, 0], dtype=np.int32)
    Mf = O.ref_kernel_matrix(n8, 1.0 / 400, 100.0, source_d=500.0)
    e_, c_, K_, Ks_ = 0.6, 0.45, 1.5, 1.0
    R.ref_srand(12345)
    nsim = 10000
    acc = np.zeros(n8)
    new = np.zeros(n8, dtype=np.int32)
    for _ in range(nsim):
        R.ref_future_simpij(z0.ctypes.data_as(ip), new.ctypes.data_as(ip), e_, c_, K_, Ks_, Mf.ctypes.data_as(dp), n8)
        acc += new
    g["simpij_z0"], g["simpij_pars"], g["simpij_freq"], g["simpij_nsim"] = z0, np.array([e_, c_, K_, Ks_, 1.0 / 400, 100.0, 500.0]), acc / nsim, np.array(nsim)

    # ---- future module: the program itself, 6 runs of 10,000 simulations each (rand() is time-seeded)
    import shutil, time
    shutil.copy(EXAMPLE, HERE / "occupancies_example.txt")          # the bundled 7-line input (data, read by the driver tests)
    for tag, extra in (("nomgmt", []), ("source", ["-S", "1", "-s", "500"])):
        runs = []
        for r in range(6):
            run("MIDASPOM_future.out", ["-a", "50", "-m", "400", "-d", "100", "-i", EXAMPLE, "-q", str(tmp / "p.txt"), "-o", str(tmp / "f.txt")] + extra)
            runs.append([int(v) for v in (tmp / "f.txt").read_text().split()])
            time.sleep(1.1)                                          # srand(time(NULL)) has one-second resolution
        g[f"future_{tag}_runs"] = np.array(runs)

    np.savez_compressed(HERE / "golden.npz", **g)
    print("wrote", HERE / "golden.npz", {k: np.shape(v) for k, v in g.items()})


if __name__ == "__main__":
    main()
