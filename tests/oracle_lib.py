"""ctypes bindings for the TEST-ONLY oracle (oracle/libspom_oracle.so) and, when it was built by hand,
the reference harness (oracle/_ref/libmidaspom_ref.so, the reference's own functions compiled from its
sources by `make -C oracle ref REF=<reference checkout>`).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
ORACLE_DIR = ROOT / "oracle"
ORACLE_SO = ORACLE_DIR / "libspom_oracle.so"
REF_SO = ORACLE_DIR / "_ref" / "libmidaspom_ref.so"
REF_BIN = ORACLE_DIR / "_ref"

NDRAW = 11
NLSIG = 8
GEOM_LINEAR, GEOM_COORDS, GEOM_DENSE = 0, 1, 2

_dp = C.POINTER(C.c_double)
_u8p = C.POINTER(C.c_uint8)
_i8p = C.POINTER(C.c_int8)


class SpomModel(C.Structure):
    _fields_ = [("n", C.c_int32), ("T", C.c_int32), ("geom", C.c_int32), ("detect", C.c_int32),
                ("spacing", C.c_double), ("prior_occ", C.c_double),
                ("px", _dp), ("py", _dp), ("dist", _dp), ("area", _dp), ("src_unit", _dp),
                ("obs", _i8p), ("era", _u8p), ("blk_nx", C.c_int32), ("blk_ny", C.c_int32), ("blk_k", C.c_int32)]


class SpomParams(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("e", "c", "alpha", "b", "p", "K", "Ksrc", "dsrc")]


class SpomSamplerCfg(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("e_min", "e_max", "c_min", "c_max", "alpha_min", "alpha_max",
                                          "b_min", "b_max", "p_min", "p_max", "K_min", "K_max", "Ksrc_min", "Ksrc_max",
                                          "dsrc_min", "dsrc_max")] + \
               [(k, C.c_int32) for k in ("sample_e", "sample_c", "sample_alpha", "sample_b", "sample_p",
                                         "n_e_steps", "n_c_steps", "n_adapt", "update_z", "update_y",
                                         "sample_K", "sample_Ksrc", "sample_dsrc", "n_v_steps")]


def build_oracle(force: bool = False) -> None:
    """Compile oracle/libspom_oracle.so (oracle/_ref is built by hand: make -C oracle ref REF=<reference checkout>)."""
    if force or not ORACLE_SO.exists() or ORACLE_SO.stat().st_mtime < (ORACLE_DIR / "spom_oracle.c").stat().st_mtime:
        subprocess.run(["make", "-C", str(ORACLE_DIR), "oracle"], check=True, capture_output=True)


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build_oracle()
        L = C.CDLL(str(ORACLE_SO))
        mp, pp, cp = C.POINTER(SpomModel), C.POINTER(SpomParams), C.POINTER(SpomSamplerCfg)
        u32p = C.POINTER(C.c_uint32)
        L.spom_philox4x32.argtypes = [u32p, u32p, u32p]
        L.spom_rng.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, u32p]
        L.spom_u01.argtypes = [C.c_uint32]; L.spom_u01.restype = C.c_double
        L.spom_weight.argtypes = [mp, C.c_double, C.c_double, C.c_int, C.c_int]; L.spom_weight.restype = C.c_double
        L.spom_connectivity.argtypes = [mp, C.c_double, C.c_double, _u8p, _dp]
        L.spom_connectivity_targets.argtypes = [mp, C.c_double, C.c_double, _u8p, C.POINTER(C.c_int32), C.c_int, _dp]
        L.spom_source_term.argtypes = [mp, pp, C.c_int]; L.spom_source_term.restype = C.c_double
        L.spom_transition_prob.argtypes = [mp, pp, C.c_int, _u8p, _u8p, _u8p, _dp, _dp]
        L.spom_transition_prob.restype = C.c_double
        L.spom_loglik.argtypes = [mp, pp, _u8p, _u8p, _dp, _dp]; L.spom_loglik.restype = C.c_double
        L.spom_marginal_loglik.argtypes = [mp, pp]; L.spom_marginal_loglik.restype = C.c_double
        L.spom_flip_delta_bruteforce.argtypes = [mp, pp, _u8p, _u8p, C.c_int, C.c_int]
        L.spom_flip_delta_bruteforce.restype = C.c_double
        L.spom_flip_delta.argtypes = [mp, pp, _u8p, _u8p, _dp, C.c_int, C.c_int]
        L.spom_flip_delta.restype = C.c_double
        L.spom_init_chain.argtypes = [mp, cp, C.c_uint64, C.c_uint32, C.c_int, pp, _dp, _u8p, _u8p, _dp]
        L.spom_refresh_S.argtypes = [mp, pp, _u8p, _dp]
        L.spom_scan_order.argtypes = [mp, C.POINTER(C.c_int32)]
        L.spom_sweep.argtypes = [mp, cp, C.c_uint64, C.c_uint32, C.c_uint32, pp, _dp, _u8p, _u8p, _dp, _dp, C.c_int64, _dp]
        L.spom_sweep.restype = C.c_int64
        L.spom_sweep_chains.argtypes = [mp, cp, C.c_uint64, C.c_int, C.c_uint32, C.c_uint32, pp, _dp, _u8p, _u8p,
                                        _dp, _dp, C.c_int64, C.c_int, _dp]
        L.spom_sweep_chains.restype = C.c_int64
        L.spom_max_threads.restype = C.c_int
        L.spom_simulate.argtypes = [mp, pp, C.c_uint64, C.c_uint32, _u8p, C.c_int, _u8p]
        _lib = L
    return _lib


def _ptr(a, ty):
    return None if a is None else a.ctypes.data_as(ty)


class Model:
    """Owns the numpy arrays behind a spom_model struct."""

    def __init__(self, obs, geom=GEOM_LINEAR, spacing=100.0, prior_occ=0.5, detect=0, px=None, py=None,
                 dist=None, area=None, src_unit=None, era=None, scan_blocks=(1, 1, 1)):
        self.obs = np.ascontiguousarray(obs, dtype=np.int8)
        self.T, self.n = self.obs.shape
        f = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
        self.px, self.py, self.dist, self.area, self.src_unit = f(px), f(py), f(dist), f(area), f(src_unit)
        self.era = None if era is None else np.ascontiguousarray(era, dtype=np.uint8)
        self.geom, self.spacing, self.prior_occ, self.detect = geom, float(spacing), float(prior_occ), int(detect)
        self.c = SpomModel(self.n, self.T, geom, self.detect, self.spacing, self.prior_occ,
                           _ptr(self.px, _dp), _ptr(self.py, _dp), _ptr(self.dist, _dp), _ptr(self.area, _dp),
                           _ptr(self.src_unit, _dp), _ptr(self.obs, _i8p), _ptr(self.era, _u8p),
                           int(scan_blocks[0]), int(scan_blocks[1]), int(scan_blocks[2]))

    def ref(self):
        return C.byref(self.c)


def params(e=0.5, c=0.5, alpha=1.0 / 400, b=0.0, p=1.0, K=1.0, Ksrc=0.0, dsrc=0.0) -> SpomParams:
    return SpomParams(e, c, alpha, b, p, K, Ksrc, dsrc)


def sampler_cfg(**kw) -> SpomSamplerCfg:
    d = dict(e_min=0.0, e_max=1.0, c_min=0.0, c_max=1.0, alpha_min=1e-4, alpha_max=1e-1, b_min=0.0, b_max=2.0,
             p_min=0.0, p_max=1.0, K_min=0.1, K_max=100.0, Ksrc_min=0.1, Ksrc_max=100.0, dsrc_min=200.0, dsrc_max=4000.0,
             sample_e=1, sample_c=1, sample_alpha=0, sample_b=0, sample_p=0,
             n_e_steps=4, n_c_steps=1, n_adapt=200, update_z=1, update_y=1, sample_K=0, sample_Ksrc=0, sample_dsrc=0, n_v_steps=2)
    d.update(kw)
    return SpomSamplerCfg(**d)


def u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


def connectivity(m: Model, alpha, b, y_row):
    y_row = u8(y_row)
    S = np.zeros(m.n)
    lib().spom_connectivity(m.ref(), alpha, b, _ptr(y_row, _u8p), _ptr(S, _dp))
    return S


def connectivity_targets(m: Model, alpha, b, y_row, targets):
    """S of the listed target patches only (same sum, same order as spom_connectivity)."""
    y_row = u8(y_row)
    targets = np.ascontiguousarray(targets, dtype=np.int32)
    S = np.zeros(len(targets))
    lib().spom_connectivity_targets(m.ref(), alpha, b, _ptr(y_row, _u8p), targets.ctypes.data_as(C.POINTER(C.c_int32)),
                                    len(targets), _ptr(S, _dp))
    return S


def scan_order(m: Model):
    """Visiting order of the y scan (slot -> patch): Morton order of planar coordinates, else index order."""
    out = np.zeros(m.n, dtype=np.int32)
    lib().spom_scan_order(m.ref(), out.ctypes.data_as(C.POINTER(C.c_int32)))
    return out


def transition_prob(m: Model, par: SpomParams, pre, z_old, y_mid, z_new):
    pe, pc = C.c_double(), C.c_double()
    z_old, y_mid, z_new = u8(z_old), u8(y_mid), u8(z_new)
    tot = lib().spom_transition_prob(m.ref(), C.byref(par), int(pre), _ptr(z_old, _u8p), _ptr(y_mid, _u8p),
                                     _ptr(z_new, _u8p), C.byref(pe), C.byref(pc))
    return tot, pe.value, pc.value


def loglik(m: Model, par: SpomParams, z, y, want_S=False):
    z, y = u8(z), u8(y)
    parts = np.zeros(4)
    S = np.zeros((m.T - 1, m.n)) if want_S else None
    tot = lib().spom_loglik(m.ref(), C.byref(par), _ptr(z, _u8p), _ptr(y, _u8p), _ptr(parts, _dp), _ptr(S, _dp))
    return (tot, parts, S) if want_S else (tot, parts)


def marginal_loglik(m: Model, par: SpomParams) -> float:
    return lib().spom_marginal_loglik(m.ref(), C.byref(par))


def flip_delta(m: Model, par: SpomParams, z, y, S, t, k) -> float:
    z, y, S = u8(z), u8(y), np.ascontiguousarray(S, dtype=np.float64)
    return lib().spom_flip_delta(m.ref(), C.byref(par), _ptr(z, _u8p), _ptr(y, _u8p), _ptr(S, _dp), t, k)


def flip_delta_bruteforce(m: Model, par: SpomParams, z, y, t, k) -> float:
    z, y = u8(z), u8(y)
    return lib().spom_flip_delta_bruteforce(m.ref(), C.byref(par), _ptr(z, _u8p), _ptr(y, _u8p), t, k)


def simulate(m: Model, par: SpomParams, seed, sim_id, z0, nyears):
    z0 = u8(z0)
    out = np.zeros((nyears + 1, m.n), dtype=np.uint8)
    lib().spom_simulate(m.ref(), C.byref(par), seed, sim_id, _ptr(z0, _u8p), nyears, _ptr(out, _u8p))
    return out


class Chains:
    """State of `nchains` CPU chains (the oracle twin of midaspom_b200.Engine's device state)."""

    def __init__(self, m: Model, cfg: SpomSamplerCfg, nchains: int, seed: int, par0, disperse=False, chain0=0):
        self.m, self.cfg, self.nchains, self.seed, self.chain0 = m, cfg, nchains, seed, chain0
        self.par = (SpomParams * nchains)()
        for i in range(nchains):
            src = par0[i] if isinstance(par0, (list, tuple)) else par0
            C.memmove(C.byref(self.par[i]), C.byref(src), C.sizeof(SpomParams))
        self.lsig = np.zeros((nchains, NLSIG))
        self.z = np.zeros((nchains, m.T, m.n), dtype=np.uint8)
        self.y = np.zeros((nchains, m.T - 1, m.n), dtype=np.uint8)
        self.S = np.zeros((nchains, m.T - 1, m.n))
        self.draws = np.zeros((nchains, NDRAW))
        self.sweep = 0
        for i in range(nchains):
            lib().spom_init_chain(m.ref(), C.byref(cfg), seed, chain0 + i, int(disperse), C.byref(self.par[i]),
                                  _ptr(self.lsig[i], _dp), _ptr(self.z[i], _u8p), _ptr(self.y[i], _u8p),
                                  _ptr(self.S[i], _dp))

    def run(self, nsweeps: int, y_flip_limit: int = -1, nthreads: int = 0):
        out = np.zeros((nsweeps, self.nchains, NDRAW))
        visited = 0
        self.phase_s = np.zeros((self.nchains, 2))           # last sweep: [everything else, y scan] seconds per chain
        for s in range(nsweeps):
            visited += lib().spom_sweep_chains(self.m.ref(), C.byref(self.cfg), self.seed, self.nchains, self.chain0,
                                               self.sweep, self.par, _ptr(self.lsig, _dp), _ptr(self.z, _u8p),
                                               _ptr(self.y, _u8p), _ptr(self.S, _dp), _ptr(self.draws, _dp),
                                               y_flip_limit, nthreads, _ptr(self.phase_s, _dp))
            out[s] = self.draws
            self.sweep += 1
        self.visited = visited
        return out

    def params_array(self):
        return np.array([[getattr(self.par[i], k) for k in ("e", "c", "alpha", "b", "p", "K", "Ksrc", "dsrc")]
                         for i in range(self.nchains)])


# ----------------------------------------------------------------------------- reference harness
_ref = None


def have_ref() -> bool:
    return REF_SO.exists()


def ref() -> C.CDLL:
    """The reference's own functions (compPePc, pije, pijc, pijcsource, simpij) -- oracle/_ref."""
    global _ref
    if _ref is None:
        R = C.CDLL(str(REF_SO))
        u32p = C.POINTER(C.c_uint32)
        ip = C.POINTER(C.c_int)
        sig = [_dp, _dp, u32p, u32p, C.c_double, _dp, _dp, C.c_uint, C.c_uint, C.c_uint, C.c_uint]
        R.ref_base_compPePc.argtypes = sig
        R.ref_mpi_compPePc.argtypes = sig
        R.ref_dieoff_pije.argtypes = [ip, ip, C.c_double, C.c_double, C.c_int]; R.ref_dieoff_pije.restype = C.c_double
        R.ref_dieoff_pijc.argtypes = [ip, ip, C.c_double, C.c_double, _dp, C.c_int]; R.ref_dieoff_pijc.restype = C.c_double
        R.ref_loss_pije.argtypes = [ip, ip, C.c_double, C.c_int]; R.ref_loss_pije.restype = C.c_double
        R.ref_loss_pijc.argtypes = [ip, ip, C.c_double, _dp, C.c_int]; R.ref_loss_pijc.restype = C.c_double
        R.ref_loss_pijcsource.argtypes = [ip, ip, C.c_double, C.c_double, _dp, C.c_int]
        R.ref_loss_pijcsource.restype = C.c_double
        R.ref_future_simpij.argtypes = [ip, ip, C.c_double, C.c_double, C.c_double, C.c_double, _dp, C.c_int]
        R.ref_future_simpij.restype = C.c_int
        R.ref_dieoff_matpow.argtypes = [_dp, C.c_int, C.c_int, _dp]
        R.ref_srand.argtypes = [C.c_uint]
        _ref = R
    return _ref


def ref_kernel_matrix(n, a, d, source_d=None):
    """M as the reference builds it (main_MIDASPOM.c:180-188); optional source row n (loss.c:365)."""
    rows = n + (1 if source_d is not None else 0)
    M = np.zeros((rows, n))
    for i in range(n):
        for j in range(i + 1, n):
            M[i, j] = M[j, i] = np.exp(-a * (j - i) * d)
    if source_d is not None:
        for j in range(n):
            M[n, j] = np.exp(-a * (j + 1) * source_d)
    return M


def parse_occupancy_stream(path) -> np.ndarray:
    """The reference's parser (main_MIDASPOM.c:138-167): n = 1 + separators on line 1, tmax = '\\n'
    count, then integers are consumed in STREAM order regardless of line breaks."""
    raw = Path(path).read_bytes()
    first = raw.split(b"\n", 1)[0]
    n = 1 + sum(1 for ch in first if ch in b" \t")
    tmax = raw.count(b"\n")
    vals = [int(v) for v in raw.split()]
    return np.array(vals[: n * tmax], dtype=np.int8).reshape(tmax, n)


def run_reference_binary(name: str, args: list[str], cwd=None) -> str:
    exe = REF_BIN / name
    env = dict(os.environ)
    return subprocess.run([str(exe)] + args, check=True, capture_output=True, text=True, cwd=cwd, env=env).stdout
