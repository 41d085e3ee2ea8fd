"""ctypes mirror of include/libmidaspom_cuda.h.

``Engine`` wraps one ``mp_engine`` handle (one GPU).  Method names follow the C entry points
(``mp_connectivity`` -> ``Engine.connectivity`` ...); arguments are numpy host arrays, exactly the
flat buffers the C driver passes.  Every call raises ``MpError`` on a non-zero status; nothing here
computes on the CPU.
"""
from __future__ import annotations

import ctypes as C
import hashlib
from pathlib import Path

import numpy as np

from . import build as _build

FP32, FP64 = 0, 1
GEOM_LINEAR, GEOM_COORDS, GEOM_DENSE = 0, 1, 2
NDRAW, NLSIG, NPART = 11, 8, 4
PPC_STATS = ("detected", "colonised", "extinct")   # the MP_NPPC statistics of mp_ppc, in order
KERNEL_CATEGORIES = ("conn", "col", "sweep_y", "sweep_z", "small", "sim")
WORK_COUNTERS = ("scan_trips", "scan_exec", "scan_retired", "scan_commit", "scan_dense", "conn_exec", "conn_total", "gemm_tiles", "scan_blocks")
DRAW_FIELDS = ("e", "c", "alpha", "b", "p", "loglik", "n_y1", "n_z1", "K", "Ksrc", "dsrc")

# every symbol include/libmidaspom_cuda.h declares
ABI_SYMBOLS = (
    "mp_version", "mp_device_count", "mp_create", "mp_destroy", "mp_last_error",
    "mp_set_landscape_linear", "mp_set_landscape_coords", "mp_set_landscape_dense", "mp_set_source_units",
    "mp_set_observations", "mp_set_era", "mp_set_params", "mp_get_params", "mp_set_state", "mp_get_state",
    "mp_set_scales", "mp_get_scales", "mp_connectivity", "mp_get_connectivity", "mp_loglik", "mp_loglik_host",
    "mp_flip_delta", "mp_init_chains", "mp_set_sampler", "mp_sweep", "mp_synchronize", "mp_num_draws",
    "mp_get_draws", "mp_reset_draws", "mp_sweep_index", "mp_simulate", "mp_device_ptr", "mp_set_timing",
    "mp_get_timing", "mp_probe_peaks", "mp_get_stream", "mp_exact_posterior", "mp_exact_last_error", "mp_simulate_ensemble", "mp_exact_variant", "mp_set_shard", "mp_sweep_phase",
    "mp_get_scan_order", "mp_get_work_counters", "mp_get_scan_geometry", "mp_get_conn_path", "mp_set_scan_blocks",
    "mp_comm_unique_id", "mp_comm_init", "mp_comm_init_all", "mp_comm_destroy", "mp_comm_rank", "mp_comm_size", "mp_comm_last_error",
    "mp_gather_draws", "mp_gather_draws_all", "mp_sweep_sharded", "mp_sweep_sharded_all", "mp_forecast",
    "mp_set_summaries", "mp_get_summaries", "mp_set_waic", "mp_get_waic", "mp_ppc", "mp_capacity",
    "mp_set_sources", "mp_get_sources",
)


class MpError(RuntimeError):
    pass


class MpConfig(C.Structure):
    _fields_ = [("n_patches", C.c_int32), ("n_years", C.c_int32), ("n_chains", C.c_int32), ("chain_offset", C.c_int32),
                ("precision", C.c_int32), ("device", C.c_int32), ("detect", C.c_int32), ("max_draws", C.c_int32),
                ("seed", C.c_uint64), ("prior_occ", C.c_double)]


class MpParams(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("e", "c", "alpha", "b", "p", "K", "Ksrc", "dsrc")]


class MpSamplerConfig(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("e_min", "e_max", "c_min", "c_max", "alpha_min", "alpha_max",
                                          "b_min", "b_max", "p_min", "p_max", "K_min", "K_max", "Ksrc_min", "Ksrc_max",
                                          "dsrc_min", "dsrc_max")] + \
               [(k, C.c_int32) for k in ("sample_e", "sample_c", "sample_alpha", "sample_b", "sample_p",
                                         "n_e_steps", "n_c_steps", "n_adapt", "update_z", "update_y",
                                         "sample_K", "sample_Ksrc", "sample_dsrc", "n_v_steps")]


PARAM_FIELDS = ("e", "c", "alpha", "b", "p", "K", "Ksrc", "dsrc")
PARAM_DEFAULTS = dict(e=0.5, c=0.5, alpha=1.0 / 400.0, b=0.0, p=1.0, K=1.0, Ksrc=0.0, dsrc=0.0)


def sampler_config(**kw) -> MpSamplerConfig:
    d = dict(e_min=0.0, e_max=1.0, c_min=0.0, c_max=1.0, alpha_min=1e-4, alpha_max=1e-1, b_min=0.0, b_max=2.0,
             p_min=0.0, p_max=1.0, K_min=0.1, K_max=100.0, Ksrc_min=0.1, Ksrc_max=100.0, dsrc_min=200.0, dsrc_max=4000.0,
             sample_e=1, sample_c=1, sample_alpha=0, sample_b=0, sample_p=0,
             n_e_steps=4, n_c_steps=1, n_adapt=200, update_z=1, update_y=1, sample_K=0, sample_Ksrc=0, sample_dsrc=0, n_v_steps=2)
    d.update(kw)
    return MpSamplerConfig(**d)


_lib = None


def load_library(build_if_missing: bool = True) -> C.CDLL:
    """dlopen lib/libmidaspom_cuda.so (building it with nvcc if needed). Fails loudly if it cannot."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if build_if_missing and _build.stale():
        path = _build.build()
    if not Path(path).exists():
        raise MpError(f"{path} is missing: build it with `python -m midaspom_b200.build` (there is no CPU fallback)")
    L = C.CDLL(str(path))
    vp, dp, u8p, i8p = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_uint8), C.POINTER(C.c_int8)
    pp, scp = C.POINTER(MpParams), C.POINTER(MpSamplerConfig)
    L.mp_version.restype = C.c_char_p
    L.mp_device_count.restype = C.c_int
    L.mp_create.argtypes = [C.POINTER(MpConfig), C.POINTER(vp)]
    L.mp_destroy.argtypes = [vp]
    L.mp_last_error.argtypes = [vp]; L.mp_last_error.restype = C.c_char_p
    L.mp_set_landscape_linear.argtypes = [vp, C.c_double, dp]
    L.mp_set_landscape_coords.argtypes = [vp, dp, dp, dp]
    L.mp_set_landscape_dense.argtypes = [vp, dp, dp]
    L.mp_set_source_units.argtypes = [vp, dp]
    L.mp_get_scan_order.argtypes = [vp, C.POINTER(C.c_int32)]
    L.mp_set_scan_blocks.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_double]
    L.mp_comm_unique_id.argtypes = [C.c_void_p]
    L.mp_comm_init.argtypes = [vp, C.c_int, C.c_int, C.c_void_p]
    L.mp_comm_init_all.argtypes = [C.POINTER(vp), C.c_int]
    L.mp_comm_destroy.argtypes = [vp]
    L.mp_comm_rank.argtypes = [vp]; L.mp_comm_size.argtypes = [vp]
    L.mp_comm_last_error.restype = C.c_char_p
    L.mp_gather_draws.argtypes = [vp, C.c_int, C.c_int, dp]
    L.mp_gather_draws_all.argtypes = [C.POINTER(vp), C.c_int, C.c_int, C.c_int, dp]
    L.mp_sweep_sharded.argtypes = [vp, C.c_int]
    L.mp_sweep_sharded_all.argtypes = [C.POINTER(vp), C.c_int, C.c_int]
    L.mp_set_observations.argtypes = [vp, i8p]
    L.mp_set_era.argtypes = [vp, u8p]
    L.mp_set_params.argtypes = [vp, pp]; L.mp_get_params.argtypes = [vp, pp]
    L.mp_set_state.argtypes = [vp, u8p, u8p]; L.mp_get_state.argtypes = [vp, u8p, u8p]
    L.mp_set_scales.argtypes = [vp, dp]; L.mp_get_scales.argtypes = [vp, dp]
    L.mp_connectivity.argtypes = [vp, dp]; L.mp_get_connectivity.argtypes = [vp, dp]
    L.mp_loglik.argtypes = [vp, dp, dp]
    L.mp_loglik_host.argtypes = [vp, pp, u8p, u8p, dp, dp]
    L.mp_flip_delta.argtypes = [vp, C.c_int, C.c_int, C.c_int, dp]
    L.mp_init_chains.argtypes = [vp, scp, C.c_int]
    L.mp_set_sampler.argtypes = [vp, scp]
    L.mp_sweep.argtypes = [vp, C.c_int]
    L.mp_synchronize.argtypes = [vp]
    L.mp_set_shard.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int]
    L.mp_sweep_phase.argtypes = [vp, C.c_int, C.POINTER(C.c_int)]
    L.mp_num_draws.argtypes = [vp]; L.mp_reset_draws.argtypes = [vp]; L.mp_sweep_index.argtypes = [vp]
    L.mp_get_draws.argtypes = [vp, C.c_int, C.c_int, dp]
    L.mp_simulate.argtypes = [vp, pp, u8p, C.c_int, C.c_int, C.c_uint64, C.c_int, u8p, C.POINTER(C.c_int32)]
    L.mp_simulate_ensemble.argtypes = [vp, pp, u8p, C.c_int, C.c_int, C.c_uint64, C.c_int, u8p, C.POINTER(C.c_int32)]
    L.mp_forecast.argtypes = [vp, C.c_int, C.c_int, C.c_uint64, dp, C.POINTER(C.c_int32), C.POINTER(C.c_uint32)]
    L.mp_ppc.argtypes = [vp, C.c_int, C.c_uint64, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_uint32),
                         C.POINTER(C.c_uint32)]
    L.mp_capacity.argtypes = [vp, C.c_int, pp, u8p, C.c_double, C.c_int, dp, C.POINTER(C.c_int32), dp, dp]
    L.mp_set_summaries.argtypes = [vp, C.c_int, C.c_int]
    L.mp_get_summaries.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_uint32), dp, C.POINTER(C.c_uint32), dp, C.c_int]
    L.mp_set_waic.argtypes = [vp, C.c_int, C.c_int]
    L.mp_get_waic.argtypes = [vp, C.POINTER(C.c_int64), dp, dp, dp, C.c_int]
    L.mp_set_sources.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_double]
    L.mp_get_sources.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_uint64), dp, dp, dp, C.c_int]
    L.mp_device_ptr.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(C.c_size_t)]
    L.mp_get_stream.argtypes = [vp, C.POINTER(vp)]
    L.mp_set_timing.argtypes = [vp, C.c_int]
    L.mp_get_timing.argtypes = [vp, dp, C.POINTER(C.c_int64), C.c_int]
    L.mp_probe_peaks.argtypes = [vp, dp]
    L.mp_get_work_counters.argtypes = [vp, C.POINTER(C.c_uint64), C.c_int]
    L.mp_get_scan_geometry.argtypes = [vp, C.POINTER(C.c_int)]
    L.mp_get_conn_path.argtypes = [vp]
    L.mp_exact_posterior.argtypes = [C.c_int, i8p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int,
                                     C.c_double, C.c_double, dp, dp, C.POINTER(C.c_int)]
    L.mp_exact_last_error.restype = C.c_char_p
    L.mp_exact_variant.argtypes = [C.c_int, C.c_int, i8p, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                   C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_double, C.c_double, dp]
    _lib = L
    return L


def _p(a, ty):
    return None if a is None else a.ctypes.data_as(ty)


_dp, _u8p, _i8p = C.POINTER(C.c_double), C.POINTER(C.c_uint8), C.POINTER(C.c_int8)


class Engine:
    """One mp_engine handle: N patches x T years x C chains resident on one B200."""

    def __init__(self, n_patches, n_years, n_chains=1, precision=FP64, device=0, seed=1, prior_occ=0.5, detect=0,
                 chain_offset=0, max_draws=0):
        self.lib = load_library()
        self.cfg = MpConfig(n_patches, n_years, n_chains, chain_offset, precision, device, detect, max_draws, seed, prior_occ)
        self.h = C.c_void_p()
        rc = self.lib.mp_create(C.byref(self.cfg), C.byref(self.h))
        if rc != 0:
            msg = self.lib.mp_last_error(None).decode()
            self.h = None
            raise MpError(f"mp_create failed ({rc}): {msg}")
        self.N, self.T, self.C = n_patches, n_years, n_chains
        self._landscape_key = b""

    # -- lifetime
    def close(self):
        if getattr(self, "h", None):
            self.lib.mp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc, what):
        if rc != 0:
            raise MpError(f"{what} failed ({rc}): {self.lib.mp_last_error(self.h).decode()}")

    # -- landscape / data
    @staticmethod
    def _f64(a, shape=None):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=np.float64)
        if shape is not None and a.shape != shape:
            raise ValueError(f"expected shape {shape}, got {a.shape}")
        return a

    def _remember_landscape(self, *parts):
        """Fingerprint of the landscape as uploaded (capacity results carry it so that results of different landscapes are not
        pooled)."""
        h = hashlib.sha256()
        for a in parts:
            h.update(b"-" if a is None else np.ascontiguousarray(a, dtype=np.float64).tobytes())
        self._landscape_key = h.digest()

    def set_landscape_linear(self, spacing, area=None):
        area = self._f64(area, (self.N,))
        self._remember_landscape(np.array([0.0, float(spacing)]), area)
        self._ck(self.lib.mp_set_landscape_linear(self.h, float(spacing), _p(area, _dp)), "mp_set_landscape_linear")

    def set_landscape_coords(self, x, y, area=None):
        x, y, area = self._f64(x, (self.N,)), self._f64(y, (self.N,)), self._f64(area, (self.N,))
        self._remember_landscape(np.array([1.0]), x, y, area)
        self._ck(self.lib.mp_set_landscape_coords(self.h, _p(x, _dp), _p(y, _dp), _p(area, _dp)), "mp_set_landscape_coords")

    def set_landscape_dense(self, dist, area=None):
        dist, area = self._f64(dist, (self.N, self.N)), self._f64(area, (self.N,))
        self._remember_landscape(np.array([2.0]), dist, area)
        self._ck(self.lib.mp_set_landscape_dense(self.h, _p(dist, _dp), _p(area, _dp)), "mp_set_landscape_dense")

    def set_source_units(self, src_unit=None):
        src_unit = self._f64(src_unit, (self.N,))
        self._ck(self.lib.mp_set_source_units(self.h, _p(src_unit, _dp)), "mp_set_source_units")

    # ---- several GPUs behind the C ABI (NCCL inside the library)
    COMM_ID_BYTES = 128

    @staticmethod
    def _prefer_bundled_nccl():
        """Point the library at the NCCL that PyTorch bundles (MP_NCCL_LIB) unless the caller chose one: the process may
        import torch later, and two different libnccl.so.2 cannot live in one process."""
        import importlib.util
        import os
        if os.environ.get("MP_NCCL_LIB"):
            return
        spec = importlib.util.find_spec("nvidia.nccl")
        for root in (spec.submodule_search_locations if spec and spec.submodule_search_locations else []):
            cand = Path(root) / "lib" / "libnccl.so.2"
            if cand.exists():
                os.environ["MP_NCCL_LIB"] = str(cand)
                return

    @staticmethod
    def comm_unique_id() -> bytes:
        """mp_comm_unique_id: the 128 bytes rank 0 hands to every rank of a communicator."""
        Engine._prefer_bundled_nccl()
        buf = C.create_string_buffer(Engine.COMM_ID_BYTES)
        rc = load_library().mp_comm_unique_id(buf)
        if rc != 0:
            raise MpError(f"mp_comm_unique_id failed ({rc}): {load_library().mp_comm_last_error().decode()}")
        return buf.raw

    def comm_init(self, nranks: int, rank: int, unique_id: bytes):
        Engine._prefer_bundled_nccl()
        buf = C.create_string_buffer(bytes(unique_id), Engine.COMM_ID_BYTES)
        self._ck(self.lib.mp_comm_init(self.h, int(nranks), int(rank), buf), "mp_comm_init")

    @staticmethod
    def comm_init_all(engines):
        """One process driving one engine per device: a communicator over all of them (mp_comm_init_all)."""
        Engine._prefer_bundled_nccl()
        arr = (C.c_void_p * len(engines))(*[e.h for e in engines])
        engines[0]._ck(engines[0].lib.mp_comm_init_all(arr, len(engines)), "mp_comm_init_all")

    def comm_destroy(self):
        self._ck(self.lib.mp_comm_destroy(self.h), "mp_comm_destroy")

    def gather_draws(self, first=0, count=None) -> np.ndarray:
        """mp_gather_draws: every rank's draws -> (ranks, sweeps, chains, NDRAW), the same on every rank."""
        count = self.num_draws() - first if count is None else count
        world = max(1, self.lib.mp_comm_size(self.h))
        out = np.empty((world, count, self.C, NDRAW), dtype=np.float64)
        self._ck(self.lib.mp_gather_draws(self.h, int(first), int(count), _p(out, _dp)), "mp_gather_draws")
        return out

    @staticmethod
    def gather_draws_all(engines, first=0, count=None) -> np.ndarray:
        """mp_gather_draws_all: one process driving all engines of the communicator -> (engines, sweeps, chains, NDRAW)."""
        e0 = engines[0]
        count = e0.num_draws() - first if count is None else count
        out = np.empty((len(engines), count, e0.C, NDRAW), dtype=np.float64)
        arr = (C.c_void_p * len(engines))(*[e.h for e in engines])
        e0._ck(e0.lib.mp_gather_draws_all(arr, len(engines), int(first), int(count), _p(out, _dp)), "mp_gather_draws_all")
        return out

    def sweep_sharded(self, nsweeps=1):
        """mp_sweep_sharded: sweeps of the chains replicated on every rank of the communicator (asynchronous)."""
        self._ck(self.lib.mp_sweep_sharded(self.h, int(nsweeps)), "mp_sweep_sharded")

    @staticmethod
    def sweep_sharded_all(engines, nsweeps=1):
        arr = (C.c_void_p * len(engines))(*[e.h for e in engines])
        engines[0]._ck(engines[0].lib.mp_sweep_sharded_all(arr, len(engines), int(nsweeps)), "mp_sweep_sharded_all")

    def set_scan_blocks(self, nx: int, ny: int, k: int, halo: float):
        """Block grid of the y scan (mp_set_scan_blocks): nx x ny cells, k x k colours, targets within `halo` of a cell."""
        self._ck(self.lib.mp_set_scan_blocks(self.h, int(nx), int(ny), int(k), float(halo)), "mp_set_scan_blocks")

    def set_scan_blocks_auto(self, px, py, alpha, s_min, area_pow_max=1.0, k=4, margin=1.15):
        """Choose the finest grid the halo allows and install it.  The halo is the distance at which the largest dispersal
        weight (area_pow_max = max_k A_k^b) falls below 2^-36 of the smallest connectivity s_min, times `margin` so that
        the per-sweep validity check keeps holding while alpha and S move.  Returns (nx, ny, k, halo); (1, 1, 1, 0) when the
        landscape is too small for more than one block."""
        halo = margin * (36.0 * np.log(2.0) + np.log(max(area_pow_max, 1e-300) / max(s_min, 1e-300))) / float(alpha)
        ex, ey = float(np.ptp(px)), float(np.ptp(py))
        nx = max(1, int(np.floor((k - 1) * ex / (2.0 * halo) * 0.999)))
        ny = max(1, int(np.floor((k - 1) * ey / (2.0 * halo) * 0.999)))
        if nx * ny <= 1 or not np.isfinite(halo):
            self.set_scan_blocks(1, 1, 1, 0.0)
            return (1, 1, 1, 0.0)
        self.set_scan_blocks(nx, ny, k, halo)
        return (nx, ny, k, halo)

    def scan_order(self) -> np.ndarray:
        """Visiting order of the y scan (slot -> patch); Morton order for planar landscapes."""
        out = np.zeros(self.N, dtype=np.int32)
        self._ck(self.lib.mp_get_scan_order(self.h, out.ctypes.data_as(C.POINTER(C.c_int32))), "mp_get_scan_order")
        return out

    def set_observations(self, obs):
        obs = np.ascontiguousarray(obs, dtype=np.int8)
        if obs.shape != (self.T, self.N):
            raise ValueError(f"obs must be {(self.T, self.N)}")
        self._ck(self.lib.mp_set_observations(self.h, _p(obs, _i8p)), "mp_set_observations")

    def set_era(self, era=None):
        era = None if era is None else np.ascontiguousarray(era, dtype=np.uint8)
        if era is not None and era.shape != (self.T - 1,):
            raise ValueError("era must have T-1 flags")
        self._ck(self.lib.mp_set_era(self.h, _p(era, _u8p)), "mp_set_era")

    # -- chain state
    def _params_array(self, params):
        arr = (MpParams * self.C)()
        if isinstance(params, dict):
            params = [params] * self.C
        if len(params) != self.C:
            raise ValueError("need one parameter set per chain")
        for i, p in enumerate(params):
            d = dict(PARAM_DEFAULTS)
            if isinstance(p, dict):
                d.update(p)
            else:
                d.update({k: getattr(p, k) for k in PARAM_FIELDS})
            arr[i] = MpParams(*[float(d[k]) for k in PARAM_FIELDS])
        return arr

    def set_params(self, params):
        self._ck(self.lib.mp_set_params(self.h, self._params_array(params)), "mp_set_params")

    def get_params(self):
        arr = (MpParams * self.C)()
        self._ck(self.lib.mp_get_params(self.h, arr), "mp_get_params")
        return [{k: getattr(arr[i], k) for k in PARAM_FIELDS} for i in range(self.C)]

    def set_state(self, z, y):
        z = np.ascontiguousarray(z, dtype=np.uint8).reshape(self.C, self.T, self.N)
        y = np.ascontiguousarray(y, dtype=np.uint8).reshape(self.C, self.T - 1, self.N)
        self._ck(self.lib.mp_set_state(self.h, _p(z, _u8p), _p(y, _u8p)), "mp_set_state")

    def get_state(self):
        z = np.zeros((self.C, self.T, self.N), dtype=np.uint8)
        y = np.zeros((self.C, self.T - 1, self.N), dtype=np.uint8)
        self._ck(self.lib.mp_get_state(self.h, _p(z, _u8p), _p(y, _u8p)), "mp_get_state")
        return z, y

    def set_scales(self, lsig):
        lsig = np.ascontiguousarray(lsig, dtype=np.float64).reshape(self.C, NLSIG)
        self._ck(self.lib.mp_set_scales(self.h, _p(lsig, _dp)), "mp_set_scales")

    def get_scales(self):
        lsig = np.zeros((self.C, NLSIG))
        self._ck(self.lib.mp_get_scales(self.h, _p(lsig, _dp)), "mp_get_scales")
        return lsig

    # -- likelihood
    def connectivity(self, fetch=True):
        S = np.zeros((self.C, self.T - 1, self.N)) if fetch else None
        self._ck(self.lib.mp_connectivity(self.h, _p(S, _dp)), "mp_connectivity")
        return S

    def get_connectivity(self):
        S = np.zeros((self.C, self.T - 1, self.N))
        self._ck(self.lib.mp_get_connectivity(self.h, _p(S, _dp)), "mp_get_connectivity")
        return S

    def loglik(self):
        ll, parts = np.zeros(self.C), np.zeros((self.C, NPART))
        self._ck(self.lib.mp_loglik(self.h, _p(ll, _dp), _p(parts, _dp)), "mp_loglik")
        return ll, parts

    def loglik_host(self, params, z, y):
        z = np.ascontiguousarray(z, dtype=np.uint8).reshape(self.C, self.T, self.N)
        y = np.ascontiguousarray(y, dtype=np.uint8).reshape(self.C, self.T - 1, self.N)
        ll, parts = np.zeros(self.C), np.zeros((self.C, NPART))
        self._ck(self.lib.mp_loglik_host(self.h, self._params_array(params), _p(z, _u8p), _p(y, _u8p), _p(ll, _dp),
                                         _p(parts, _dp)), "mp_loglik_host")
        return ll, parts

    def flip_delta(self, chain, t, k):
        out = C.c_double()
        self._ck(self.lib.mp_flip_delta(self.h, chain, t, k, C.byref(out)), "mp_flip_delta")
        return out.value

    # -- sampler
    def init_chains(self, sc: MpSamplerConfig, disperse=False):
        self.sc = sc
        self._ck(self.lib.mp_init_chains(self.h, C.byref(sc), int(disperse)), "mp_init_chains")

    def set_sampler(self, sc: MpSamplerConfig):
        self.sc = sc
        self._ck(self.lib.mp_set_sampler(self.h, C.byref(sc)), "mp_set_sampler")

    def sweep(self, nsweeps=1, sync=True):
        self._ck(self.lib.mp_sweep(self.h, int(nsweeps)), "mp_sweep")
        if sync:
            self.synchronize()

    def set_shard(self, conn_lo=0, conn_hi=-1, task_first=0, task_stride=1):
        self._ck(self.lib.mp_set_shard(self.h, conn_lo, conn_hi, task_first, task_stride), "mp_set_shard")

    def sweep_phase(self, phase):
        flags = C.c_int(0)
        self._ck(self.lib.mp_sweep_phase(self.h, phase, C.byref(flags)), "mp_sweep_phase")
        return flags.value

    def synchronize(self):
        self._ck(self.lib.mp_synchronize(self.h), "mp_synchronize")

    def num_draws(self):
        return self.lib.mp_num_draws(self.h)

    def reset_draws(self):
        self._ck(self.lib.mp_reset_draws(self.h), "mp_reset_draws")

    def get_draws(self, first=0, count=None):
        if count is None:
            count = self.num_draws() - first
        out = np.zeros((count, self.C, NDRAW))
        if count:
            self._ck(self.lib.mp_get_draws(self.h, first, count, _p(out, _dp)), "mp_get_draws")
        return out

    # -- forward simulator
    def simulate(self, params, z0, nyears, nsims=1, seed=1, era_all=False, want_states=True, want_counts=True):
        par = self._one_param(params)
        z0 = np.ascontiguousarray(z0, dtype=np.uint8)
        z_out = np.zeros((nsims, nyears + 1, self.N), dtype=np.uint8) if want_states else None
        occ = np.zeros((nsims, nyears + 1), dtype=np.int32) if want_counts else None
        self._ck(self.lib.mp_simulate(self.h, C.byref(par), _p(z0, _u8p), nyears, nsims, seed, int(era_all),
                                      _p(z_out, _u8p), _p(occ, C.POINTER(C.c_int32))), "mp_simulate")
        return z_out, occ

    def simulate_ensemble(self, params, z0, nyears, seed=1, era_all=False, want_states=False):
        """One parameter set and one start state per trajectory (mp_simulate_ensemble)."""
        z0 = np.ascontiguousarray(z0, dtype=np.uint8)
        nsims = z0.shape[0]
        arr = (MpParams * nsims)()
        for i, p in enumerate(params):
            arr[i] = self._one_param(p)
        z_out = np.zeros((nsims, nyears + 1, self.N), dtype=np.uint8) if want_states else None
        occ = np.zeros((nsims, nyears + 1), dtype=np.int32)
        self._ck(self.lib.mp_simulate_ensemble(self.h, arr, _p(z0, _u8p), nyears, nsims, seed, int(era_all), _p(z_out, _u8p),
                                               _p(occ, C.POINTER(C.c_int32))), "mp_simulate_ensemble")
        return z_out, occ

    def forecast(self, nyears, nrep, seed=1, scenario=None, want_counts=True, want_incidence=True):
        """Posterior-predictive forecast from the chains' current state (mp_forecast): nrep trajectories per chain from the
        chain's z[c][T-1] and parameters.  scenario: dict with K, Ksrc, dsrc applied every year, or None for the plain model.
        Returns (occupied [C, nrep, nyears+1] int32, incidence [nyears+1, N] uint32), each None when not requested."""
        scen = None
        if scenario is not None:
            scen = np.array([float(scenario["K"]), float(scenario.get("Ksrc", 0.0)), float(scenario.get("dsrc", 0.0))])
        occ = np.zeros((self.C, nrep, nyears + 1), dtype=np.int32) if want_counts else None
        inc = np.zeros((nyears + 1, self.N), dtype=np.uint32) if want_incidence else None
        self._ck(self.lib.mp_forecast(self.h, int(nyears), int(nrep), int(seed), _p(scen, _dp), _p(occ, C.POINTER(C.c_int32)),
                                      _p(inc, C.POINTER(C.c_uint32))), "mp_forecast")
        return occ, inc

    def ppc(self, nrep, seed=1):
        """Posterior-predictive replicates of the observation table (mp_ppc): nrep per chain from the chain's imputed year 0,
        parameters and era flags, observed through the table's mask (and detection).  Returns dict(stats [C, nrep, T, 3] int32,
        obs_stats [T, 3] int32, patch_ge, patch_gt [N] uint32, nrep_total = C * nrep); statistics in PPC_STATS order.  Pool
        calls and chain shards with midaspom_b200.ppc_check."""
        stats = np.zeros((self.C, nrep, self.T, len(PPC_STATS)), dtype=np.int32)
        obs_stats = np.zeros((self.T, len(PPC_STATS)), dtype=np.int32)
        ge, gt = np.zeros(self.N, dtype=np.uint32), np.zeros(self.N, dtype=np.uint32)
        i32p, u32p = C.POINTER(C.c_int32), C.POINTER(C.c_uint32)
        self._ck(self.lib.mp_ppc(self.h, int(nrep), int(seed), _p(stats, i32p), _p(obs_stats, i32p), _p(ge, u32p), _p(gt, u32p)),
                 "mp_ppc")
        return dict(stats=stats, obs_stats=obs_stats, patch_ge=ge, patch_gt=gt, nrep_total=self.C * int(nrep))

    def capacity(self, params=None, keep=None, rtol=1e-6, max_iter=1000, values=False):
        """Metapopulation capacity lambda_M and patch values of the landscape (mp_capacity), one eigenproblem per parameter set.
        params: None (the chains' resident parameters), a list of parameter dicts, or rows of ``get_draws`` (any array whose last
        axis holds the NDRAW fields; the alpha and b columns are read).  keep: N flags, 0 removes a patch.  Returns dict(lam,
        residual, cull_bound, iters [nsets], values [nsets, N] or None, value_sum [N] or None, fingerprint); pool the results of
        several calls with the matching draws through midaspom_b200.persistence."""
        if params is None:
            arr, nsets = None, self.C
        else:
            if isinstance(params, np.ndarray):
                rows = np.asarray(params, dtype=np.float64).reshape(-1, NDRAW)
                params = [dict(alpha=r[DRAW_FIELDS.index("alpha")], b=r[DRAW_FIELDS.index("b")]) for r in rows]
            elif isinstance(params, dict):
                params = [params]
            nsets = len(params)
            arr = (MpParams * nsets)()
            for i, p in enumerate(params):
                arr[i] = self._one_param(p)
        keep_a = None if keep is None else np.ascontiguousarray(np.asarray(keep) != 0, dtype=np.uint8)
        if keep_a is not None and keep_a.shape != (self.N,):
            raise ValueError(f"keep must have shape {(self.N,)}")
        out3 = np.zeros((nsets, 3))
        iters = np.zeros(nsets, dtype=np.int32)
        vals = np.zeros((nsets, self.N)) if values else None
        vsum = np.zeros(self.N) if values else None
        self._ck(self.lib.mp_capacity(self.h, int(nsets), arr, _p(keep_a, _u8p), float(rtol), int(max_iter), _p(out3, _dp),
                                      _p(iters, C.POINTER(C.c_int32)), _p(vals, _dp), _p(vsum, _dp)), "mp_capacity")
        kept = np.ones(self.N, dtype=np.uint8) if keep_a is None else keep_a
        fp = hashlib.sha256(self._landscape_key + kept.tobytes()).hexdigest()
        return dict(lam=out3[:, 0].copy(), residual=out3[:, 1].copy(), cull_bound=out3[:, 2].copy(), iters=iters, values=vals,
                    value_sum=vsum, fingerprint=fp)

    # -- posterior summaries of the latent state
    def set_summaries(self, first_sweep=0, thin=1):
        """mp_set_summaries: accumulate the latent state at the end of sweeps first_sweep, first_sweep + thin, ... (thin=0: off).
        Zeroes the sums."""
        self._ck(self.lib.mp_set_summaries(self.h, int(first_sweep), int(thin)), "mp_set_summaries")

    def summaries(self, reset=False):
        """mp_get_summaries: dict(nsamples, z_count [T, N] uint32, z_prob [T, N], y_count [T-1, N] uint32, S_sum [T-1, N]),
        sums over the accumulated sweeps and this engine's chains; z_prob / nsamples is the posterior occupancy."""
        ns = C.c_int64()
        zc = np.zeros((self.T, self.N), dtype=np.uint32)
        zp = np.zeros((self.T, self.N))
        yc = np.zeros((self.T - 1, self.N), dtype=np.uint32)
        ss = np.zeros((self.T - 1, self.N))
        u32p = C.POINTER(C.c_uint32)
        self._ck(self.lib.mp_get_summaries(self.h, C.byref(ns), _p(zc, u32p), _p(zp, _dp), _p(yc, u32p), _p(ss, _dp), int(reset)),
                 "mp_get_summaries")
        return dict(nsamples=ns.value, z_count=zc, z_prob=zp, y_count=yc, S_sum=ss)

    # -- pointwise predictive densities for WAIC
    def set_waic(self, first_sweep=0, thin=1):
        """mp_set_waic: accumulate the predictive density of every observation at the end of sweeps first_sweep,
        first_sweep + thin, ... (thin=0: off).  Zeroes the sums."""
        self._ck(self.lib.mp_set_waic(self.h, int(first_sweep), int(thin)), "mp_set_waic")

    def waic_sums(self, reset=False):
        """mp_get_waic: dict(nsamples, lik_sum, loglik_sum, loglik_sq [T, N]), sums over the accumulated sweeps and this engine's
        chains, 0 in cells that are not observations; reduce them with midaspom_b200.waic."""
        ns = C.c_int64()
        out = [np.zeros((self.T, self.N)) for _ in range(3)]
        self._ck(self.lib.mp_get_waic(self.h, C.byref(ns), *[_p(a, _dp) for a in out], int(reset)), "mp_get_waic")
        return dict(nsamples=ns.value, lik_sum=out[0], loglik_sum=out[1], loglik_sq=out[2])

    # -- colonisations attributed to their sources
    def set_sources(self, first_sweep=0, thin=1, nbins=0, bin_width=0.0):
        """mp_set_sources: attribute the colonisations of every transition to their source patches at the end of sweeps
        first_sweep, first_sweep + thin, ... (thin=0: off); nbins > 0 adds a histogram of the shares over source-target
        distance bins of width bin_width (the last bin open).  Zeroes the sums."""
        self._ck(self.lib.mp_set_sources(self.h, int(first_sweep), int(thin), int(nbins), float(bin_width)), "mp_set_sources")
        self._src_bins = (int(nbins), float(bin_width) if int(nbins) > 0 else 0.0)

    def sources(self, reset=False):
        """mp_get_sources: dict(nsamples, events, unattributed [T-1] uint64, src_sum [T-1, N], ext_sum [T-1], dist_hist
        [T-1, nbins] or None, bin_width, fingerprint), sums over the accumulated sweeps and this engine's chains; reduce them
        with midaspom_b200.colonisation_sources."""
        nbins, width = getattr(self, "_src_bins", (0, 0.0))
        ns = C.c_int64()
        ev = np.zeros((2, self.T - 1), dtype=np.uint64)
        src = np.zeros((self.T - 1, self.N))
        ext = np.zeros(self.T - 1)
        hist = np.zeros((self.T - 1, nbins)) if nbins > 0 else None
        self._ck(self.lib.mp_get_sources(self.h, C.byref(ns), _p(ev, C.POINTER(C.c_uint64)), _p(src, _dp), _p(ext, _dp),
                                         _p(hist, _dp), int(reset)), "mp_get_sources")
        return dict(nsamples=ns.value, events=ev[0].copy(), unattributed=ev[1].copy(), src_sum=src, ext_sum=ext, dist_hist=hist,
                    bin_width=width, fingerprint=hashlib.sha256(self._landscape_key).hexdigest())

    @staticmethod
    def _one_param(p):
        d = dict(PARAM_DEFAULTS)
        d.update(p if isinstance(p, dict) else {k: getattr(p, k) for k in PARAM_FIELDS})
        return MpParams(*[float(d[k]) for k in PARAM_FIELDS])

    # -- plumbing
    def device_ptr(self, which):
        ptr, nbytes = C.c_void_p(), C.c_size_t()
        self._ck(self.lib.mp_device_ptr(self.h, which, C.byref(ptr), C.byref(nbytes)), "mp_device_ptr")
        return ptr.value, nbytes.value

    def stream(self):
        """Raw cudaStream_t of the engine (wrap with torch.cuda.ExternalStream for event timing)."""
        st = C.c_void_p()
        self._ck(self.lib.mp_get_stream(self.h, C.byref(st)), "mp_get_stream")
        return st.value or 0

    def set_timing(self, enabled=True):
        self._ck(self.lib.mp_set_timing(self.h, int(enabled)), "mp_set_timing")

    def get_timing(self, reset=False):
        ms = np.zeros(len(KERNEL_CATEGORIES))
        launches = np.zeros(len(KERNEL_CATEGORIES), dtype=np.int64)
        self._ck(self.lib.mp_get_timing(self.h, _p(ms, _dp), _p(launches, C.POINTER(C.c_int64)), int(reset)), "mp_get_timing")
        return dict(zip(KERNEL_CATEGORIES, ms.tolist())), dict(zip(KERNEL_CATEGORIES, launches.tolist()))

    def work_counters(self, reset=False):
        """Work executed by the hot kernels since the last reset (mp_get_work_counters)."""
        out = (C.c_uint64 * len(WORK_COUNTERS))()
        self._ck(self.lib.mp_get_work_counters(self.h, out, int(reset)), "mp_get_work_counters")
        return dict(zip(WORK_COUNTERS, [int(v) for v in out]))

    def conn_path(self):
        """Kernel that evaluated the connectivity last: "k_conn" or "gemm" (tcgen05 contraction for chains sharing alpha, b)."""
        return ("k_conn", "gemm")[self.lib.mp_get_conn_path(self.h)]

    def scan_geometry(self):
        out = (C.c_int * 4)()
        self._ck(self.lib.mp_get_scan_geometry(self.h, out), "mp_get_scan_geometry")
        return dict(threads_per_task=out[0], cluster=out[1], candidates_per_trip=out[2], culled=bool(out[3]), blocks=out[3] == 2)

    def probe_peaks(self):
        out = np.zeros(4)
        self._ck(self.lib.mp_probe_peaks(self.h, _p(out, _dp)), "mp_probe_peaks")
        return dict(mufu_gops=out[0], ffma_gfma=out[1], dadd_gops=out[2], copy_gbs=out[3])


def exact_posterior(obs, a=1.0 / 400.0, d=100.0, prior_occ=0.5, nstep=101, ecmin=0.0, ecmax=1.0, device=0):
    """mp_exact_posterior: the reference's exact grid likelihood (MIDASPOM.out's table) on the GPU.
    Returns (loglik[nstep, nstep], ltot, info dict); posterior density = exp(loglik - ltot)."""
    lib = load_library()
    obs = np.ascontiguousarray(obs, dtype=np.int8)
    T, n = obs.shape
    ll = np.zeros((nstep, nstep))
    ltot = C.c_double()
    info = (C.c_int * 4)()
    rc = lib.mp_exact_posterior(device, _p(obs, _i8p), T, n, float(a), float(d), float(prior_occ), int(nstep), float(ecmin),
                                float(ecmax), _p(ll, _dp), C.byref(ltot), info)
    if rc != 0:
        raise MpError(f"mp_exact_posterior failed ({rc}): {lib.mp_exact_last_error().decode()}")
    return ll, ltot.value, dict(nvar=info[0], nstates=info[1], nextid=info[2], max_states_per_year=info[3])


def exact_variant(variant, first_row, eB, cB, ts=20, tdis=10, a=1.0 / 400.0, d=200.0, prior_occ=0.5, nstepK=151, Kmin=0.1,
                  Kmax=100.0, nstepd=20, dmin=200.0, dmax=4000.0, device=0):
    """mp_exact_variant: MIDASPOM_dieoff.out ("dieoff") / MIDASPOM_loss.out ("loss") likelihood grids on the GPU."""
    lib = load_library()
    v = {"dieoff": 1, "loss": 2}[variant]
    row = np.ascontiguousarray(first_row, dtype=np.int8)
    out = np.zeros((nstepK, nstepd if v == 2 else 1))
    rc = lib.mp_exact_variant(device, v, _p(row, _i8p), len(row), float(a), float(d), float(prior_occ), float(eB), float(cB), int(ts),
                              int(tdis), int(nstepK), float(Kmin), float(Kmax), int(nstepd), float(dmin), float(dmax), _p(out, _dp))
    if rc != 0:
        raise MpError(f"mp_exact_variant failed ({rc}): {lib.mp_exact_last_error().decode()}")
    return out[:, 0] if v == 1 else out
