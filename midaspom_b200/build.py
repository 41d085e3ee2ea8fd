"""In-tree build of libmidaspom_cuda.so (sm_100a only; nvcc cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB_DIR = PKG / "lib"
OBJ_DIR = LIB_DIR / "obj"
LIB = LIB_DIR / "libmidaspom_cuda.so"
SOURCES = [CSRC / "mp_engine.cu", CSRC / "mp_sweep_fast_linear.cu", CSRC / "mp_sweep_fast_coords.cu",
           CSRC / "mp_sweep_fast_dense.cu", CSRC / "mp_exact.cu", CSRC / "mp_conn_gemm.cu", CSRC / "mp_comm.cu", CSRC / "mp_conn32.cu"]
HEADERS = [CSRC / "mp_device.cuh", CSRC / "mp_kernels.cuh", CSRC / "mp_conn.cuh", CSRC / "mp_sweep_fast.cuh", CSRC / "mp_sweep_cull.cuh", CSRC / "mp_capacity.cuh", CSRC / "mp_sources.cuh", CSRC / "mp_host.h", CSRC / "mp_comm.h",
           PKG.parent / "include" / "libmidaspom_cuda.h"]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"] + os.environ.get("MP_NVCC_EXTRA", "").split()


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(exe).exists():
        raise RuntimeError("nvcc not found: libmidaspom_cuda.so cannot be built (there is no CPU fallback)")
    return exe


def stale() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    return any(p.stat().st_mtime > t for p in SOURCES + HEADERS)


def _compile(src: Path, verbose: bool):
    obj = OBJ_DIR / (src.stem + ".o")
    cmd = [nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", str(obj), str(src)]
    res = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ))
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed on {src.name}:\n{res.stdout}{res.stderr}")
    return obj, res.stderr


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not stale():
        return LIB
    OBJ_DIR.mkdir(parents=True, exist_ok=True)
    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(lambda s: _compile(s, verbose), SOURCES))
    cmd = [nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(LIB)] + [str(o) for o, _ in results] + ["-ldl"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    if verbose:
        (LIB_DIR / "ptxas.log").write_text("".join(log for _, log in results))
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
