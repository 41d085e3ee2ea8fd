"""bench.py --dump-outputs on the GPU: what the last timed sweep returned, and the same arrays from two runs with the same
arguments (seeded workload, Philox draws keyed by chain and sweep), so that two builds can be compared output for output."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent


def run_bench(out_dir):
    args = [sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--workload", "tiny", "--steps", "2", "--warmup", "1",
            "--no-extra", "--no-cpu-baseline", "--ess-sweeps", "0", "--dump-outputs", str(out_dir)]
    res = subprocess.run(args, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    return line, {p.stem: np.load(p) for p in sorted(Path(out_dir).glob("*.npy"))}


def test_bench_dump_outputs_are_the_last_sweep_and_repeat_exactly(tmp_path):
    line, a = run_bench(tmp_path / "a")
    _, b = run_bench(tmp_path / "b")
    assert line["steps"] == 2 and line["config"]["chains"] == 4
    C, T, n = 4, 6, 256                                               # synth.WORKLOADS["tiny"], 4 chains on one GPU
    assert sorted(a) == ["S", "draws", "y", "z"]
    assert a["draws"].shape == (C, 11) and a["draws"].dtype == np.float64 and np.isfinite(a["draws"][:, 5]).all()
    assert a["z"].shape == (C, T, n) and a["z"].dtype == np.float32
    assert a["y"].shape == (C, T - 1, n) and a["y"].dtype == np.float32
    assert a["S"].shape == (C, T - 1, n) and a["S"].dtype == np.float64 and (a["S"] >= 0).all()
    z, y = a["z"], a["y"]
    assert np.isin(z, (0, 1)).all() and ((y <= z[:, :-1]) & (y <= z[:, 1:])).all()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
