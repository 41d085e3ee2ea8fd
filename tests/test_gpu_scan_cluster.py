"""Launch shape of the culled y scan at 512 threads per task: clusters of 4 x 128 threads whatever the number of (chain, year)
tasks (several such CTAs of different tasks share an SM), and the decisions of that shape against the FP64 path."""
import numpy as np
import pytest

import midaspom_b200 as mb
import oracle_lib as O
from gpu_util import make_engine, pdict, random_landscape

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("C", [64, 16, 8])
def test_culled_scan_runs_in_clusters_of_four(monkeypatch, C):
    monkeypatch.delenv("MP_FAST_TPT", raising=False); monkeypatch.delenv("MP_FAST_CS", raising=False)
    rng = np.random.default_rng(300 + C)
    n, T = 10000, 20
    spec, z, y = random_landscape(rng, n, T, O.GEOM_COORDS, occ=0.5, miss=0.03)
    par = pdict(e=0.35, c=0.004, alpha=1 / 400, b=0.5)
    sc = mb.engine.sampler_config(sample_e=0, sample_c=0, update_z=0, n_adapt=0)
    out = {}
    for prec in ((mb.FP64, mb.FP32) if C <= 8 else (mb.FP32,)):         # the FP64 scan of 64 chains is slow; one case suffices
        with make_engine(spec, n_chains=C, precision=prec, seed=13, max_draws=1) as eng:
            eng.set_params([par] * C)
            eng.set_state(np.stack([z] * C), np.stack([y] * C))
            eng.set_sampler(sc)
            eng.connectivity(fetch=False)
            eng.sweep(1)
            out[prec] = (eng.get_state()[1], eng.get_connectivity(), eng.connectivity(), eng.scan_geometry())
    y32, S32, S32new, geo = out[mb.FP32]
    assert geo["threads_per_task"] == 512 and geo["cluster"] == 4 and geo["culled"] and not geo["blocks"], geo
    cand = ((z[:-1] & z[1:]) == 1).sum() * C
    if mb.FP64 in out:
        assert (out[mb.FP64][0] != y32).sum() <= max(2, 2e-3 * cand)
    assert ((y32 <= z[None, :-1]) & (y32 <= z[None, 1:])).all()
    err = np.abs(S32 - S32new) / np.maximum(np.abs(S32new), 1e-9)
    assert err.max() <= 1e-6, err.max()
