"""WAIC from the pointwise sums the engine accumulates during sweeps (``Engine.set_waic`` / ``Engine.waic_sums``), and the
paired comparison of two fits to the same observations.  Host-side numpy; the sums themselves come from ``k_waic``.

With S samples (sweeps x chains) and, per observed cell i, L_i = sum p, G_i = sum log p, Q_i = sum (log p)^2 of the
predictive density p of the observation (DESIGN.md §2):

    lppd_i   = log(L_i / S)
    p_waic_i = max(0, (Q_i - G_i^2 / S) / (S - 1))        (the sample variance of log p; NaN when S < 2)
    elpd_i   = lppd_i - p_waic_i

elpd_waic = sum_i elpd_i, waic = -2 elpd_waic (Watanabe 2010; Vehtari, Gelman and Gabry 2017).  The densities are
conditional on the chain's state of the previous year, so values compare only between fits to the same observation table
with the same prior_occ.
"""
from __future__ import annotations

import numpy as np


def waic(obs, *sums):
    """Reduce the WAIC sums of one or more engines (chain shards of one fit: their raw sums are added first).

    obs: the T x N observation table (-1 missing, 0, 1) the engines were given.  sums: dicts as ``Engine.waic_sums`` returns.
    Returns dict(observed [T, N] bool, lppd, p_waic, elpd [T, N] (NaN where not observed), elpd_waic, p_waic_total, waic,
    lppd_total, n_obs, nsamples)."""
    if not sums:
        raise ValueError("waic: no sums given")
    obs = np.asarray(obs)
    observed = obs >= 0
    S = int(sum(int(s["nsamples"]) for s in sums))
    tot = {}
    for key in ("lik_sum", "loglik_sum", "loglik_sq"):
        arrs = [np.asarray(s[key], dtype=np.float64) for s in sums]
        if any(a.shape != obs.shape for a in arrs):
            raise ValueError(f"waic: {key} does not have the shape {obs.shape} of the observations")
        tot[key] = np.sum(arrs, axis=0)
    if S < 1:
        raise ValueError("waic: no samples accumulated")
    L, G, Q = (tot[k][observed] for k in ("lik_sum", "loglik_sum", "loglik_sq"))
    with np.errstate(divide="ignore", invalid="ignore"):
        lppd_i = np.log(L / S)
        pw_i = np.maximum(0.0, (Q - G * G / S) / (S - 1)) if S >= 2 else np.full(L.shape, np.nan)
    elpd_i = lppd_i - pw_i

    def full(v):
        out = np.full(obs.shape, np.nan)
        out[observed] = v
        return out

    return dict(observed=observed, lppd=full(lppd_i), p_waic=full(pw_i), elpd=full(elpd_i),
                elpd_waic=float(elpd_i.sum()), p_waic_total=float(pw_i.sum()), waic=float(-2.0 * elpd_i.sum()),
                lppd_total=float(lppd_i.sum()), n_obs=int(observed.sum()), nsamples=S)


def compare_waic(a, b):
    """Paired comparison of two ``waic`` results on the same observed cells: dict(delta_elpd = sum_i (elpd_i^a - elpd_i^b),
    se = sqrt(n_obs var_i(elpd_i^a - elpd_i^b)), n_obs).  Positive delta_elpd favours a.  Raises ValueError when the two were
    computed on different observed-cell masks."""
    if a["observed"].shape != b["observed"].shape or not np.array_equal(a["observed"], b["observed"]):
        raise ValueError("compare_waic: the two fits were computed on different observed cells")
    m = a["observed"]
    d = a["elpd"][m] - b["elpd"][m]
    n = int(m.sum())
    se = float(np.sqrt(n * np.var(d, ddof=1))) if n >= 2 else float("nan")
    return dict(delta_elpd=float(d.sum()), se=se, n_obs=n)
