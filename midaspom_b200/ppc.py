"""Posterior-predictive check of a fit from the replicates ``Engine.ppc`` (``mp_ppc``) simulates on the device: Bayesian
p-values of the three statistics per year, an omnibus p-value per statistic over the years, and per-patch p-values.
Host-side numpy; the statistics themselves come from ``k_ppc_obs`` (definitions in DESIGN.md §2).

With M pooled replicates, T_rep[i, t, s] the statistic s of replicate i in year t and T_obs[t, s] that of the observations:

    p[t, s]      = min(1, 2 min(P(T_rep >= T_obs), P(T_rep <= T_obs)))                 (two-sided, per year)
    D[s]         = sum_{t >= 1, v_t > 0} (T[t, s] - m_t)^2 / v_t                        (m_t, v_t: replicate mean, variance)
    p_omnibus[s] = fraction of replicates with D_rep >= D_obs
    p_patch[k]   = min(1, 2 min(ge_k / M, 1 - gt_k / M))   ge_k / gt_k: replicates with D_k >= / > the observed D_k

Replicates start from the chains' imputed year 0, so year 0 enters neither the omnibus statistic nor, without detection, any
contrast with the data; years whose statistic does not vary over the replicates (v_t = 0) are left out of D.
"""
from __future__ import annotations

import numpy as np

from .engine import PPC_STATS


def _two_sided(p_ge, p_le):
    return np.minimum(1.0, 2.0 * np.minimum(p_ge, p_le))


def ppc_check(*results):
    """Pool any number of ``Engine.ppc`` results (calls on states taken every k sweeps with distinct seeds, chain shards of
    one fit) along the replicate axis and reduce them.  Raises ValueError when their ``obs_stats`` differ: the replicates
    were checked against different data.

    Returns dict(stats = PPC_STATS, nrep_total M, obs_stats [T, 3], rep_mean / rep_var [T, 3], p_year [T, 3],
    D_obs [3], D_rep [M, 3], p_omnibus [3], p_patch [N])."""
    if not results:
        raise ValueError("ppc_check: no results given")
    obs = np.asarray(results[0]["obs_stats"], dtype=np.int64)
    for r in results[1:]:
        o = np.asarray(r["obs_stats"], dtype=np.int64)
        if o.shape != obs.shape or not np.array_equal(o, obs):
            raise ValueError("ppc_check: the results were computed on different observations")
    T, ns = obs.shape
    rep = np.concatenate([np.asarray(r["stats"], dtype=np.int64).reshape(-1, T, ns) for r in results])
    M = rep.shape[0]
    if M != sum(int(r["nrep_total"]) for r in results):
        raise ValueError("ppc_check: stats do not hold nrep_total replicates")
    p_year = _two_sided((rep >= obs).mean(axis=0), (rep <= obs).mean(axis=0))
    m, v = rep.mean(axis=0), rep.var(axis=0)
    use = v > 0
    use[0] = False
    w = np.where(use, 1.0 / np.where(use, v, 1.0), 0.0)
    D_rep = (((rep - m) ** 2) * w).sum(axis=1)
    D_obs = (((obs - m) ** 2) * w).sum(axis=0)
    p_omnibus = (D_rep >= D_obs).mean(axis=0)
    ge = np.sum([np.asarray(r["patch_ge"], dtype=np.int64) for r in results], axis=0)
    gt = np.sum([np.asarray(r["patch_gt"], dtype=np.int64) for r in results], axis=0)
    p_patch = _two_sided(ge / M, 1.0 - gt / M)
    return dict(stats=PPC_STATS, nrep_total=M, obs_stats=obs, rep_mean=m, rep_var=v, p_year=p_year, D_obs=D_obs, D_rep=D_rep,
                p_omnibus=p_omnibus, p_patch=p_patch)
