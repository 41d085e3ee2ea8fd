"""Persistence of a fitted SPOM from the metapopulation capacity ``Engine.capacity`` (``mp_capacity``) computes on the device for
every retained draw.  Host-side numpy; the definitions are in DESIGN.md §2.

With lambda_M the capacity of a draw's (alpha, b) and e, c, K its other parameters:

    R     = (1 - e) (1 + c lambda_M)                          growth factor of the model linearised at the empty state
    R_pre = (1 - min(1, e / K)) (1 + c K lambda_M)            the same before the event of a die-off fit (draws with K != 1)
    loss_k = -2 lambda_M V_k                                  first-order change of lambda_M when patch k is removed

R > 1 is the persistence threshold of this discrete-time model.  R_pre is not defined for fits with an external source
(Ksrc > 0): the empty state is not absorbing before the event.
"""
from __future__ import annotations

import numpy as np

from .engine import DRAW_FIELDS, NDRAW


def _summary(x):
    q = np.quantile(x, [0.025, 0.5, 0.975])
    return dict(mean=float(np.mean(x)), q025=float(q[0]), q50=float(q[1]), q975=float(q[2]))


def _seq(a):
    return list(a) if isinstance(a, (list, tuple)) else [a]


def persistence(draws, lam, values=None):
    """Reduce per-draw capacities to posterior summaries of lambda_M and R.

    draws  rows of ``Engine.get_draws`` (any array whose last axis holds the NDRAW fields), or a list of them: one per call or
           chain shard, pooled in order
    lam    the matching ``Engine.capacity`` results (dicts) or arrays of lambda_M, one per entry of ``draws``.  Results that carry a
           fingerprint must all carry the same one: capacities of different landscapes or patch masks are not pooled (ValueError)
    values (optional) the matching per-draw patch values [M, N]; taken from the results when they hold them

    Returns dict(n_draws, lam, R, R_pre (None without K != 1 or with Ksrc > 0), lam_summary, R_summary, R_pre_summary,
    P_R_gt_1, P_R_pre_gt_1, value_mean [N] and loss_mean [N] (None without values))."""
    ds, ls = _seq(draws), _seq(lam)
    if len(ds) != len(ls):
        raise ValueError("persistence: need one capacity result per block of draws")
    fps = {r["fingerprint"] for r in ls if isinstance(r, dict) and r.get("fingerprint") is not None}
    if len(fps) > 1:
        raise ValueError("persistence: the capacities were computed on different landscapes or patch masks")
    rows = np.concatenate([np.asarray(d, dtype=np.float64).reshape(-1, NDRAW) for d in ds])
    lam_v = np.concatenate([np.asarray(r["lam"] if isinstance(r, dict) else r, dtype=np.float64).reshape(-1) for r in ls])
    if lam_v.shape[0] != rows.shape[0]:
        raise ValueError(f"persistence: {rows.shape[0]} draws but {lam_v.shape[0]} capacities")
    if values is None and all(isinstance(r, dict) and r.get("values") is not None for r in ls):
        values = [r["values"] for r in ls]
    col = {k: rows[:, DRAW_FIELDS.index(k)] for k in ("e", "c", "K", "Ksrc")}
    e, c, K = col["e"], col["c"], col["K"]
    R = (1.0 - e) * (1.0 + c * lam_v)
    R_pre = None
    if np.any(K != 1.0) and not np.any(col["Ksrc"] > 0.0):
        R_pre = (1.0 - np.minimum(1.0, e / K)) * (1.0 + c * K * lam_v)
    out = dict(n_draws=int(rows.shape[0]), lam=lam_v, R=R, R_pre=R_pre, lam_summary=_summary(lam_v), R_summary=_summary(R),
               R_pre_summary=None if R_pre is None else _summary(R_pre), P_R_gt_1=float(np.mean(R > 1.0)),
               P_R_pre_gt_1=None if R_pre is None else float(np.mean(R_pre > 1.0)), value_mean=None, loss_mean=None)
    if values is not None:
        V = np.concatenate([np.asarray(v, dtype=np.float64).reshape(-1, np.shape(v)[-1]) for v in _seq(values)])
        if V.shape[0] != rows.shape[0]:
            raise ValueError(f"persistence: {rows.shape[0]} draws but {V.shape[0]} rows of patch values")
        out["value_mean"] = V.mean(axis=0)
        out["loss_mean"] = (-2.0 * lam_v[:, None] * V).mean(axis=0)
    return out
