"""Colonisation sources and realised dispersal distances from the sums ``Engine.sources`` (``mp_get_sources``) accumulates on
the device during sweeps.  Host-side numpy; the definitions are in DESIGN.md §2.

Every colonisation event (y_tk = 0, z_{t+1,k} = 1) of a sample is split over the occupied sources l in proportion to their
share of the colonisation pressure, rho_tkl = K_t w(k<-l) / P_tk, with the rest going to the external source.  Summed over the
events and divided by the number of samples, a patch's shares are the expected number of colonisations it seeded.  The shares
are of the pressure, not observed causal links: they read as "which source colonised k" only under independent propagule
contributions.
"""
from __future__ import annotations

import numpy as np

QUANTILES = (0.05, 0.5, 0.95)


def _seq(a):
    return list(a) if isinstance(a, (list, tuple)) else [a]


def _hist_stats(H, width):
    """Distance summaries of a pooled histogram H [nbins] with bins [b w, (b + 1) w), the last one open."""
    tot = float(H.sum())
    nb = H.shape[0]
    out = dict(density=np.zeros(nb - 1), mean_distance=float("nan"), beyond=float("nan"),
               quantiles={q: float("nan") for q in QUANTILES})
    if tot <= 0.0:
        return out
    out["density"] = H[:-1] / (tot * width)
    out["beyond"] = float(H[-1] / tot)
    closed = H[:-1]
    if closed.sum() > 0.0:
        out["mean_distance"] = float(np.sum((np.arange(nb - 1) + 0.5) * width * closed) / closed.sum())
    cdf = np.cumsum(H) / tot
    for q in QUANTILES:
        b = int(np.searchsorted(cdf, q, side="left"))
        if b >= nb - 1:
            out["quantiles"][q] = float("inf")          # in the open bin: at or beyond (nbins - 1) w
            continue
        lo = cdf[b - 1] if b > 0 else 0.0
        mass = H[b] / tot
        out["quantiles"][q] = float((b + (q - lo) / mass) * width) if mass > 0 else float(b * width)
    return out


def colonisation_sources(parts, summaries=None):
    """Pool source sums and reduce them to per-sample quantities.

    parts      one ``Engine.sources`` result or a list of them (calls or chain shards), pooled by addition.  Results of different
               landscapes (fingerprint), shapes (T, N) or distance bins are refused (ValueError)
    summaries  (optional) the matching ``Engine.summaries`` results, pooled the same way; their nsamples must equal the
               sources' (ValueError otherwise)

    Returns dict(nsamples, caused [N] (colonisations each patch seeded per sample, all transitions), caused_t [T-1, N],
    colonisations [T-1] (events per sample), unattributed [T-1], external [T-1] (external share per sample), share [N] (each
    patch's fraction of all attributed colonisations; the external source holds the rest), received [N] and net = caused -
    received (None without summaries), and with a histogram: dist_hist [nbins] per sample, density [nbins - 1] (normalised
    over all pairs, per unit distance, closed bins), mean_distance (bin midpoints, closed bins), beyond (fraction in the open
    bin) and quantiles {0.05, 0.5, 0.95} interpolated inside bins (inf in the open bin); these are None without a histogram."""
    ps = _seq(parts)
    if not ps:
        raise ValueError("colonisation_sources: no results")
    fps = {p.get("fingerprint") for p in ps}
    if len(fps) > 1:
        raise ValueError("colonisation_sources: the sums were computed on different landscapes")
    shapes = {np.shape(p["src_sum"]) for p in ps}
    if len(shapes) > 1:
        raise ValueError(f"colonisation_sources: different shapes (T-1, N): {sorted(shapes)}")
    bins = {(None if p.get("dist_hist") is None else np.shape(p["dist_hist"])[-1], float(p.get("bin_width", 0.0))) for p in ps}
    if len(bins) > 1:
        raise ValueError("colonisation_sources: the sums have different distance bins")
    ns = int(sum(int(p["nsamples"]) for p in ps))
    if ns <= 0:
        raise ValueError("colonisation_sources: no samples")
    src = sum(np.asarray(p["src_sum"], dtype=np.float64) for p in ps)
    ext = sum(np.asarray(p["ext_sum"], dtype=np.float64) for p in ps)
    events = sum(np.asarray(p["events"], dtype=np.int64) for p in ps)
    unattr = sum(np.asarray(p["unattributed"], dtype=np.int64) for p in ps)
    caused_t = src / ns
    caused = caused_t.sum(axis=0)
    attributed = float((events - unattr).sum()) / ns
    out = dict(nsamples=ns, caused=caused, caused_t=caused_t, colonisations=events / ns, unattributed=unattr / ns, external=ext / ns,
               share=caused / attributed if attributed > 0 else np.zeros_like(caused), received=None, net=None, dist_hist=None,
               density=None, mean_distance=None, beyond=None, quantiles=None)
    if summaries is not None:
        ss = _seq(summaries)
        if int(sum(int(s["nsamples"]) for s in ss)) != ns:
            raise ValueError("colonisation_sources: the summaries hold a different number of samples")
        zc = sum(np.asarray(s["z_count"], dtype=np.int64) for s in ss)
        yc = sum(np.asarray(s["y_count"], dtype=np.int64) for s in ss)
        if yc.shape != src.shape or zc.shape != (src.shape[0] + 1, src.shape[1]):
            raise ValueError("colonisation_sources: the summaries have another shape")
        out["received"] = (zc[1:] - yc).sum(axis=0) / ns
        out["net"] = caused - out["received"]
    nbins, width = next(iter(bins))
    if nbins is not None and nbins > 0:
        H = sum(np.asarray(p["dist_hist"], dtype=np.float64) for p in ps).sum(axis=0)
        out["dist_hist"] = H / ns
        out.update(_hist_stats(H, width))
    return out
