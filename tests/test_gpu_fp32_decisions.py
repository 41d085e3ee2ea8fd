"""The FP32 sampler's Metropolis moves and z update against the FP64 engine, decision by decision.

The y scan of the FP32 engine follows the FP64 engine flip by flip (test_gpu_parity, test_gpu_blocks, test_gpu_scan_*).
This file covers every other decision of a sweep: the (alpha, b) ridge move with its proposal connectivity S_prop, the
c steps, the K / K_src / d_src steps, the Gibbs update of the latent z cells, e and p, and the recorded log-likelihood.

Two engines, FP32 and FP64, hold the same chains (update_y = 0, so y and with it S depend on (alpha, b) only).  Every
sweep runs phases 0-3 on both; the FP32 engine is then written back to the FP64 engine's parameters and z through the
device buffers, which leaves its resident S, its refresh cadence (every 16th sweep) and the culling of its k_conn
untouched.  A host replay in FP64 (numpy, a host Philox) recomputes every proposal, log u and acceptance log-ratio d from
the FP64 engine's S and S_prop; it must take the FP64 engine's decisions wherever |d - log u| exceeds the FP64 summation
slack.  The FP32 engine must take the same decisions except where |d - log u| <= delta, delta being the FP32 error bound
of DESIGN §5 summed over the cells whose colonisation term differs between the two parameter sets of the decision.
"""
import itertools
import math

import numpy as np
import pytest

import midaspom_b200 as mb
import oracle_lib as O
from gpu_util import make_engine
from midaspom_b200 import synth

# ------------------------------------------------------------------ host Philox4x32-10 with the key / counter layout of mp::rng
RK_INIT_PARAM, RK_INIT_Z, RK_SIM_EXT, RK_SIM_COL, RK_Z, RK_Y = 1, 2, 3, 4, 5, 6
RK_AB, RK_C, RK_E, RK_P, RK_K, RK_KSRC, RK_DSRC = 7, 8, 9, 10, 11, 12, 13
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: 4 uint32 arrays, key: 2 uint32 arrays (broadcastable) -> 4 uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) for x in ctr]
    k0, k1 = (np.asarray(x, dtype=np.uint64) for x in key)
    shape = np.broadcast_shapes(*(x.shape for x in c), k0.shape, k1.shape)
    c = [np.broadcast_to(x, shape).copy() for x in c]
    k0, k1 = np.broadcast_to(k0, shape).copy(), np.broadcast_to(k1, shape).copy()
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        h0, l0, h1, l1 = p0 >> np.uint64(32), p0 & _M32, p1 >> np.uint64(32), p1 & _M32
        c = [h1 ^ c[1] ^ k0, l1, h0 ^ c[3] ^ k1, l0]
        k0 = (k0 + np.uint64(0x9E3779B9)) & _M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & _M32
    return [x.astype(np.uint32) for x in c]


def rng(seed, chain, sweep, kind, a, b):
    seed = int(seed)
    key1 = (np.uint64((seed >> 32) & 0xFFFFFFFF) + np.asarray(chain, dtype=np.uint64)) & _M32
    return philox4x32_10((a, b, kind, sweep), (np.uint64(seed & 0xFFFFFFFF), key1))


def u01(x):
    return (np.asarray(x, dtype=np.float64) + 0.5) * (1.0 / 4294967296.0)


def logit_u(x):
    u = u01(x)
    return np.log(u) - np.log1p(-u)


def box_muller(x0, x1):
    r = np.sqrt(-2.0 * np.log(u01(x0)))
    th = 6.283185307179586476925286766559 * u01(x1)
    return r * np.cos(th), r * np.sin(th)


def test_host_philox_matches_the_oracle_bit_for_bit():
    L = O.lib()
    g = np.random.default_rng(2024)
    n = 12000
    kinds = np.array([RK_AB, RK_C, RK_K, RK_KSRC, RK_DSRC, RK_Z, RK_E, RK_P], dtype=np.uint32)
    seed = g.integers(0, 2 ** 64, n, dtype=np.uint64)
    seed[:8] = [0, 1, 2 ** 32 - 1, 2 ** 32, 2 ** 64 - 1, 12345, 7, 2 ** 63]      # key words at their edges
    chain = g.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    chain[:16] = np.arange(16)
    sweep = g.integers(0, 1 << 20, n).astype(np.uint32)
    kind = kinds[np.arange(n) % len(kinds)]
    a = g.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    b = g.integers(0, 64, n).astype(np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    p = out.ctypes.data_as(O.C.POINTER(O.C.c_uint32))
    want = np.empty((n, 4), dtype=np.uint32)
    for i in range(n):
        L.spom_rng(int(seed[i]), int(chain[i]), int(sweep[i]), int(kind[i]), int(a[i]), int(b[i]), p)
        want[i] = out
    # every row carries its own seed: split it into the two key words as mp::rng does
    k0 = seed & _M32
    k1 = ((seed >> np.uint64(32)) + chain.astype(np.uint64)) & _M32
    got = np.stack(philox4x32_10((a, b, kind, sweep), (k0, k1)), axis=1)
    assert np.array_equal(got, want)
    for i in range(0, n, 997):                                                   # the scalar entry point agrees too
        assert np.array_equal(np.array([int(w) for w in rng(int(seed[i]), chain[i], sweep[i], kind[i], a[i], b[i])],
                                       dtype=np.uint32), want[i])
    x = want.reshape(-1)
    assert np.array_equal(u01(x[:20000]), np.array([L.spom_u01(int(v)) for v in x[:20000]]))
    assert np.array_equal(u01(np.array([0, 2 ** 32 - 1], np.uint32)), [0.5 / 2 ** 32, (2 ** 32 - 0.5) / 2 ** 32])
    # logit_u and box_muller are the device formulas on u01 (their outputs enter every decision the GPU tests replay)
    u = u01(x[:1000])
    assert np.allclose(logit_u(x[:1000]), np.log(u / (1 - u)), rtol=1e-12, atol=1e-12)
    n1, n2 = box_muller(x[:1000], x[1000:2000])
    assert np.allclose(n1 ** 2 + n2 ** 2, -2.0 * np.log(u), rtol=1e-12)


# ------------------------------------------------------------------ FP32 error model (DESIGN §5) of one colonisation term
U = 2.0 ** -24                 # FP32 unit roundoff
LG2_ERR = 2.0 ** -22           # lg2.approx.ftz.f32: absolute error for x in [0.5, 2], else 2 ulp of the result (PTX ISA)
EX2_ERR = 2.0 ** -22           # ex2.approx.ftz.f32: relative error
LN2 = math.log(2.0)
BUF_Z, BUF_PARAMS, BUF_S_PROP = 1, 4, 5
PF = mb.engine.PARAM_FIELDS    # e, c, alpha, b, p, K, Ksrc, dsrc


def log_err(x):
    """Error bound of 0.6931472f * lg2.approx.ftz(x) against log(x) for an exact float x (natural-log units)."""
    a = np.abs(np.log2(x))
    return LN2 * LG2_ERR * np.maximum(1.0, a) + U * LN2 * a


def term_bound(v, zn, eps):
    """Bound on |FP32 term - FP64 term| of a y = 0 cell: v = the FP64 c (K_t S + K_src,t g) before the clamp, zn = z_{t+1},
    eps = relative error bound of the FP32 value of v.  z' = 1: log C; z' = 0: log(1 - C), where 1 - C is exact for
    C >= 1/2 and one rounding otherwise.  Infinite when the FP32 C may reach the clamp of a z' = 0 cell or underflow; 0 for
    a z' = 0 cell that both engines clamp (-inf in both: see certain_ninf)."""
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        C = np.minimum(v, 1.0)
        hi = np.minimum(v * (1.0 + eps), 1.0)
        b1 = np.where(v * (1.0 - eps) >= 1.0, log_err(1.0), eps / (1.0 - eps) + log_err(C))
        b0 = np.where(v * (1.0 - eps) >= 1.0, 0.0, np.where(hi >= 1.0, np.inf, (hi - C) / (1.0 - hi) + U + log_err(1.0 - C)))
        b = np.where(zn, b1, b0)
    return np.where(zn & (v > 0) & (v * (1.0 - eps) < 2.0 ** -126), np.inf, b)   # the FP32 C may flush to 0: log C = -inf


def pair_bound(v1, v0, zn, ecom, eown):
    """Bound on the FP32 error of term(v1) - term(v0) for two parameter sets that share one S (the c and K / K_src / d_src
    steps): the relative error ecom of the engine's S enters both terms through the same float and is bounded by its
    effect on the difference; eown (the casts, products and source term) by term_bound per set."""
    def G(v):
        C = np.minimum(v, 1.0)
        return np.where(zn, np.log(C), np.log1p(-C))
    with np.errstate(divide="ignore", invalid="ignore"):
        g1, g0 = G(v1), G(v0)
        com = np.zeros_like(v1)
        for e in (ecom, -ecom):
            h = np.abs((G(v1 * (1.0 + e)) - g1) - (G(v0 * (1.0 + e)) - g0))
            com = np.maximum(com, np.where(np.isnan(h), np.inf, h))
    return com + term_bound(v1, zn, eown) + term_bound(v0, zn, eown)


def certain_ninf(v, zn, eps, s32, src):
    """Cells whose FP32 term is -inf for certain, so that the FP32 engine rejects the parameter set: z' = 0 cells clamped to
    C = 1 in both precisions (-inf in both), and z' = 1 cells whose FP32 C is 0 -- an FP32 S of 0 without a source term
    (every weight flushed by ex2.approx.ftz, DESIGN §5) or a v below the smallest normal float (flushed by the cast)."""
    return (~zn & (v * (1.0 - eps) >= 1.0)) | (zn & (((s32 == 0) & ~src) | (v * (1.0 + eps) < 2.0 ** -126)))


class Replay:
    """FP64 host restatement of phases 1 and 3 of a sweep (k_propose_*, k_sum_S / k_ridge_c, k_col_ll, k_decide_*,
    k_update_z, k_update_ep, k_record) for C chains with a fixed y."""

    def __init__(self, spec, y, sc, seed, prior_occ):
        self.obs = np.asarray(spec["obs"], np.int8)
        self.T, self.N = self.obs.shape
        self.C = y.shape[0]
        self.y = y.astype(bool)
        self.sc, self.seed, self.p0 = sc, seed, prior_occ
        self.detect = int(spec.get("detect", 0))
        T, N = self.T, self.N
        self.era = np.zeros(T - 1, bool) if spec.get("era") is None else np.asarray(spec["era"]).astype(bool)
        su = spec.get("src_unit")
        self.unit = np.arange(1, N + 1, dtype=np.float64) if su is None else np.asarray(su, np.float64)
        # y = 0 cells of every chain (y is fixed: update_y = 0)
        ch, t, k = np.nonzero(~self.y)
        self.ych, self.yt, self.yk = ch, t, k
        self.yflat = (ch * (T - 1) + t) * N + k
        self.ypre = self.era[t]
        # latent z cells that no adjacent y = 1 forces
        lat = (self.obs == -1) | ((self.obs == 0) if self.detect else False)
        forced = np.zeros((self.C, T, N), bool)
        forced[:, 1:] |= self.y
        forced[:, :-1] |= self.y
        ch, t, k = np.nonzero(lat[None] & ~forced)
        self.lch, self.lt, self.lk = ch, t, k
        self.lobs = self.obs[t, k]

    # ---- colonisation terms
    def col_v(self, P, S, ch, t, k, pre, flat):
        s = S.reshape(-1)[flat]
        c, K, Ks, al, ds = (P[f][ch] for f in ("c", "K", "Ksrc", "alpha", "dsrc"))
        src = pre & (Ks != 0.0)
        g = np.where(src, np.exp(-((al * self.unit[k]) * ds)), 0.0)
        ks = np.where(pre, K, 1.0) * s
        v = c * (ks + np.where(pre, Ks, 0.0) * g)
        # relative error the FP32 source term carries into v: ex2.approx of an FP32 argument alpha u dsrc log2 e, weighted
        # by the source term's share of v
        with np.errstate(divide="ignore", invalid="ignore"):
            share = np.where(src, Ks * g / (ks + Ks * g), 0.0)
        esrc = share * (EX2_ERR + 4 * U * LN2 * np.where(src, al * self.unit[k] * ds / LN2, 0.0))
        return v, src, esrc

    def col_terms(self, P, S, z):
        v, src, esrc = self.col_v(P, S, self.ych, self.yt, self.yk, self.ypre, self.yflat)
        zn = z[self.ych, self.yt + 1, self.yk].astype(bool)
        C = np.minimum(v, 1.0)
        with np.errstate(divide="ignore"):
            term = np.where(zn, np.log(C), np.log1p(-C))
        return term, v, zn, src, esrc

    def chain_sum(self, x):
        return np.bincount(self.ych, weights=x, minlength=self.C)

    def ll_col(self, P, S, z):
        term, v, zn, src, esrc = self.col_terms(P, S, z)
        bad = (self.y & ~z[:, 1:].astype(bool)).reshape(self.C, -1).any(1)
        with np.errstate(invalid="ignore"):
            ll = self.chain_sum(term)
            return np.where(bad, -np.inf, ll), self.chain_sum(np.abs(np.where(np.isfinite(term), term, 0.0))), (v, zn, src, esrc)

    @staticmethod
    def eS_of(S32, S64, flat):
        """Relative difference of the engines' S per cell."""
        s64 = S64.reshape(-1)[flat]
        with np.errstate(divide="ignore", invalid="ignore"):
            return np.where(s64 > 0, np.abs(S32.reshape(-1)[flat] - s64) / s64, 0.0)

    @staticmethod
    def eps_of(S32, S64, flat, c_rel, src, esrc, pre=False):
        """Relative error bound of the FP32 v: the engines' S (measured), c, the casts and products of col_prob, and the
        source term exp(-alpha u dsrc) (esrc, from col_v).  c S: three roundings (the casts of S and c, the
        product); c (K S + K_src g): three more (the cast of K, its product, the sum)."""
        eS = 0.0 if S32 is None else Replay.eS_of(S32, S64, flat)
        return eS + c_rel + 3 * U + np.where(pre, 3 * U, 0.0) + np.where(src, esrc, 0.0)

    # ---- sufficient counts (k_counts)
    def counts(self, z):
        T = self.T
        zz = z.astype(bool)
        zt = zz[:, :T - 1]
        pre = self.era[None, :, None]
        f = lambda m: m.reshape(self.C, -1).sum(1)
        cn = dict(N10=f(zt & ~self.y & ~pre), N11=f(zt & self.y & ~pre), N10P=f(zt & ~self.y & pre), N11P=f(zt & self.y & pre),
                  BADEXT=f(~zt & self.y), SY=f(self.y), SZ=f(zz))
        o = self.obs[None]
        cn["ND"] = f((o == 1) & zz)
        cn["NM"] = f((o == 0) & zz) if self.detect else np.zeros(self.C, int)
        cn["BADDET"] = f((o == 1) & ~zz) + (0 if self.detect else f((o == 0) & zz))
        return cn

    @staticmethod
    def xlogd(n, v):
        with np.errstate(divide="ignore", invalid="ignore"):
            return np.where(n > 0, n * np.log(v), 0.0)

    def ll_ext(self, e, K, cn):
        E0, E1 = np.minimum(e, 1.0), np.minimum(e / K, 1.0)
        v = self.xlogd(cn["N10"], E0) + self.xlogd(cn["N11"], 1 - E0) + self.xlogd(cn["N10P"], E1) + self.xlogd(cn["N11P"], 1 - E1)
        return np.where(cn["BADEXT"] > 0, -np.inf, v)

    def ll_det(self, p, cn):
        v = self.xlogd(cn["ND"], p) + self.xlogd(cn["NM"], 1 - p) if self.detect else 0.0 * p
        return np.where(cn["BADDET"] > 0, -np.inf, v)

    def rng(self, sweep, kind, a, b=0):
        return rng(self.seed, np.arange(self.C), sweep, kind, a, b)

    # ---- latent z cells (z_logodds): log-odds and the FP32 error bound of each
    def z_logodds(self, P, S, S32=None, c_rel=0.0):
        ch, t, k = self.lch, self.lt, self.lk
        T, N = self.T, self.N
        lo = np.zeros(len(ch))
        band = np.zeros(len(ch))
        m = t > 0
        tp = np.maximum(t - 1, 0)
        flat = (ch * (T - 1) + tp) * N + k
        v, src, esrc = self.col_v(P, S, ch, tp, k, self.era[tp], flat)
        C = np.minimum(v, 1.0)
        with np.errstate(divide="ignore", invalid="ignore"):
            col = np.log(C) - np.log1p(-C)
            if S32 is not None:
                eps = self.eps_of(S32, S, flat, c_rel, src, esrc, self.era[tp])
                # C clamped to 1 in FP32 too (log-odds +inf in both engines) or C = 0 in both (-inf): no band
                band = np.where(m & (v * (1.0 - eps) < 1.0) & (v > 0),
                                term_bound(v, True, eps) + term_bound(v, False, eps) + 2 * U * np.abs(col), 0.0)
        lo = np.where(m, col, 0.0)
        e, K = P["e"][ch], P["K"][ch]
        E = np.minimum(np.where(self.era[np.minimum(t, T - 2)], e / K, e), 1.0)
        with np.errstate(divide="ignore"):
            logE = np.log(E)
        me = t < T - 1
        lo = lo + np.where(me, logE, 0.0)
        band = band + np.where(me & np.isfinite(lo), U * np.abs(logE) + 2 * U * np.abs(lo), 0.0)
        lo = lo + np.where(t == 0, math.log(self.p0) - math.log(1 - self.p0), 0.0)
        if self.detect:
            with np.errstate(divide="ignore"):
                lo = lo + np.where(self.lobs == 0, np.log(1 - P["p"][ch]), 0.0)
        return lo, band

    def z_draws(self, sweep):
        return logit_u(rng(self.seed, self.lch, sweep, RK_Z, self.lk, self.lt)[0])


def paths(v0, ls0, normals, mul, lo, hi, adapt, g):
    """Every accept / reject sequence of a group of random-walk steps: (decisions, final value, final log scale)."""
    out = []
    for dec in itertools.product((0, 1), repeat=len(normals)):
        v, ls, ok = v0, ls0, True
        for a, n1 in zip(dec, normals):
            q = v * math.exp(math.exp(ls) * n1) if mul else v + math.exp(ls) * n1
            if a and not (lo <= q <= hi):
                ok = False
            if a:
                v = q
            if adapt:
                ls += g * (a - 0.44)
        if ok:
            out.append((dec, v, ls))
    return out


def infer(cands, v, ls, rtol):
    """The decision sequence whose outcome is the engine's (v, ls)."""
    hit = [d for d, pv, pls in cands if abs(pv - v) <= rtol * abs(v) + 1e-300 and abs(pls - ls) <= 1e-9]
    assert len(hit) >= 1, f"no accept/reject sequence reproduces the engine's value {v!r}"
    return hit[0]


# ------------------------------------------------------------------ the two engines, sweep by sweep
def as_arrays(plist):
    return {f: np.array([p.get(f, mb.engine.PARAM_DEFAULTS[f]) for p in plist], dtype=np.float64) for f in PF}


def as_matrix(P):
    return np.stack([P[f] for f in PF], axis=1)


def s_error(S32, S64, P, y, spec, rtol=1e-5):
    """Largest relative error of an FP32 connectivity against the FP64 one over the entries within rtol, and the number of
    entries beyond it.  Each of those must be explained by the FP32 weights of DESIGN §5: either the sum lacks weights
    that ex2.approx.ftz flushes to zero (2^(log2 A^b - alpha d log2 e) < 2^-126; checked against the FP64 sums of the
    weights the FP32 engine keeps and of those it may keep), or its weights are far enough down for the error of the FP32
    exponent (|log2 w| (8 u) for the argument's roundings and sqrt.approx, alpha log2 e times 4 x 2^-24 of the half extent
    for the coordinates) to pass rtol."""
    assert (S32[S64 == 0] == 0).all()
    with np.errstate(divide="ignore", invalid="ignore"):
        rel = np.where(S64 > 0, np.abs(S32 - S64) / S64, 0.0)
    bad = np.argwhere(rel > rtol)
    assert len(bad) <= 20000, f"{len(bad)} connectivity entries off by more than {rtol}"
    px, py = np.asarray(spec["px"]), np.asarray(spec["py"])
    half = 0.5 * max(np.ptp(px), np.ptp(py))
    area = np.ones(len(px)) if spec.get("area") is None else np.asarray(spec["area"])
    for c, t, k in bad:
        src = np.nonzero(y[c, t])[0]
        src = src[src != k]
        d = np.hypot(px[k] - px[src], py[k] - py[src])
        lw = -P["alpha"][c] * d / LN2 + P["b"][c] * np.log2(area[src])      # log2 of each weight
        w = np.exp2(lw)
        lo = w[lw > -126.0 + 1e-3].sum()
        hi = w[lw > -126.0 - 1e-3].sum()
        e = EX2_ERR + LN2 * (np.abs(lw) * 8 * U + P["alpha"][c] / LN2 * 4 * U * half)
        model = (w * e).sum() / w.sum() + 1e-12
        if hi >= S64[c, t, k] * (1 - rtol):
            assert rel[c, t, k] <= model, (f"connectivity of chain {c}, year {t}, patch {k}: FP32 {S32[c, t, k]!r}, FP64 "
                                           f"{S64[c, t, k]!r}, relative error {rel[c, t, k]:.3g} > {model:.3g}")
            continue
        tol = max(rtol, model)
        assert lo * (1 - tol) <= S32[c, t, k] <= hi * (1 + tol), \
            (f"connectivity of chain {c}, year {t}, patch {k}: FP32 {S32[c, t, k]!r}, FP64 {S64[c, t, k]!r}, FP64 sum of the "
             f"weights above the flush limit {lo!r}..{hi!r}, alpha {P['alpha'][c]!r}")
    ok = np.ones(S64.shape, bool)
    ok[tuple(bad.T)] = False
    return float(rel[ok].max(initial=0.0)), len(bad)


class Pair:
    def __init__(self, spec, z, y, plist, lsig, sc, seed=31, prior_occ=0.5):
        import torch
        self.torch = torch
        self.C = len(plist)
        self.e = {}
        for prec in (mb.FP64, mb.FP32):
            eng = make_engine(dict(spec, prior_occ=prior_occ), n_chains=self.C, precision=prec, seed=seed, max_draws=64)
            eng.init_chains(sc)
            eng.set_params(plist)
            eng.set_state(z, y)
            eng.set_scales(lsig)
            self.e[prec] = eng
        self.T, self.N = spec["obs"].shape

    def view(self, prec, which, shape, typestr):
        from midaspom_b200.distributed import engine_tensor
        return engine_tensor(self.e[prec], which, shape, typestr, "cuda:0")

    def s_prop(self, prec):
        self.e[prec].synchronize()
        return self.view(prec, BUF_S_PROP, (self.C, self.T - 1, self.N), "<f8").cpu().numpy()

    def read(self, prec):
        eng = self.e[prec]
        z, _ = eng.get_state()
        return as_arrays(eng.get_params()), eng.get_scales(), z

    def sync_fp32(self, P, lsig, z, reset_S):
        """Write the FP64 engine's parameters, scales and z into the FP32 engine.  Through the device buffers unless (alpha, b)
        changed for a chain (then its resident S is stale and set_params makes the next sweep recompute it)."""
        e32 = self.e[mb.FP32]
        if reset_S:
            e32.set_params([dict(zip(PF, row)) for row in as_matrix(P)])
        else:
            e32.synchronize()
            self.view(mb.FP32, BUF_PARAMS, (self.C, 8), "<f8").copy_(self.torch.from_numpy(as_matrix(P)))
            self.torch.cuda.synchronize()
        e32.synchronize()
        self.view(mb.FP32, BUF_Z, (self.C, self.T, self.N), "|u1").copy_(self.torch.from_numpy(np.ascontiguousarray(z)))
        self.torch.cuda.synchronize()
        e32.set_scales(lsig)

    def close(self):
        for eng in self.e.values():
            eng.close()


def run_case(name, spec, z0, y0, plist, lsig, sc_kw, nsweeps, seed=31):
    sc = mb.engine.sampler_config(**sc_kw)
    scd = {f: getattr(sc, f) for f, _ in mb.engine.MpSamplerConfig._fields_}
    pair = Pair(spec, z0, y0, plist, lsig, sc, seed=seed)
    rp = Replay(spec, y0, scd, seed, 0.5)
    C = pair.C
    ch = np.arange(C)
    groups = [(w, f, i) for w, f, i, on in ((0, "K", 5, scd["sample_K"]), (1, "Ksrc", 6, scd["sample_Ksrc"]),
                                           (2, "dsrc", 7, scd["sample_dsrc"])) if on]
    lims = dict(K=("K_min", "K_max"), Ksrc=("Ksrc_min", "Ksrc_max"), dsrc=("dsrc_min", "dsrc_max"))
    st = dict(band_by_step={}, delta_by_step={}, beyond=0, inf_band=0, decisions=0, in_band=0, disagree=0, sprop_err=0.0, s_err=0.0, z_cells=0, z_band=0, z_disagree=0,
              rep_checked=0, refresh_sweeps=0, ab_delta_max=0.0)
    P, L, z = as_arrays(plist), np.array(lsig, dtype=np.float64).reshape(C, -1), np.array(z0)
    reset = False
    for s in range(nsweeps):
        adapt, gain = s < scd["n_adapt"], 1.0 / (s + 1.0) ** 0.6
        f64, f32 = pair.e[mb.FP64].sweep_phase(0), pair.e[mb.FP32].sweep_phase(0)
        st["refresh_sweeps"] += f32 & 1
        S64, S32 = pair.e[mb.FP64].get_connectivity(), pair.e[mb.FP32].get_connectivity()
        Sp64, Sp32 = pair.s_prop(mb.FP64), pair.s_prop(mb.FP32)
        Q0 = dict(P)
        r = rp.rng(s, RK_AB, 0)
        n1, n2 = box_muller(r[0], r[1])
        Q0["alpha"], Q0["b"] = P["alpha"] * np.exp(np.exp(L[:, 2]) * n1), P["b"] + np.exp(L[:, 3]) * n2
        for a, b, key, par in ((Sp32, Sp64, "sprop_err", Q0), (S32, S64, "s_err", P)):
            err, nflush = s_error(a, b, par, y0, spec)
            st[key] = max(st[key], err)
            st["beyond"] += nflush
        for prec in (mb.FP64, mb.FP32):
            pair.e[prec].sweep_phase(1)
        P64, L64, z64 = pair.read(mb.FP64)
        P32, L32, z32 = pair.read(mb.FP32)

        steps = []         # per decision: (d64, logu, delta, replay decision, FP64 decision, FP32 decision)
        # -- (alpha, b) ridge move
        r = rp.rng(s, RK_AB, 0)
        n1, n2 = box_muller(r[0], r[1])
        logu = np.log(u01(r[2]))
        Q = {f: P[f].copy() for f in PF}
        Q["alpha"] = P["alpha"] * np.exp(np.exp(L[:, 2]) * n1)
        Q["b"] = P["b"] + np.exp(L[:, 3]) * n2
        inb = (Q["alpha"] >= scd["alpha_min"]) & (Q["alpha"] <= scd["alpha_max"]) & (Q["b"] >= scd["b_min"]) & (Q["b"] <= scd["b_max"])
        m1_64, m2_64 = S64.reshape(C, -1).sum(1), Sp64.reshape(C, -1).sum(1)
        m1_32, m2_32 = S32.reshape(C, -1).sum(1), Sp32.reshape(C, -1).sum(1)
        c2_64, c2_32 = P["c"] * (m1_64 / m2_64), P["c"] * (m1_32 / m2_32)
        ljac64, ljac32 = np.log(c2_64 / P["c"]), np.log(c2_32 / P["c"])
        Q["c"] = c2_64
        inb &= (c2_64 >= scd["c_min"]) & (c2_64 <= scd["c_max"])
        cur, cabs, (v0, zn0, src0, esrc0) = rp.ll_col(P, S64, z)
        pr, pabs, (v1, zn1, src1, esrc1) = rp.ll_col(Q, Sp64, z)
        with np.errstate(invalid="ignore"):
            d = pr - cur + ljac64
        dec_rep = inb & ~np.isnan(d) & (logu < d)
        dec64 = P64["alpha"] != P["alpha"]
        dec32 = P32["alpha"] != P["alpha"]
        assert np.allclose(P64["alpha"][dec64], Q["alpha"][dec64], rtol=1e-12, atol=0)
        assert np.allclose(P64["b"][dec64], Q["b"][dec64], rtol=1e-12, atol=0) and (P64["b"][~dec64] == P["b"][~dec64]).all()
        c_rel = np.abs(c2_32 - c2_64) / c2_64
        eps1 = rp.eps_of(Sp32, Sp64, rp.yflat, c_rel[rp.ych], src1, esrc1, rp.ypre)
        bnd = rp.chain_sum(term_bound(v1, zn1, eps1) + term_bound(v0, zn0, rp.eps_of(S32, S64, rp.yflat, 0.0, src0, esrc0, rp.ypre)))
        slack = 1e-9 + 1e-14 * (cabs + pabs)
        delta = bnd + np.abs(ljac32 - ljac64) + slack
        ninf = rp.chain_sum(certain_ninf(v1, zn1, eps1, Sp32.reshape(-1)[rp.yflat], src1)) > 0
        delta = np.where(ninf, 0.0, delta)                      # the FP32 engine rejects for certain
        st["ab_delta_max"] = max(st["ab_delta_max"], float(np.max(np.where(np.isfinite(delta), delta, 0))))
        steps.append(('ab', d, logu, delta, slack, dec_rep, dec64, dec32))
        llc = np.where(dec64, pr, cur)
        llc_abs = np.where(dec64, pabs, cabs)
        cells = tuple(np.where(dec64[rp.ych], a1, a0) for a1, a0 in ((v1, v0), (zn1, zn0), (src1, src0), (esrc1, esrc0)))
        Sa64 = np.where(dec64[:, None, None], Sp64, S64)
        Sa32 = np.where(dec64[:, None, None], Sp32, S32)
        Pc = {f: np.where(dec64, Q[f], P[f]) for f in PF}
        c_start32 = np.where(dec32, c2_32, P["c"])
        c_off = np.where(dec64, c_rel, 0.0)                     # the FP32 engine's c carries its own ridge factor
        ls_ab = L[:, 2] + (gain * (dec64 - 0.30) if adapt else 0.0)
        assert np.allclose(L64[:, 2], ls_ab, rtol=0, atol=1e-12)

        # -- c steps: decisions of each engine from its final c and scale
        nc = scd["n_c_steps"]
        rc = [rp.rng(s, RK_C, j) for j in range(nc)]
        nrm = [box_muller(x[0], x[1])[0] for x in rc]
        lus = [np.log(u01(x[2])) for x in rc]
        dc64 = np.zeros((C, nc), bool)
        dc32 = np.zeros((C, nc), bool)
        for i in range(C):
            nn = [nrm[j][i] for j in range(nc)]
            dc64[i] = infer(paths(Pc["c"][i], L[i, 1], nn, False, scd["c_min"], scd["c_max"], adapt, gain), P64["c"][i], L64[i, 1], 1e-9)
            dc32[i] = infer(paths(c_start32[i], L[i, 1], nn, False, scd["c_min"], scd["c_max"], adapt, gain), P32["c"][i], L32[i, 1], 1e-9)
        ls = L[:, 1].copy()
        for j in range(nc):
            Q = {f: Pc[f].copy() for f in PF}
            Q["c"] = Pc["c"] + np.exp(ls) * nrm[j]
            inb = (Q["c"] >= scd["c_min"]) & (Q["c"] <= scd["c_max"])
            pr, pabs, (v1, zn1, src1, esrc1) = rp.ll_col(Q, Sa64, z)
            v0, zn0, src0, esrc0 = cells
            with np.errstate(invalid="ignore"):
                d = pr - llc
            # the same v (S = 0 without a source) or clamped in both sets: the same FP32 term, which cancels
            diff = (v1 != v0) & ~((v0 >= 1.0) & (v1 >= 1.0) & zn0)
            eS = rp.eS_of(Sa32, Sa64, rp.yflat)
            eps = eS + rp.eps_of(None, None, rp.yflat, c_off[rp.ych], src0, esrc0, rp.ypre)
            bnd = rp.chain_sum(np.where(diff, pair_bound(v1, v0, zn0, eS, eps - eS), 0.0))
            slack = 1e-9 + 1e-14 * (pabs + llc_abs)
            bnd = np.where(rp.chain_sum(certain_ninf(v1, zn1, eps, Sa32.reshape(-1)[rp.yflat], src1)) > 0, -slack, bnd)
            steps.append(('c', d, lus[j], bnd + slack, slack, inb & ~np.isnan(d) & (lus[j] < d), dc64[:, j], dc32[:, j]))
            acc = dc64[:, j]
            Pc["c"] = np.where(acc, Q["c"], Pc["c"])
            llc, llc_abs = np.where(acc, pr, llc), np.where(acc, pabs, llc_abs)
            cells = tuple(np.where(acc[rp.ych], a1, a0) for a1, a0 in ((v1, v0), (zn1, zn0), (src1, src0), (esrc1, esrc0)))
            if adapt:
                ls = ls + gain * (acc - 0.44)

        # -- variant parameters from the counts of the current z
        cn = rp.counts(z)
        nv = scd["n_v_steps"]
        for which, f, li in groups:
            lo_, hi_ = scd[lims[f][0]], scd[lims[f][1]]
            rv = [rp.rng(s, RK_K + which, j) for j in range(nv)]
            nrm = [box_muller(x[0], x[1])[0] for x in rv]
            lus = [np.log(u01(x[2])) for x in rv]
            dv64 = np.zeros((C, nv), bool)
            dv32 = np.zeros((C, nv), bool)
            for i in range(C):
                cand = paths(Pc[f][i], L[i, li], [nrm[j][i] for j in range(nv)], f != "dsrc", lo_, hi_, adapt, gain)
                dv64[i] = infer(cand, P64[f][i], L64[i, li], 1e-12)
                dv32[i] = infer(cand, P32[f][i], L32[i, li], 1e-12)
            ls = L[:, li].copy()
            for j in range(nv):
                Q = {g: Pc[g].copy() for g in PF}
                Q[f] = Pc[f] * np.exp(np.exp(ls) * nrm[j]) if f != "dsrc" else Pc[f] + np.exp(ls) * nrm[j]
                inb = (Q[f] >= lo_) & (Q[f] <= hi_)
                pr, pabs, (v1, zn1, src1, esrc1) = rp.ll_col(Q, Sa64, z)
                v0, zn0, src0, esrc0 = cells
                with np.errstate(invalid="ignore"):
                    d = (pr - llc) + (rp.ll_ext(Q["e"], Q["K"], cn) - rp.ll_ext(Pc["e"], Pc["K"], cn))
                diff = v1 != v0                                      # pre-event cells with K S > 0 (K) or a source term
                eS = rp.eS_of(Sa32, Sa64, rp.yflat)
                eps = eS + rp.eps_of(None, None, rp.yflat, c_off[rp.ych], src0 | src1, np.maximum(esrc0, esrc1), rp.ypre)
                bnd = rp.chain_sum(np.where(diff, pair_bound(v1, v0, zn0, eS, eps - eS), 0.0))
                slack = 1e-9 + 1e-14 * (pabs + llc_abs)
                bnd = np.where(rp.chain_sum(certain_ninf(v1, zn1, eps, Sa32.reshape(-1)[rp.yflat], src1)) > 0, -slack, bnd)
                steps.append((f, d, lus[j], bnd + slack, slack, inb & ~np.isnan(d) & (lus[j] < d), dv64[:, j], dv32[:, j]))
                acc = dv64[:, j]
                Pc[f] = np.where(acc, Q[f], Pc[f])
                llc, llc_abs = np.where(acc, pr, llc), np.where(acc, pabs, llc_abs)
                cells = tuple(np.where(acc[rp.ych], a1, a0) for a1, a0 in ((v1, v0), (zn1, zn0), (src1, src0), (esrc1, esrc0)))
                if adapt:
                    ls = ls + gain * (acc - 0.44)

        # -- the replay takes the FP64 engine's decisions; the FP32 engine's up to its first one inside the band
        for f in ("alpha", "b", "K", "Ksrc", "dsrc"):
            assert np.allclose(P64[f], Pc[f], rtol=1e-12, atol=0), f
        assert np.allclose(P64["c"], Pc["c"], rtol=1e-9, atol=0)
        follows = np.ones(C, bool)                                # FP32 chain still in the FP64 chain's state
        for kind, d, lu, delta, slack, drep, d64, d32 in steps:
            gap = np.abs(d - lu)
            far = ~(gap <= slack)                                  # NaN d (rejected in both) counts as far
            bad = far & (drep != d64)
            assert not bad.any(), f"{name} sweep {s}: the FP64 replay and the FP64 engine differ (chains {np.nonzero(bad)[0]})"
            st["rep_checked"] += int(far.sum())
            band = gap <= delta
            st["decisions"] += int(follows.sum())
            st["in_band"] += int((follows & band).sum())
            st["inf_band"] += int((follows & band & ~np.isfinite(delta)).sum())
            st["band_by_step"][kind] = st["band_by_step"].get(kind, 0) + int((follows & band).sum())
            st["delta_by_step"][kind] = max(st["delta_by_step"].get(kind, 0.0), float(np.median(delta)))
            wrong = follows & (d32 != d64)
            out = wrong & ~band
            assert not out.any(), (f"{name} sweep {s}: FP32 decision differs outside the band: chains {np.nonzero(out)[0]}, "
                                   f"d={d[out]}, log u={lu[out]}, delta={delta[out]}")
            st["disagree"] += int(wrong.sum())
            follows &= ~wrong
        for f in ("alpha", "b", "K", "Ksrc", "dsrc"):               # FP64 arithmetic on the same draws: bit-identical
            assert (P32[f][follows] == P64[f][follows]).all(), f
        assert np.allclose(P32["c"][follows], P64["c"][follows], rtol=1e-6, atol=0)
        assert (L32[follows] == L64[follows]).all()

        # -- Gibbs update of the latent z cells
        lod, zband = rp.z_logodds(P64, Sa64, Sa32, c_off[rp.lch] + np.abs(P32["c"] - P64["c"])[rp.lch] / P64["c"][rp.lch])
        lu = rp.z_draws(s)
        zrep = np.where(np.isnan(lod), False, lu < lod)
        zg64 = z64[rp.lch, rp.lt, rp.lk].astype(bool)
        zg32 = z32[rp.lch, rp.lt, rp.lk].astype(bool)
        with np.errstate(invalid="ignore"):
            gap = np.abs(lod - lu)
        far = ~(gap <= 1e-9 * (1 + np.abs(lod)))
        assert not (far & (zrep != zg64)).any(), f"{name} sweep {s}: the z replay and the FP64 engine differ"
        m = follows[rp.lch]
        zb = gap <= zband
        zw = m & (zg32 != zg64)
        assert not (zw & ~zb).any(), f"{name} sweep {s}: FP32 z differs outside the band: lod {lod[zw & ~zb][:5]}, band {zband[zw & ~zb][:5]}"
        st["z_cells"] += int(m.sum())
        st["z_band"] += int((m & zb).sum())
        st["z_disagree"] += int(zw.sum())
        same_z = follows & ~np.bincount(rp.lch[zw], minlength=C).astype(bool)
        # non-latent cells never move
        keep = np.ones(z64.shape, bool)
        keep[rp.lch, rp.lt, rp.lk] = False
        assert (z64[keep] == z[keep]).all() and (z32[keep] == z[keep]).all()

        # -- phase 3: e and p from the counts, the recorded draw
        pair.e[mb.FP64].sweep_phase(2)
        pair.e[mb.FP32].sweep_phase(2)
        pair.e[mb.FP64].sweep_phase(3)
        pair.e[mb.FP32].sweep_phase(3)
        Pf64, Lf64, _ = pair.read(mb.FP64)
        Pf32, Lf32, _ = pair.read(mb.FP32)
        cn = rp.counts(z64)
        Pr = {f: P64[f].copy() for f in PF}
        Lr = L64.copy()
        for field, li, kind, on, fn in (("e", 0, RK_E, scd["sample_e"], lambda q: rp.ll_ext(q, Pr["K"], cn)),
                                        ("p", 4, RK_P, scd["sample_p"] and rp.detect, lambda q: rp.ll_det(q, cn))):
            if not on:
                continue
            llx = fn(Pr[field])
            for j in range(scd["n_e_steps"]):
                x = rp.rng(s, kind, j)
                q = Pr[field] + np.exp(Lr[:, li]) * box_muller(x[0], x[1])[0]
                ok = (q >= scd[field + "_min"]) & (q <= scd[field + "_max"])
                with np.errstate(invalid="ignore"):
                    l2 = fn(q)
                    acc = ok & ~np.isnan(l2 - llx) & (np.log(u01(x[2])) < l2 - llx)
                Pr[field] = np.where(acc, q, Pr[field])
                llx = np.where(acc, l2, llx)
                if adapt:
                    Lr[:, li] += gain * (acc - 0.44)
        for f in PF:
            assert np.allclose(Pf64[f], Pr[f], rtol=1e-12, atol=0), f
        assert np.allclose(Lf64, Lr, rtol=0, atol=1e-12)
        for f in PF:
            if f != "c":
                assert (Pf32[f][same_z] == Pf64[f][same_z]).all(), f
        assert (Lf32[same_z] == Lf64[same_z]).all()
        dr64 = pair.e[mb.FP64].get_draws(s, 1)[0]
        dr32 = pair.e[mb.FP32].get_draws(s, 1)[0]
        assert (dr32[same_z, 6:8] == dr64[same_z, 6:8]).all()
        assert (dr64[:, 6] == cn["SY"]).all() and (dr64[:, 7] == cn["SZ"]).all()
        a, b = dr32[same_z, 5], dr64[same_z, 5]
        assert np.isfinite(b).all() and (np.abs(a - b) <= 1e-5 * np.abs(b)).all(), np.max(np.abs(a - b) / np.abs(b))

        # -- next sweep from the FP64 engine's state
        _, _, zf64 = pair.read(mb.FP64)
        reset = bool(((Pf32["alpha"] != Pf64["alpha"]) | (Pf32["b"] != Pf64["b"])).any())
        P, L, z = Pf64, Lf64, zf64
        pair.sync_fp32(P, L, z, reset)
    pair.close()
    print(f"\n{name}: {nsweeps} sweeps x {C} chains, decisions compared {st['decisions']}, in band {st['in_band']} ({st['inf_band']} of them with an infinite bound; by step {st['band_by_step']}, largest median delta by step {st['delta_by_step']}), "
          f"disagreements {st['disagree']}, FP64 replay decisions checked {st['rep_checked']}; "
          f"largest S_prop error {st['sprop_err']:.2e}, S error {st['s_err']:.2e} (entries beyond 1e-5, each within the FP32 "
          f"weight error or at the ex2 flush limit: {st['beyond']}); latent cells compared {st['z_cells']}, "
          f"in band {st['z_band']}, disagreements {st['z_disagree']}; FP32 sweeps with a refresh of S {st['refresh_sweeps']}; "
          f"largest (alpha, b) delta {st['ab_delta_max']:.3g}")
    return st


def check_stats(st):
    assert st["sprop_err"] <= 1e-5 and st["s_err"] <= 1e-5, st
    assert st["in_band"] <= 0.01 * st["decisions"], st
    assert st["z_band"] <= 1e-4 * st["z_cells"], st


# ------------------------------------------------------------------ cases
SC = dict(sample_e=1, sample_c=1, sample_alpha=1, sample_b=1, n_c_steps=2, update_y=0, update_z=1, n_adapt=1000)


def feasible_c(spec, y, plist, frac=0.9, seed=31):
    """Largest c per chain that keeps every empty cell of the next year possible (C < 1), times frac; also returns the
    FP64 connectivity of each chain's (alpha, b)."""
    C = len(plist)
    z = np.zeros((C,) + spec["obs"].shape, np.uint8)
    with make_engine(spec, n_chains=C, precision=mb.FP64, seed=seed) as eng:
        eng.set_params(plist)
        eng.set_state(z, y)
        S = eng.connectivity()
    return S


def start_params(truth, C, g, spread=1.0, **extra):
    out = []
    for i in range(C):
        p = dict(e=truth["e"] * g.uniform(0.8, 1.2), c=truth["c"], alpha=truth["alpha"] * math.exp(spread * g.uniform(-0.3, 0.3)),
                 b=min(2.0, max(0.0, truth["b"] + spread * g.uniform(-0.2, 0.2))), p=truth.get("p", 1.0) * g.uniform(0.95, 1.0))
        for k, v in extra.items():
            p[k] = v * g.uniform(0.8, 1.2)
        out.append(p)
    return out


def set_c(spec, z, y, plist, g, scale):
    """c of every chain: scale x the largest value that keeps every y = 0, z' = 0 cell below the clamp."""
    S = feasible_c(spec, y, [dict(p, c=1.0) for p in plist])
    rp = Replay(spec, y, {}, 0, 0.5)
    P1 = as_arrays([dict(mb.engine.PARAM_DEFAULTS, **dict(p, c=1.0)) for p in plist])
    v, _, _ = rp.col_v(P1, S, rp.ych, rp.yt, rp.yk, rp.ypre, rp.yflat)
    zn = z[rp.ych, rp.yt + 1, rp.yk].astype(bool)
    vmax = np.full(len(plist), 1e-300)
    np.maximum.at(vmax, rp.ych[~zn], v[~zn])
    for i, p in enumerate(plist):
        p["c"] = min(scale[i] / vmax[i], 1.0)
    return S, v, zn


def workload_case(name, C=64, extra=None):
    wl = synth.make_workload(name)
    spec = dict(geom=O.GEOM_COORDS, px=wl["px"], py=wl["py"], area=wl["area"], obs=wl["obs"], detect=wl["detect"],
                era=wl.get("era"), src_unit=wl.get("src_unit"))
    g = np.random.default_rng(7)
    z1 = wl["z_true"].astype(np.uint8)
    z = np.broadcast_to(z1, (C,) + z1.shape).copy()
    y = (z[:, :-1] & z[:, 1:] & (g.random(z[:, :-1].shape) < 0.7)).astype(np.uint8)
    plist = start_params(wl["truth"], C, g, **(extra or {}))
    set_c(spec, z, y, plist, g, g.uniform(0.3, 0.8, C))
    lsig = np.array([[math.log(0.05), math.log(0.1 * p["c"]), math.log(0.05), math.log(0.05), math.log(0.05),
                      math.log(0.1), math.log(0.1), math.log(0.1 * 3800.0)] for p in plist])
    return spec, z, y, plist, lsig


def edge_case(n, C=64, T=10):
    """Random landscape with three edges at once: >= 5 % of the y = 0 cells at the clamp C = 1, E = min(1, e/K) = 1 in the
    pre-event years, and proposal steps of (alpha, b) of scale 1 (alpha'/alpha spans about e^+-2)."""
    g = np.random.default_rng(n)
    from gpu_util import random_landscape
    spec, z1, _ = random_landscape(g, n, T, O.GEOM_COORDS, occ=0.45, miss=0.05)
    era = (np.arange(T - 1) < T // 2).astype(np.uint8)
    spec["era"] = era
    y1 = (z1[:-1] & z1[1:] & (g.random((T - 1, n)) < 0.6)).astype(np.uint8)
    y1[era.astype(bool)] = 0                                      # E = 1 before the event: no patch survives ...
    spec["src_unit"] = 1.0 + 2.0 * (spec["px"] - spec["px"].min()) / np.ptp(spec["px"])   # ... and colonists come from a source
    y = np.broadcast_to(y1, (C, T - 1, n)).copy()
    truth = dict(e=0.3, c=1.0, alpha=1.0 / 400, b=0.5)
    plist = start_params(truth, C, g, spread=0.3, K=0.22, Ksrc=2.0, dsrc=200.0)   # e / K > 1
    # the y = 0 cells with the largest connectivity are occupied next year and sit at the clamp
    S = feasible_c(spec, y, [dict(p, c=1.0) for p in plist])
    s0 = S[0]
    q = np.quantile(s0[y1 == 0], 0.92)
    z1 = z1.copy()
    z1[1:][(y1 == 0) & (s0 >= q)] = 1
    obs = z1.astype(np.int8)
    obs[spec["obs"] == -1] = -1
    spec["obs"] = obs
    z = np.broadcast_to(z1, (C, T, n)).copy()
    _, v, zn = set_c(spec, z, y, plist, g, np.full(C, 0.999))
    P = as_arrays([dict(mb.engine.PARAM_DEFAULTS, **p) for p in plist])
    rp = Replay(spec, y, {}, 0, 0.5)
    vc = v * P["c"][rp.ych]
    clamped = rp.chain_sum((vc >= 1.0).astype(float)) / rp.chain_sum(np.ones_like(vc))
    assert np.median(clamped) >= 0.05, clamped
    lsig = np.array([[math.log(0.05), math.log(0.1 * p["c"]), 0.0, 0.0, math.log(0.05), math.log(0.1), math.log(0.1),
                      math.log(380.0)] for p in plist])
    return spec, z, y, plist, lsig


CASES = {
    # name: (builder, sampler switches, sweeps).  17 sweeps take the FP32 engine through its refresh of S at sweep 16.
    "cfg3": (lambda: workload_case("cfg3"), {}, 3),
    "cfg2": (lambda: workload_case("cfg2"), dict(sample_p=1), 17),
    "cfg4": (lambda: workload_case("cfg4", C=16, extra=dict(K=3.0)), dict(sample_K=1), 3),
    "cfg4l": (lambda: workload_case("cfg4l", C=16, extra=dict(Ksrc=5.0, dsrc=500.0)), dict(sample_Ksrc=1, sample_dsrc=1), 3),
    "edges700": (lambda: edge_case(700), dict(sample_K=1), 17),
    "edges4100": (lambda: edge_case(4100), dict(sample_K=1), 17),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_fp32_decisions_follow_the_fp64_engine(case):
    build, sw, nsweeps = CASES[case]
    spec, z, y, plist, lsig = build()
    st = run_case(case, spec, z, y, plist, lsig, dict(SC, **sw), nsweeps)
    check_stats(st)
    assert st["refresh_sweeps"] == (2 if nsweeps > 16 else 1)


@pytest.mark.gpu
def test_fp32_weights_flush_to_zero_beyond_the_documented_distance():
    """ex2.approx.ftz flushes a weight to 0 once alpha d - b ln A > 126 ln 2 (DESIGN §5).  Two clusters of three patches
    east of a 700-patch landscape, at alpha d = 80 and 95 from every other patch, each with an observed colonisation: the
    FP32 S of the far cluster is exactly 0 and its log-likelihood -inf, where the FP64 engine stays finite."""
    from gpu_util import random_landscape
    g = np.random.default_rng(90)
    n0, T, alpha = 700, 3, 1.0 / 400
    spec, z0, _ = random_landscape(g, n0, T, O.GEOM_COORDS, occ=0.45, areas=False)
    px, py = list(spec["px"]), list(spec["py"])
    xe, yc = max(px), float(np.median(py))
    for gap in (80.0, 95.0):
        for j in range(3):
            px.append(xe + gap / alpha + 30.0 * j)
            py.append(yc + 20.0 * j)
    n = n0 + 6
    spec.update(px=np.array(px), py=np.array(py))
    z = np.zeros((2, T, n), np.uint8)
    z[:, :, :n0] = z0
    z[0, 1, n0] = 1                                               # chain 0: colonisation in the near cluster
    z[1, 1, n0 + 3] = 1                                           # chain 1: colonisation in the far cluster
    y = (z[:, :-1] & z[:, 1:]).astype(np.uint8)
    res = {}
    for prec in (mb.FP64, mb.FP32):
        sp = dict(spec, obs=np.full((T, n), -1, np.int8))
        with make_engine(sp, n_chains=2, precision=prec) as eng:
            eng.set_params([dict(mb.engine.PARAM_DEFAULTS, e=0.3, c=0.01, alpha=alpha)] * 2)
            eng.set_state(z, y)
            S = eng.connectivity()
            ll, parts = eng.loglik()
        res[prec] = (S, ll, parts)
    S64, S32 = res[mb.FP64][0], res[mb.FP32][0]
    X, Y = np.array(px), np.array(py)
    for c in range(2):
        for t in range(T - 1):
            src = np.nonzero(y[c, t])[0]
            d = np.sqrt((X[:, None] - X[None, src]) ** 2 + (Y[:, None] - Y[None, src]) ** 2)
            w = np.exp(-alpha * d)
            w[src, np.arange(len(src))] = 0.0
            arg = alpha * d / LN2                                 # -log2 of each weight
            flushed, kept = arg > 126.0 * (1 + 1e-5), arg < 126.0 * (1 - 1e-5)
            lo = np.where(kept, w, 0.0).sum(1)                    # the FP32 sum holds every kept weight ...
            hi = np.where(flushed, 0.0, w).sum(1)                 # ... and none of the flushed ones
            assert np.allclose(S64[c, t], w.sum(1), rtol=1e-9, atol=0) and (S64[c, t] > 0).all()
            assert (S32[c, t][hi == 0] == 0).all()
            assert ((S32[c, t] >= lo * (1 - 1e-5)) & (S32[c, t] <= hi * (1 + 1e-5))).all()
    assert S32[0, 0, n0] > 0 and S32[1, 0, n0 + 3] == 0
    ll64, ll32 = res[mb.FP64][1], res[mb.FP32][1]
    assert np.isfinite(ll64).all()
    assert abs(ll32[0] - ll64[0]) <= 1e-5 * abs(ll64[0])
    assert ll32[1] == -np.inf


@pytest.mark.gpu
def test_fp32_colonisation_terms_near_the_clamp():
    """log(1 - C) in FP32 as C -> 1: the largest C of each chain's empty-next-year cells sits 8 to 64 FP32 units of
    roundoff below the clamp.  The FP32 colonisation log-likelihood stays finite and within the summed per-cell bound of
    the FP64 one."""
    from gpu_util import random_landscape
    g = np.random.default_rng(701)
    n, T, C = 700, 6, 64
    spec, z1, _ = random_landscape(g, n, T, O.GEOM_COORDS, occ=0.45)
    y1 = (z1[:-1] & z1[1:] & (g.random((T - 1, n)) < 0.6)).astype(np.uint8)
    z = np.broadcast_to(z1, (C, T, n)).copy()
    y = np.broadcast_to(y1, (C, T - 1, n)).copy()
    plist = start_params(dict(e=0.3, c=1.0, alpha=1.0 / 400, b=0.5), C, g)
    k = np.linspace(8.0, 64.0, C)
    S64, v, zn = set_c(spec, z, y, plist, g, 1.0 - k * U)
    P = as_arrays([dict(mb.engine.PARAM_DEFAULTS, **p) for p in plist])
    rp = Replay(spec, y, {}, 0, 0.5)
    vc = v * P["c"][rp.ych]
    top = np.zeros(C)
    np.maximum.at(top, rp.ych[~zn], vc[~zn])
    assert np.allclose(1.0 - top, k * U, rtol=1e-6, atol=0)
    res = {}
    for prec in (mb.FP64, mb.FP32):
        with make_engine(spec, n_chains=C, precision=prec) as eng:
            eng.set_params(plist)
            eng.set_state(z, y)
            _, parts = eng.loglik()
            res[prec] = (parts[:, 1], eng.get_connectivity())
    ll64, ll32, S32 = res[mb.FP64][0], res[mb.FP32][0], res[mb.FP32][1]
    term, v64, zn64, src, arg = rp.col_terms(P, res[mb.FP64][1], z)
    assert np.allclose(rp.chain_sum(term), ll64, rtol=1e-12, atol=0)
    bound = rp.chain_sum(term_bound(v64, zn64, rp.eps_of(S32, res[mb.FP64][1], rp.yflat, 0.0, src, arg, rp.ypre)))
    assert np.isfinite(bound).all() and np.isfinite(ll32).all(), ll32
    err = np.abs(ll32 - ll64)
    print(f"\nnear the clamp: |FP32 - FP64| of the colonisation log-likelihood {err.max():.3g}, bound {bound.min():.3g}..{bound.max():.3g}")
    assert (err <= bound).all(), (err, bound)
