"""Pins the CPU oracle (oracle/spom_oracle.c) to the reference: golden vectors produced by the
reference binaries / functions (tests/golden/golden.npz, see make_golden.py) and, when oracle/_ref
was built in this container, live calls into the reference's own functions."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

import oracle_lib as O

A, D = 1.0 / 400, 100.0


def test_philox_known_answers():
    """Random123 kat_vectors for philox4x32-10."""
    L = O.lib()

    def ph(c, k):
        c = (C.c_uint32 * 4)(*c); k = (C.c_uint32 * 2)(*k); o = (C.c_uint32 * 4)()
        L.spom_philox4x32(c, k, o)
        return [int(x) for x in o]

    assert ph([0] * 4, [0] * 2) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert ph([0xffffffff] * 4, [0xffffffff] * 2) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert ph([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_example_parse_matches_reference_echo(example_obs):
    """Stream-order parse (main_MIDASPOM.c:138-167): 8 patches x 7 years, ragged rows wrap."""
    rows = ["01111010", "0?101010", "10110101", "1011?010", "10011100", "010011?0", "00100101"]
    want = np.array([[-1 if ch == "?" else int(ch) for ch in r] for r in rows], dtype=np.int8)
    assert (example_obs == want).all()


def test_kernel_matrix_bit_exact():
    """spom_weight reproduces M[i][j]=exp(-a*(j-i)*d) (main_MIDASPOM.c:184) bit for bit."""
    n = 12
    m = O.Model(np.zeros((2, n), dtype=np.int8), spacing=D)
    M = O.ref_kernel_matrix(n, A, D)
    for i in range(n):
        for j in range(n):
            if i != j:
                assert O.lib().spom_weight(m.ref(), A, 0.0, i, j) == M[j, i]


def test_marginal_loglik_matches_reference_grid(golden, example_obs):
    """Sum over y and over the -1 completions == the reference's Lik (main_MIDASPOM.c:363-392)."""
    m = O.Model(example_obs, spacing=D, prior_occ=0.5)
    grid = [0.3, 0.5, 0.7]
    ll = np.array([[O.marginal_loglik(m, O.params(e=e, c=c, alpha=A)) for c in grid] for e in grid])
    np.testing.assert_allclose(ll, golden["loglik_s3_survey"], rtol=0, atol=2e-12)
    # and through the program's own output: table = exp(Lik - Ltot)  =>  log-ratios of entries
    tab = golden["post_s3"]
    np.testing.assert_allclose(ll - ll[0, 0], np.log(tab) - np.log(tab[0, 0]), rtol=0, atol=1e-9)
    # trapezoid normalisation (main_MIDASPOM.c:414-424)
    win = 0.2
    coef = np.outer([0.5, 1, 0.5], [0.5, 1, 0.5])
    ltot = 2 * np.log(win) + np.log((np.exp(ll) * coef).sum())
    assert abs(ltot - golden["ltot_s3"]) < 6e-6


def test_marginal_loglik_on_edges(golden, example_obs):
    """-s 11 grid over [0,1]: e=0 or c=0 rows/columns have likelihood 0 (table entry 0)."""
    m = O.Model(example_obs, spacing=D)
    tab = golden["post_s11"]
    grid = np.linspace(0, 1, 11); grid[-1] = 1.0
    ll = np.array([[O.marginal_loglik(m, O.params(e=e, c=c, alpha=A)) for c in grid] for e in grid])
    assert np.isneginf(ll[tab == 0]).all() and np.isfinite(ll[tab > 0]).all()
    win = 0.1
    coef = np.outer([0.5] + [1] * 9 + [0.5], [0.5] + [1] * 9 + [0.5])
    ltot = 2 * np.log(win) + np.log((np.exp(ll) * coef).sum())
    assert abs(ltot - golden["ltot_s11"]) < 6e-6
    np.testing.assert_allclose(np.exp(ll - ltot), tab, rtol=1e-9, atol=1e-14)


def test_transition_factors_match_compPePc(golden):
    """Every (short state i, enumerated state j) pair of the bundled example: Pe[i][j], Pc[j][i]."""
    piall, a2s = golden["cpp_piall"].astype(np.uint8), golden["cpp_all2short"]
    a, d, e, c = golden["cpp_params"]
    n = piall.shape[1]
    m = O.Model(np.zeros((2, n), dtype=np.int8), spacing=d)
    par = O.params(e=e, c=c, alpha=a)
    for tag, rtol in (("base", 1e-14), ("mpi", 1e-12)):
        Pe, Pc = golden[f"cpp_{tag}_Pe"], golden[f"cpp_{tag}_Pc"]
        for i, sid in enumerate(a2s):
            obs_state = piall[sid]
            for j in range(piall.shape[0]):
                _, pe, _ = O.transition_prob(m, par, 0, obs_state, piall[j], obs_state)
                _, _, pc = O.transition_prob(m, par, 0, np.maximum(obs_state, piall[j]), piall[j], obs_state)
                possible = not (piall[j].astype(int) * (1 - obs_state.astype(int))).any()
                if not possible:
                    assert Pe[i, j] == 0 and Pc[j, i] == 0 and pe == 0 and pc == 0
                else:
                    np.testing.assert_allclose(pe, Pe[i, j], rtol=rtol, atol=0)
                    np.testing.assert_allclose(pc, Pc[j, i], rtol=rtol, atol=1e-300)


def test_variant_terms_match_pije_pijc_pijcsource(golden):
    """dieoff.c:51-83 (E=e/K, C=c*S*K), loss.c:52-105 (source term) on 300 random triples."""
    zo, y, zn = (golden[k].astype(np.uint8) for k in ("var_zo", "var_y", "var_zn"))
    pars, res = golden["var_pars"], golden["var_res"]
    a, d = golden["var_geom"]
    n = zo.shape[1]
    m = O.Model(np.zeros((2, n), dtype=np.int8), spacing=d)
    for i in range(len(zo)):
        e, c, K, Ks, dL = pars[i]
        ones = np.ones(n, dtype=np.uint8)
        # extinction factors ignore z_new: use all-ones so feasibility depends on (z_old, y) only
        _, pe_d, _ = O.transition_prob(m, O.params(e=e, c=c, alpha=a, K=K), 1, zo[i], y[i], ones)
        _, _, pc_d = O.transition_prob(m, O.params(e=e, c=c, alpha=a, K=K), 1, ones, y[i], zn[i])
        _, pe_l, _ = O.transition_prob(m, O.params(e=e, c=c, alpha=a), 0, zo[i], y[i], ones)
        _, _, pc_l = O.transition_prob(m, O.params(e=e, c=c, alpha=a), 0, ones, y[i], zn[i])
        _, _, pc_s = O.transition_prob(m, O.params(e=e, c=c, alpha=a, K=1.0, Ksrc=Ks, dsrc=dL), 1, ones, y[i], zn[i])
        got = np.array([pe_d, pc_d, pe_l, pc_l, pc_s])
        np.testing.assert_allclose(got, res[i], rtol=1e-13, atol=0)


@pytest.mark.skipif(not O.have_ref(), reason="oracle/_ref not built (make -C oracle ref REF=<reference checkout>)")
def test_live_reference_compPePc_random():
    """Live call into the reference's compPePc on random small landscapes (not only the fixture)."""
    rng = np.random.default_rng(7)
    R = O.ref()
    u32p, dp = C.POINTER(C.c_uint32), C.POINTER(C.c_double)
    for n in (3, 5, 9):
        nstates = 2 ** n
        piall = np.array([[(i >> (n - 1 - j)) & 1 for j in range(n)] for i in range(nstates)], dtype=np.uint32)
        a2s = rng.choice(nstates, size=4, replace=False).astype(np.uint32)
        a, d, e, c = 1 / rng.uniform(100, 900), rng.uniform(50, 300), rng.uniform(0.05, 1.2), rng.uniform(0.1, 3.0)
        M = O.ref_kernel_matrix(n, a, d)
        m = O.Model(np.zeros((2, n), dtype=np.int8), spacing=d)
        par = O.params(e=e, c=c, alpha=a)
        Pe, Pc = np.zeros((4, nstates)), np.zeros((nstates, 4))
        for j in range(nstates):
            S = O.connectivity(m, a, 0.0, piall[j].astype(np.uint8))
            pC = np.minimum(1.0, c * S)
            R.ref_base_compPePc(Pe.ctypes.data_as(dp), Pc.ctypes.data_as(dp), piall.ctypes.data_as(u32p),
                                a2s.ctypes.data_as(u32p), e, pC.ctypes.data_as(dp), M.ctypes.data_as(dp), n, 4, nstates, j)
            for i, sid in enumerate(a2s):
                st = piall[sid].astype(np.uint8)
                tot, pe, pc = O.transition_prob(m, par, 0, st, piall[j].astype(np.uint8), st)
                np.testing.assert_allclose([pe, pc], [Pe[i, j], Pc[j, i]], rtol=1e-13, atol=0)


def test_complete_loglik_sums_to_marginal(example_obs):
    """log sum_{y, z_missing} exp(complete-data loglik) == marginal loglik: the augmented form is the
    reference's likelihood (SURVEY section 0 'bridge')."""
    m = O.Model(example_obs, spacing=D, prior_occ=0.5)
    par = O.params(e=0.62, c=0.41, alpha=A)
    T, n = example_obs.shape
    miss = np.argwhere(example_obs == -1)
    total = -np.inf
    for mask in range(2 ** len(miss)):
        z = (example_obs == 1).astype(np.uint8)
        for b, (t, k) in enumerate(miss):
            z[t, k] = (mask >> b) & 1
        free = [np.flatnonzero(z[t] & z[t + 1]) for t in range(T - 1)]
        # sum over y factorises over years: enumerate per year and combine in log space
        yr_tot = 0.0
        y = np.zeros((T - 1, n), dtype=np.uint8)
        base_parts = None
        lls = []
        for t in range(T - 1):
            acc = -np.inf
            for fm in range(2 ** len(free[t])):
                y[:] = 0
                for b, k in enumerate(free[t]):
                    y[t, k] = (fm >> b) & 1
                # year-t terms only: difference to the all-zero-y evaluation of other years is constant,
                # so evaluate the single-transition model instead
                mt = O.Model(np.stack([np.where(z[t], 1, 0), np.where(z[t + 1], 1, 0)]).astype(np.int8), spacing=D)
                ll, _ = O.loglik(mt, par, np.stack([z[t], z[t + 1]]), y[t:t + 1])
                acc = np.logaddexp(acc, ll)
            lls.append(acc)
        total = np.logaddexp(total, sum(lls))   # later-year missing cells have weight 1 (:386-390)
    assert abs(total - O.marginal_loglik(m, par)) < 1e-10


def test_rank1_flip_delta_equals_bruteforce():
    """spom_flip_delta (incremental) == difference of two full evaluations, incl. variants/areas."""
    rng = np.random.default_rng(3)
    n, T = 40, 5
    px, py = rng.uniform(0, 3000, n), rng.uniform(0, 3000, n)
    area = rng.lognormal(0, 0.5, n)
    z = (rng.random((T, n)) < 0.5).astype(np.uint8)
    y = (z[:-1] & z[1:] & (rng.random((T - 1, n)) < 0.6)).astype(np.uint8)
    obs = z.astype(np.int8)
    era = np.array([1, 1, 0, 0], dtype=np.uint8)
    m = O.Model(obs, geom=O.GEOM_COORDS, px=px, py=py, area=area, era=era)
    par = O.params(e=0.4, c=0.02, alpha=1 / 500, b=0.7, K=2.0, Ksrc=0.3, dsrc=40.0)
    _, _, S = O.loglik(m, par, z, y, want_S=True)
    cand = np.argwhere((z[:-1] & z[1:]) == 1)
    for t, k in cand[rng.choice(len(cand), 25, replace=False)]:
        inc = O.flip_delta(m, par, z, y, S, int(t), int(k))
        bf = O.flip_delta_bruteforce(m, par, z, y, int(t), int(k))
        assert abs(inc - bf) < 1e-9 * max(1.0, abs(bf))


def test_simulator_matches_simpij_distribution(golden):
    """spom_simulate one-year occupancy frequencies vs 10,000 draws of the reference's simpij."""
    z0 = golden["simpij_z0"].astype(np.uint8)
    e, c, K, Ks, a, d, ds = golden["simpij_pars"]
    n = len(z0)
    m = O.Model(np.zeros((2, n), dtype=np.int8), spacing=d, era=np.array([1], dtype=np.uint8))
    par = O.params(e=e, c=c, alpha=a, K=K, Ksrc=Ks, dsrc=ds)
    nsim = 20000
    acc = np.zeros(n)
    for s in range(nsim):
        acc += O.simulate(m, par, 99, s, z0, 1)[1]
    freq = acc / nsim
    se = np.sqrt(golden["simpij_freq"] * (1 - golden["simpij_freq"]) * (1 / nsim + 1 / int(golden["simpij_nsim"])))
    assert (np.abs(freq - golden["simpij_freq"]) < 4.5 * se + 1e-9).all()


def test_marginal_loglik_matches_reference_on_wide_inputs():
    """Inputs beyond the bundled example, run through the reference binary by tests/golden/make_golden_wide.py: a year with 6
    missing cells (64 completions) and a 45-year record with more than 32 distinct rows.  The oracle's marginal likelihood
    reproduces the posterior table the reference printed (density = exp(loglik - ltot))."""
    g = dict(np.load(Path(__file__).resolve().parent / "golden" / "golden_wide.npz"))
    for tag, nstep in (("a", 21), ("b", 11)):
        obs, tab, ltot = g[f"wide_{tag}_obs"].astype(np.int8), g[f"wide_{tag}_post"], float(g[f"wide_{tag}_ltot"])
        m = O.Model(obs, spacing=100.0, prior_occ=0.5)
        axis = np.linspace(0.0, 1.0, nstep)
        for ie, ic in ((nstep // 2, nstep // 2), (3, 7), (nstep - 2, 1), (1, nstep - 2)):
            ll = O.marginal_loglik(m, O.params(e=axis[ie], c=axis[ic], alpha=1.0 / 400))
            # ltot is printed with 5 decimals: exp(ll - ltot) carries a relative error of up to 5e-6 from it
            assert abs(np.exp(ll - ltot) - tab[ie, ic]) <= 6e-6 * tab[ie, ic] + 5.1e-21, (tag, ie, ic)
