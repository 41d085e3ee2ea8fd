// mp_kernels.cuh -- the CUDA kernels of the SPOM engine (sm_100a).  Included by mp_engine.cu only.
//
//  (mp_conn.cuh)   k_pack_sources, k_group_min_S, k_conn: the connectivity contraction
//  k_area_weights  aw[set][chain][l] = A_l^b (FP64) or log2 A_l^b (FP32), see pair_weight
//  k_col_ll        colonisation log-terms + per-chain segmented reduction      (compPePc:40,44)
//  k_counts        integer bookkeeping: extinction / detection / prior counts  (compPePc:38-39)
//  k_flip_delta    rank-1 log-odds of one intermediate-state flip
//  k_sweep_y       Gibbs scan of y_t | z with rank-1 updates of S_t in shared memory
//  k_update_z      Gibbs update of latent occupancy cells (conditionally independent given y)
//  k_summaries     posterior sums of z, P(z = 1 | y, theta), y and S over the chains (mp_set_summaries)
//  k_waic          sums of the pointwise predictive density of every observation, its log and squared log (mp_set_waic)
//  k_propose_* / k_decide_* / k_update_ep / k_record   Metropolis bookkeeping, one warp per chain
//  k_sim_init / k_sim_ext / k_sim_col   forward simulator (future.c:64-110)
//  k_fc_init / k_fc_ext / k_fc_col      posterior-predictive forecast from the chains (with k_pack_sources + k_conn)
//  k_ppc_obs       observations and statistics of posterior-predictive replicates of the data (mp_ppc, with the forecast's year)
#pragma once
#include "mp_device.cuh"
#include "mp_conn.cuh"   // k_pack_sources, k_group_min_S, k_conn

namespace mp {

constexpr int COL_THREADS = 256;
constexpr int MAX_COL_BLOCKS = 64;  // partial sums per chain (fixed => deterministic reduction order)
constexpr int NCOUNT = 12;          // per-chain integer counters, see k_counts
enum { CNT_N10 = 0, CNT_N10P = 1, CNT_N11 = 2, CNT_N11P = 3, CNT_BADEXT = 4, CNT_ND = 5, CNT_NM = 6,
       CNT_BADDET = 7, CNT_LAT1 = 8, CNT_LAT0 = 9, CNT_SY = 10, CNT_SZ = 11 };

template <typename R>
__global__ void k_area_weights(const mp_params *__restrict__ par, const double *__restrict__ area, R *__restrict__ aw, int n)
{
    const int c = blockIdx.y;
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= n) return;
    const double b = par[c].b;
    aw[(size_t)c * n + l] = area_pre<R>((area && b != 0.0) ? pow(area[l], b) : 1.0);
}

// ------------------------------------------------------------------ colonisation log-likelihood
// Sum over cells (t,k) with y=0 of  z'? log C : log(1-C)  (-inf for y=1,z'=0), per chain.
// Grid (nblk, chains, nsets); fixed block->cell mapping and a fixed-order second stage make the
// per-chain sum deterministic.
struct ColArgs {
    const mp_params *par[2];
    const double *S[2];
    double *partial[2];      // [chain][nblk]
};
template <typename R>
__global__ void __launch_bounds__(COL_THREADS) k_col_ll(ColArgs a, Landscape<R> ls, const uint8_t *__restrict__ z,
                                                        const uint8_t *__restrict__ y, const uint8_t *__restrict__ era,
                                                        int T)
{
    __shared__ double scratch[32];
    const int n = ls.n, c = blockIdx.y, set = blockIdx.z, ntrans = T - 1;
    const mp_params p = a.par[set][c];
    const double *S = a.S[set] + (size_t)c * ntrans * n;
    const uint8_t *zc = z + (size_t)c * T * n, *yc = y + (size_t)c * ntrans * n;
    double acc = 0.0;
    const long long cells = (long long)ntrans * n;
    const Trans<R> tr0 = make_trans<R>(p, 0), tr1 = make_trans<R>(p, 1);
    for (long long i = (long long)blockIdx.x * COL_THREADS + threadIdx.x; i < cells; i += (long long)gridDim.x * COL_THREADS) {
        const int t = (int)(i / n), k = (int)(i - (long long)t * n);
        const int zn = zc[i + n];
        if (yc[i]) { if (!zn) acc += -INFINITY; continue; }
        const Trans<R> tr = pick_trans<R>(tr0, tr1, era ? era[t] != 0 : 0);
        const R C = col_prob<R>(tr, (R)S[i], source_term<R>(ls, tr, k));
        acc += (double)log_col<R>(zn, C);
    }
    const double tot = block_sum(acc, scratch);
    if (threadIdx.x == 0) a.partial[set][(size_t)c * gridDim.x + blockIdx.x] = tot;
}
// fixed-order sum of the per-block partials of one chain by one warp
__device__ __forceinline__ double reduce_partials(const double *partial, int nblk)
{
    const int lane = threadIdx.x & 31;
    double v = 0.0;
    for (int i = lane; i < nblk; i += 32) v += partial[i];
    return warp_sum(v);
}

// ------------------------------------------------------------------ integer bookkeeping
// Per chain: extinction counts by era (#(z=1,y=0), #(z=1,y=1); compPePc:38-39), impossible cells,
// detection counts, latent year-0 cells by state, totals.  Integer atomics => order independent.
__global__ void k_counts(const int8_t *__restrict__ obs, const uint8_t *__restrict__ era, const uint8_t *__restrict__ z,
                         const uint8_t *__restrict__ y, unsigned long long *__restrict__ counts, int n, int T, int detect)
{
    __shared__ unsigned int sc[NCOUNT];
    const int c = blockIdx.y, ntrans = T - 1;
    if (threadIdx.x < NCOUNT) sc[threadIdx.x] = 0;
    __syncthreads();
    unsigned int loc[NCOUNT];
#pragma unroll
    for (int i = 0; i < NCOUNT; i++) loc[i] = 0;
    const uint8_t *zc = z + (size_t)c * T * n, *yc = y + (size_t)c * ntrans * n;
    const long long cells = (long long)T * n;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += (long long)gridDim.x * blockDim.x) {
        const int t = (int)(i / n);
        const int zz = zc[i] != 0, o = obs[i];
        loc[CNT_SZ] += zz;
        if (t < ntrans) {
            const int yy = yc[i] != 0, pre = era ? era[t] != 0 : 0;
            loc[CNT_SY] += yy;
            if (zz) { if (yy) loc[CNT_N11 + pre]++; else loc[CNT_N10 + pre]++; }
            else if (yy) loc[CNT_BADEXT]++;
        }
        if (o == 1) { if (zz) loc[CNT_ND]++; else loc[CNT_BADDET]++; }
        else if (o == 0 && zz) { if (detect) loc[CNT_NM]++; else loc[CNT_BADDET]++; }
        if (t == 0 && (o == -1 || (detect && o == 0))) { if (zz) loc[CNT_LAT1]++; else loc[CNT_LAT0]++; }
    }
#pragma unroll
    for (int i = 0; i < NCOUNT; i++) if (loc[i]) atomicAdd(&sc[i], loc[i]);
    __syncthreads();
    if (threadIdx.x < NCOUNT && sc[threadIdx.x]) atomicAdd(&counts[(size_t)c * NCOUNT + threadIdx.x], (unsigned long long)sc[threadIdx.x]);
}

__device__ __forceinline__ double xlogd(unsigned long long cnt, double v) { return cnt ? (double)cnt * log(v) : 0.0; }
__device__ inline double ll_ext_counts(const mp_params &p, const unsigned long long *cn)
{
    if (cn[CNT_BADEXT]) return -INFINITY;
    double E0 = p.e > 1.0 ? 1.0 : p.e, E1 = p.e / p.K > 1.0 ? 1.0 : p.e / p.K;
    return xlogd(cn[CNT_N10], E0) + xlogd(cn[CNT_N11], 1.0 - E0) + xlogd(cn[CNT_N10P], E1) + xlogd(cn[CNT_N11P], 1.0 - E1);
}
__device__ inline double ll_det_counts(const mp_params &p, const unsigned long long *cn, int detect)
{
    if (cn[CNT_BADDET]) return -INFINITY;
    if (!detect) return 0.0;
    return xlogd(cn[CNT_ND], p.p) + xlogd(cn[CNT_NM], 1.0 - p.p);
}
__device__ inline double ll_prior_counts(double p0, const unsigned long long *cn)
{
    return xlogd(cn[CNT_LAT1], p0) + xlogd(cn[CNT_LAT0], 1.0 - p0);
}

// ------------------------------------------------------------------ Metropolis bookkeeping (one warp per chain)
struct SamplerDev {
    mp_sampler_config sc;
    uint64_t seed;
    int chain_offset;
    int detect;
    double p0;
};
__device__ __forceinline__ double adapt_gain(uint32_t sweep) { return 1.0 / pow((double)sweep + 1.0, 0.6); }

// flags[c*4+0] = proposal in bounds, +1 = accepted, +2/+3 spare ; logu[c] = log of the MH uniform
__global__ void k_propose_ab(SamplerDev sd, const uint32_t *__restrict__ sweep_p /* device-resident sweep counter (k_advance) */, const mp_params *__restrict__ par, mp_params *__restrict__ prop,
                             const double *__restrict__ lsig, int *__restrict__ flags, double *__restrict__ logu, int nchains)
{
    const uint32_t sweep = *sweep_p;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchains) return;
    const uint4 r = rng(sd.seed, (uint32_t)(sd.chain_offset + c), sweep, RK_AB, 0, 0);
    double n1, n2;
    box_muller(r.x, r.y, n1, n2);
    mp_params q = par[c];
    if (sd.sc.sample_alpha) q.alpha = q.alpha * exp(exp(lsig[c * MP_NLSIG + 2]) * n1);
    if (sd.sc.sample_b) q.b = q.b + exp(lsig[c * MP_NLSIG + 3]) * n2;
    prop[c] = q;
    flags[c * 4 + 0] = q.alpha >= sd.sc.alpha_min && q.alpha <= sd.sc.alpha_max && q.b >= sd.sc.b_min && q.b <= sd.sc.b_max;
    flags[c * 4 + 1] = 0;
    logu[c] = log(u01(r.z));
}
// Ridge move: (alpha, b) mostly rescale S, and c S is what the data pin down.  The proposal carries
// c' = c mean(S)/mean(S') -- a deterministic, reversible shift of log c (mean S depends on (alpha, b, y)
// only) -- and the Hastings ratio gains the Jacobian c'/c of the uniform-in-c prior seen in log c.
// One CTA per chain; fixed-order sums.  ljac[c] = log(c'/c); flags[c*4+0] &= c' within bounds.
__global__ void __launch_bounds__(COL_THREADS)
k_sum_S(const double *__restrict__ S, const double *__restrict__ S2, long long cells, double *__restrict__ part0,
        double *__restrict__ part1)
{   // grid (nblk, chains, 2): partial sums of S (set 0) and S' (set 1), same block->cell map as k_col_ll
    __shared__ double scratch[32];
    const int c = blockIdx.y;
    const double *src = (blockIdx.z ? S2 : S) + (size_t)c * cells;
    double acc = 0.0;
    for (long long i = (long long)blockIdx.x * COL_THREADS + threadIdx.x; i < cells; i += (long long)gridDim.x * COL_THREADS) acc += src[i];
    const double tot = block_sum(acc, scratch);
    if (threadIdx.x == 0) (blockIdx.z ? part1 : part0)[(size_t)c * gridDim.x + blockIdx.x] = tot;
}
__global__ void k_ridge_c(SamplerDev sd, const mp_params *__restrict__ par, mp_params *__restrict__ prop,
                          const double *__restrict__ part0, const double *__restrict__ part1, int nblk,
                          int *__restrict__ flags, double *__restrict__ ljac)
{   // one warp per chain
    const int c = blockIdx.x;
    const double m1 = reduce_partials(part0 + (size_t)c * nblk, nblk), m2 = reduce_partials(part1 + (size_t)c * nblk, nblk);
    if (threadIdx.x != 0) return;
    double lj = 0.0;
    if (sd.sc.sample_c && m1 > 0.0 && m2 > 0.0) {
        const double c2 = par[c].c * (m1 / m2);
        lj = log(c2 / par[c].c);
        prop[c].c = c2;
        if (!(c2 >= sd.sc.c_min && c2 <= sd.sc.c_max)) flags[c * 4 + 0] = 0;
    }
    ljac[c] = lj;
}
// llc[c] receives the colonisation log-likelihood of the state kept
__global__ void k_decide_ab(SamplerDev sd, const uint32_t *__restrict__ sweep_p /* device-resident sweep counter (k_advance) */, mp_params *__restrict__ par, const mp_params *__restrict__ prop,
                            double *__restrict__ lsig, int *__restrict__ flags, const double *__restrict__ logu,
                            const double *__restrict__ part_cur, const double *__restrict__ part_prop, int nblk,
                            double *__restrict__ llc, int do_mh, const double *__restrict__ ljac)
{
    const uint32_t sweep = *sweep_p;
    const int c = blockIdx.x;
    const double cur = reduce_partials(part_cur + (size_t)c * nblk, nblk);
    double pr = 0.0;
    if (do_mh) pr = reduce_partials(part_prop + (size_t)c * nblk, nblk);
    if (threadIdx.x != 0) return;
    int acc = 0;
    double keep = cur;
    if (do_mh) {
        const double d = pr - cur + ljac[c];
        if (flags[c * 4 + 0] && !isnan(d) && logu[c] < d) { acc = 1; keep = pr; par[c] = prop[c]; }
        flags[c * 4 + 1] = acc;
        if (sweep < (uint32_t)sd.sc.n_adapt) {
            const double g = adapt_gain(sweep);
            if (sd.sc.sample_alpha) lsig[c * MP_NLSIG + 2] += g * (acc - 0.30);
            if (sd.sc.sample_b) lsig[c * MP_NLSIG + 3] += g * (acc - 0.30);
        }
    }
    llc[c] = keep;
}
// S_cur <- S_prop, aw_cur <- aw_prop for accepted chains
template <typename R>
__global__ void k_commit_ab(const int *__restrict__ flags, double *__restrict__ S_cur, const double *__restrict__ S_prop,
                            R *__restrict__ aw_cur, const R *__restrict__ aw_prop, long long cells, int n)
{
    const int c = blockIdx.y;
    if (!flags[c * 4 + 1]) return;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += (long long)gridDim.x * blockDim.x) {
        S_cur[(size_t)c * cells + i] = S_prop[(size_t)c * cells + i];
        if (i < n) aw_cur[(size_t)c * n + i] = aw_prop[(size_t)c * n + i];
    }
}
__global__ void k_propose_c(SamplerDev sd, const uint32_t *__restrict__ sweep_p /* device-resident sweep counter (k_advance) */, int step, const mp_params *__restrict__ par,
                            mp_params *__restrict__ prop, const double *__restrict__ lsig, int *__restrict__ flags,
                            double *__restrict__ logu, int nchains)
{
    const uint32_t sweep = *sweep_p;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchains) return;
    const uint4 r = rng(sd.seed, (uint32_t)(sd.chain_offset + c), sweep, RK_C, (uint32_t)step, 0);
    double n1, n2;
    box_muller(r.x, r.y, n1, n2);
    mp_params q = par[c];
    q.c = q.c + exp(lsig[c * MP_NLSIG + 1]) * n1;
    prop[c] = q;
    flags[c * 4 + 0] = q.c >= sd.sc.c_min && q.c <= sd.sc.c_max;
    logu[c] = log(u01(r.z));
}
__global__ void k_decide_c(SamplerDev sd, const uint32_t *__restrict__ sweep_p /* device-resident sweep counter (k_advance) */, mp_params *__restrict__ par, const mp_params *__restrict__ prop,
                           double *__restrict__ lsig, const int *__restrict__ flags, const double *__restrict__ logu,
                           const double *__restrict__ part_prop, int nblk, double *__restrict__ llc)
{
    const uint32_t sweep = *sweep_p;
    const int c = blockIdx.x;
    const double pr = reduce_partials(part_prop + (size_t)c * nblk, nblk);
    if (threadIdx.x != 0) return;
    const double d = pr - llc[c];
    int acc = 0;
    if (flags[c * 4 + 0] && !isnan(d) && logu[c] < d) { acc = 1; par[c] = prop[c]; llc[c] = pr; }
    if (sweep < (uint32_t)sd.sc.n_adapt) lsig[c * MP_NLSIG + 1] += adapt_gain(sweep) * (acc - 0.44);
}
// variant parameters: which = 0 K (log random walk), 1 Ksrc (log random walk), 2 dsrc (additive)
__global__ void k_propose_var(SamplerDev sd, const uint32_t *__restrict__ sweep_p /* device-resident sweep counter (k_advance) */, int which, int step, const mp_params *__restrict__ par,
                              mp_params *__restrict__ prop, const double *__restrict__ lsig, int *__restrict__ flags,
                              double *__restrict__ logu, int nchains)
{
    const uint32_t sweep = *sweep_p;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchains) return;
    const uint4 r = rng(sd.seed, (uint32_t)(sd.chain_offset + c), sweep, RK_K + (uint32_t)which, (uint32_t)step, 0);
    double n1, n2;
    box_muller(r.x, r.y, n1, n2);
    mp_params q = par[c];
    int inb;
    if (which == 0) { q.K = q.K * exp(exp(lsig[c * MP_NLSIG + 5]) * n1); inb = q.K >= sd.sc.K_min && q.K <= sd.sc.K_max; }
    else if (which == 1) { q.Ksrc = q.Ksrc * exp(exp(lsig[c * MP_NLSIG + 6]) * n1); inb = q.Ksrc >= sd.sc.Ksrc_min && q.Ksrc <= sd.sc.Ksrc_max; }
    else { q.dsrc = q.dsrc + exp(lsig[c * MP_NLSIG + 7]) * n1; inb = q.dsrc >= sd.sc.dsrc_min && q.dsrc <= sd.sc.dsrc_max; }
    prop[c] = q;
    flags[c * 4 + 0] = inb;
    logu[c] = log(u01(r.z));
}
__global__ void k_decide_var(SamplerDev sd, const uint32_t *__restrict__ sweep_p /* device-resident sweep counter (k_advance) */, int which, mp_params *__restrict__ par, const mp_params *__restrict__ prop,
                             double *__restrict__ lsig, const int *__restrict__ flags, const double *__restrict__ logu,
                             const double *__restrict__ part_prop, int nblk, double *__restrict__ llc,
                             const unsigned long long *__restrict__ counts)
{
    const uint32_t sweep = *sweep_p;
    const int c = blockIdx.x;
    const double pr = reduce_partials(part_prop + (size_t)c * nblk, nblk);
    if (threadIdx.x != 0) return;
    const unsigned long long *cn = counts + (size_t)c * NCOUNT;
    const double d = (pr - llc[c]) + (ll_ext_counts(prop[c], cn) - ll_ext_counts(par[c], cn));
    int acc = 0;
    if (flags[c * 4 + 0] && !isnan(d) && logu[c] < d) { acc = 1; par[c] = prop[c]; llc[c] = pr; }
    if (sweep < (uint32_t)sd.sc.n_adapt) lsig[c * MP_NLSIG + 5 + which] += adapt_gain(sweep) * (acc - 0.44);
}
// e and p from the sufficient counts: random-walk MH sub-steps, one thread per chain
__global__ void k_update_ep(SamplerDev sd, const uint32_t *__restrict__ sweep_p /* device-resident sweep counter (k_advance) */, mp_params *__restrict__ par, double *__restrict__ lsig,
                            const unsigned long long *__restrict__ counts, int nchains)
{
    const uint32_t sweep = *sweep_p;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchains) return;
    const unsigned long long *cn = counts + (size_t)c * NCOUNT;
    mp_params p = par[c];
    const bool adapting = sweep < (uint32_t)sd.sc.n_adapt;
    const double g = adapt_gain(sweep);
    if (sd.sc.sample_e) {
        double ll = ll_ext_counts(p, cn), ls = lsig[c * MP_NLSIG + 0];
        for (int s = 0; s < sd.sc.n_e_steps; s++) {
            const uint4 r = rng(sd.seed, (uint32_t)(sd.chain_offset + c), sweep, RK_E, (uint32_t)s, 0);
            double n1, n2;
            box_muller(r.x, r.y, n1, n2);
            mp_params q = p;
            q.e = p.e + exp(ls) * n1;
            int acc = 0;
            if (q.e >= sd.sc.e_min && q.e <= sd.sc.e_max) {
                const double l2 = ll_ext_counts(q, cn), d = l2 - ll;
                if (!isnan(d) && log(u01(r.z)) < d) { acc = 1; p = q; ll = l2; }
            }
            if (adapting) ls += g * (acc - 0.44);
        }
        lsig[c * MP_NLSIG + 0] = ls;
    }
    if (sd.sc.sample_p && sd.detect) {
        double ll = ll_det_counts(p, cn, 1), ls = lsig[c * MP_NLSIG + 4];
        for (int s = 0; s < sd.sc.n_e_steps; s++) {
            const uint4 r = rng(sd.seed, (uint32_t)(sd.chain_offset + c), sweep, RK_P, (uint32_t)s, 0);
            double n1, n2;
            box_muller(r.x, r.y, n1, n2);
            mp_params q = p;
            q.p = p.p + exp(ls) * n1;
            int acc = 0;
            if (q.p >= sd.sc.p_min && q.p <= sd.sc.p_max) {
                const double l2 = ll_det_counts(q, cn, 1), d = l2 - ll;
                if (!isnan(d) && log(u01(r.z)) < d) { acc = 1; p = q; ll = l2; }
            }
            if (adapting) ls += g * (acc - 0.44);
        }
        lsig[c * MP_NLSIG + 4] = ls;
    }
    par[c] = p;
}
// draws[c] = (e, c, alpha, b, p, loglik, #y=1, #z=1); parts (nullable) = ext, col, prior, det
// ctr (nullable): {sweep, recorded draws}; with it the row is draws + ctr[1] * chains * MP_NDRAW while ctr[1] < max_draws
__global__ void k_record(SamplerDev sd, const mp_params *__restrict__ par, const unsigned long long *__restrict__ counts,
                         const double *__restrict__ part_cur, int nblk, double *__restrict__ draw, double *__restrict__ parts,
                         const uint32_t *__restrict__ ctr, int max_draws)
{
    const int c = blockIdx.x;
    if (ctr) draw = (int)ctr[1] < max_draws ? draw + (size_t)ctr[1] * gridDim.x * MP_NDRAW : nullptr;
    const double lc = reduce_partials(part_cur + (size_t)c * nblk, nblk);
    if (threadIdx.x != 0) return;
    const unsigned long long *cn = counts + (size_t)c * NCOUNT;
    const mp_params p = par[c];
    const double le = ll_ext_counts(p, cn), lp = ll_prior_counts(sd.p0, cn), ld = ll_det_counts(p, cn, sd.detect);
    if (draw) {
        double *d = draw + (size_t)c * MP_NDRAW;
        d[0] = p.e; d[1] = p.c; d[2] = p.alpha; d[3] = p.b; d[4] = p.p; d[5] = le + lc + lp + ld;
        d[6] = (double)cn[CNT_SY]; d[7] = (double)cn[CNT_SZ]; d[8] = p.K; d[9] = p.Ksrc; d[10] = p.dsrc;
    }
    if (parts) { double *q = parts + (size_t)c * MP_NPART; q[0] = le; q[1] = lc; q[2] = lp; q[3] = ld; }
}

// end of a sweep: the device-resident counters every kernel of the next sweep reads (so that a captured sweep can be replayed)
static __global__ void k_advance(uint32_t *__restrict__ ctr, int max_draws)
{
    if ((int)ctr[1] < max_draws) ctr[1]++;
    ctr[0]++;
}

// ------------------------------------------------------------------ latent occupancy cells
// Log-odds of z_tk = 1 given y and theta for a latent cell (observation o) that no adjacent y = 1 forces: colonisation
// term of t-1 -> t, extinction term of t -> t+1, year-0 prior, missed detection.  The colonisation and extinction terms are
// formed in R, the rest in FP64.  Shared by the Gibbs draw (k_update_z) and its Rao-Blackwellised mean (k_summaries) so that
// both see the same number.  Sc: the chain's S [transition][patch]; i = t n + k.
template <typename R>
__device__ __forceinline__ double z_logodds(const SamplerDev &sd, const Landscape<R> &ls, const mp_params &p, const Trans<R> &tr0,
                                            const Trans<R> &tr1, const uint8_t *__restrict__ era, const double *__restrict__ Sc,
                                            int o, long long i, int t, int k, int ntrans)
{
    R lo = 0;
    if (t > 0) {
        const Trans<R> tr = pick_trans<R>(tr0, tr1, era ? era[t - 1] != 0 : 0);
        const R C = col_prob<R>(tr, (R)Sc[i - ls.n], source_term<R>(ls, tr, k));
        lo += Num<R>::logv(C) - Num<R>::log1m(C);
    }
    if (t < ntrans) lo += (era && era[t]) ? tr1.logE : tr0.logE;
    double lod = (double)lo;
    if (t == 0) lod += log(sd.p0) - log(1.0 - sd.p0);
    if (sd.detect && o == 0) lod += log(1.0 - p.p);
    return lod;
}
// Log predictive density of the observation o (0 or 1) of cell (t, k) given the chain's state of the previous year (DESIGN
// §2, WAIC): pi = p0 in year 0; for t >= 1 pi = s + (1 - s) C with s = z_{t-1,k} (1 - E_{t-1}), which marginalises the
// patch's own y_{t-1,k} (S excludes the patch itself).  C is formed in R exactly as z_logodds forms it, the rest in FP64;
// p = q pi for o = 1, 1 - q pi for o = 0 (its log by log1p), q the detection probability (1 without detection).  Returns
// log p and writes p to dens.
template <typename R>
__device__ __forceinline__ double obs_logpred(const SamplerDev &sd, const Landscape<R> &ls, const mp_params &p, const Trans<R> &tr0,
                                              const Trans<R> &tr1, const uint8_t *__restrict__ era, const double *__restrict__ Sc,
                                              int o, bool zprev, long long i, int t, int k, double &dens)
{
    double pi = sd.p0;
    if (t > 0) {
        const bool pre = era ? era[t - 1] != 0 : false;
        const Trans<R> tr = pick_trans<R>(tr0, tr1, pre);
        const double C = (double)col_prob<R>(tr, (R)Sc[i - ls.n], source_term<R>(ls, tr, k));
        double E = pre ? p.e / p.K : p.e;
        if (E > 1.0) E = 1.0;
        const double s = zprev ? 1.0 - E : 0.0;
        pi = s + (1.0 - s) * C;
    }
    const double qpi = sd.detect ? p.p * pi : pi;
    dens = o ? qpi : 1.0 - qpi;
    return o ? log(qpi) : log1p(-qpi);
}
// z_tk | y, theta for every latent cell at once: S depends on y only, so the cells are
// conditionally independent.  Forced to 1 when an adjacent intermediate state is 1.
template <typename R>
__global__ void k_update_z(SamplerDev sd, const uint32_t *__restrict__ sweep_p /* device-resident sweep counter (k_advance) */, Landscape<R> ls, const mp_params *__restrict__ par,
                           const int8_t *__restrict__ obs, const uint8_t *__restrict__ era, uint8_t *__restrict__ z,
                           const uint8_t *__restrict__ y, const double *__restrict__ S, int T)
{
    const uint32_t sweep = *sweep_p;
    const int n = ls.n, c = blockIdx.y, ntrans = T - 1;
    const long long cells = (long long)T * n;
    const mp_params p = par[c];
    uint8_t *zc = z + (size_t)c * cells;
    const uint8_t *yc = y + (size_t)c * ntrans * n;
    const double *Sc = S + (size_t)c * ntrans * n;
    const Trans<R> tr0 = make_trans<R>(p, 0), tr1 = make_trans<R>(p, 1);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += (long long)gridDim.x * blockDim.x) {
        const int o = obs[i];
        if (!(o == -1 || (sd.detect && o == 0))) continue;
        const int t = (int)(i / n), k = (int)(i - (long long)t * n);
        const bool forced = (t > 0 && yc[i - n]) || (t < ntrans && yc[i]);
        if (forced) { zc[i] = 1; continue; }
        const double lod = z_logodds<R>(sd, ls, p, tr0, tr1, era, Sc, o, i, t, k, ntrans);
        const uint4 r = rng(sd.seed, (uint32_t)(sd.chain_offset + c), sweep, RK_Z, (uint32_t)k, (uint32_t)t);
        zc[i] = isnan(lod) ? 0 : (logit_u(r.x) < lod);
    }
}

// ------------------------------------------------------------------ posterior summaries of the latent state (mp_set_summaries)
// Sums over this engine's chains, added at the end of every sweep s with s >= first and (s - first) % thin == 0 (the sweep
// counter is read on the device, so a captured sweep replays unchanged).  Layout [year][patch]; y_count and S_sum have T-1 rows.
struct SumBufs {
    double *z_prob, *S_sum;
    uint32_t *z_count, *y_count;
    unsigned long long *nsamples;
};
// whether sweep s adds to sums set with (first, thin > 0): the gate of k_summaries and k_waic
__device__ __forceinline__ bool sweep_due(uint32_t s, int first, int thin)
{
    return s >= (uint32_t)first && (s - (uint32_t)first) % (uint32_t)thin == 0;
}
// 4 bytes of a row of z or y, byte j = patch k0 + j (m <= 4 valid patches); rows start on a 4-byte boundary when n % 4 == 0
__device__ __forceinline__ uint32_t load_cells4(const uint8_t *__restrict__ p, int m, bool words)
{
    if (words) return *reinterpret_cast<const uint32_t *>(p);
    uint32_t v = 0;
    for (int j = 0; j < m; j++) v |= (uint32_t)p[j] << (8 * j);
    return v;
}
// One thread per (year, 4 consecutive patches) visits the chains in order c = 0 .. C-1 and read-modify-writes only its own
// cells: no atomics, and every sum is the same whatever the launch geometry.  z_prob adds P(z_tk = 1 | y, theta) for the latent
// cells (1 when forced, 0 for a NaN log-odds, as k_update_z draws there) and the indicator for the cells the data fix.
template <typename R>
__global__ void __launch_bounds__(256)
k_summaries(SamplerDev sd, const uint32_t *__restrict__ sweep_p /* device-resident sweep counter (k_advance) */, int first, int thin,
            Landscape<R> ls, const mp_params *__restrict__ par, const int8_t *__restrict__ obs, const uint8_t *__restrict__ era,
            const uint8_t *__restrict__ z, const uint8_t *__restrict__ y, const double *__restrict__ S, int T, int nchains, SumBufs b)
{
    if (!sweep_due(*sweep_p, first, thin)) return;
    const int n = ls.n, ntrans = T - 1, nq = (n + 3) >> 2;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx == 0) *b.nsamples += (unsigned long long)nchains;
    if (idx >= (long long)T * nq) return;
    const int t = (int)(idx / nq), k0 = 4 * (int)(idx - (long long)t * nq), m = min(4, n - k0);
    const bool words = (n & 3) == 0, has_y = t < ntrans;
    const size_t row = (size_t)t * n + k0;
    int o[4];
    bool latent[4], any_latent = false;
    uint32_t zc[4] = { 0, 0, 0, 0 }, yc[4] = { 0, 0, 0, 0 };
    double zp[4] = { 0, 0, 0, 0 }, ss[4] = { 0, 0, 0, 0 };
#pragma unroll
    for (int j = 0; j < 4; j++) {
        o[j] = j < m ? obs[row + j] : 1;
        latent[j] = o[j] == -1 || (sd.detect && o[j] == 0);
        any_latent |= latent[j];
        if (j < m) {
            zc[j] = b.z_count[row + j]; zp[j] = b.z_prob[row + j];
            if (has_y) { yc[j] = b.y_count[row + j]; ss[j] = b.S_sum[row + j]; }
        }
    }
    for (int c = 0; c < nchains; c++) {
        const uint8_t *zch = z + (size_t)c * T * n, *ych = y + (size_t)c * ntrans * n;
        const double *Sc = S + (size_t)c * ntrans * n;
        const uint32_t zw = load_cells4(zch + row, m, words);
        const uint32_t yw = has_y ? load_cells4(ych + row, m, words) : 0u;
        const uint32_t yprev = t > 0 ? load_cells4(ych + row - n, m, words) : 0u;
        mp_params p;
        Trans<R> tr0, tr1;
        if (any_latent) { p = par[c]; tr0 = make_trans<R>(p, 0); tr1 = make_trans<R>(p, 1); }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (j >= m) continue;
            const uint32_t zz = ((zw >> (8 * j)) & 0xffu) != 0u;
            double pr = (double)zz;
            if (latent[j]) {
                if (((yw | yprev) >> (8 * j)) & 0xffu) pr = 1.0;
                else {
                    const double lod = z_logodds<R>(sd, ls, p, tr0, tr1, era, Sc, o[j], (long long)(row + j), t, k0 + j, ntrans);
                    pr = isnan(lod) ? 0.0 : 1.0 / (1.0 + exp(-lod));
                }
            }
            zc[j] += zz; zp[j] += pr;
            if (has_y) { yc[j] += ((yw >> (8 * j)) & 0xffu) != 0u; ss[j] += Sc[row + j]; }
        }
    }
#pragma unroll
    for (int j = 0; j < 4; j++)
        if (j < m) {
            b.z_count[row + j] = zc[j]; b.z_prob[row + j] = zp[j];
            if (has_y) { b.y_count[row + j] = yc[j]; b.S_sum[row + j] = ss[j]; }
        }
}

// ------------------------------------------------------------------ pointwise predictive densities for WAIC (mp_set_waic)
// Sums over this engine's chains and the qualifying sweeps (the gate of k_summaries), per observed cell (obs 0 or 1):
// lik = sum p, loglik = sum log p, loglik_sq = sum (log p)^2, p from obs_logpred.  Layout [year][patch]; cells that are
// not observations are never written.
struct WaicBufs {
    double *lik, *loglik, *loglik_sq;
    unsigned long long *nsamples;
};
// One thread per (year, 4 consecutive patches), the chains in order c = 0 .. C-1, only its own cells: no atomics, the sums
// do not depend on the launch geometry.  Reads z of the previous year and S of the previous transition.
template <typename R>
__global__ void __launch_bounds__(256)
k_waic(SamplerDev sd, const uint32_t *__restrict__ sweep_p /* device-resident sweep counter (k_advance) */, int first, int thin,
       Landscape<R> ls, const mp_params *__restrict__ par, const int8_t *__restrict__ obs, const uint8_t *__restrict__ era,
       const uint8_t *__restrict__ z, const double *__restrict__ S, int T, int nchains, WaicBufs b)
{
    if (!sweep_due(*sweep_p, first, thin)) return;
    const int n = ls.n, ntrans = T - 1, nq = (n + 3) >> 2;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx == 0) *b.nsamples += (unsigned long long)nchains;
    if (idx >= (long long)T * nq) return;
    const int t = (int)(idx / nq), k0 = 4 * (int)(idx - (long long)t * nq), m = min(4, n - k0);
    const bool words = (n & 3) == 0;
    const size_t row = (size_t)t * n + k0;
    int o[4];
    bool any = false;
    double L[4] = { 0, 0, 0, 0 }, G[4] = { 0, 0, 0, 0 }, Q[4] = { 0, 0, 0, 0 };
#pragma unroll
    for (int j = 0; j < 4; j++) {
        o[j] = j < m ? obs[row + j] : -1;
        if (o[j] >= 0) { any = true; L[j] = b.lik[row + j]; G[j] = b.loglik[row + j]; Q[j] = b.loglik_sq[row + j]; }
    }
    if (!any) return;
    for (int c = 0; c < nchains; c++) {
        const uint32_t zprev = t > 0 ? load_cells4(z + (size_t)c * T * n + row - n, m, words) : 0u;
        const double *Sc = S + (size_t)c * ntrans * n;
        const mp_params p = par[c];
        const Trans<R> tr0 = make_trans<R>(p, 0), tr1 = make_trans<R>(p, 1);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (o[j] < 0) continue;
            double pd;
            const double lp = obs_logpred<R>(sd, ls, p, tr0, tr1, era, Sc, o[j], ((zprev >> (8 * j)) & 0xffu) != 0u,
                                             (long long)(row + j), t, k0 + j, pd);
            L[j] += pd; G[j] += lp; Q[j] += lp * lp;
        }
    }
#pragma unroll
    for (int j = 0; j < 4; j++)
        if (o[j] >= 0) { b.lik[row + j] = L[j]; b.loglik[row + j] = G[j]; b.loglik_sq[row + j] = Q[j]; }
}

// ------------------------------------------------------------------ rank-1 flip of the intermediate state
// Contribution of target q to the log-odds of flipping source k (current value cur), and the
// updated (S, L) of q.  Shared by k_flip_delta and k_sweep_y so both use identical arithmetic.
template <typename R, int GEOM>
__device__ __forceinline__ R flip_pair(const Landscape<R> &ls, const Trans<R> &tr, R awk, int k, R kx, R ky, int q,
                                       int cur, bool zero_after, double Sq, int yq, int znq, R Lq, bool haveL,
                                       double &S_alt, R &L_alt)
{
    R qx = 0, qy = 0;
    if (GEOM == MP_GEOM_COORDS) { qx = ls.px[q]; qy = ls.py[q]; }
    const R w = pair_weight<R, GEOM>(ls, alpha_pre<R>((double)tr.alpha), awk, q, k, qx, qy, kx, ky);
    double sa = cur ? Sq - (double)w : Sq + (double)w;
    if (zero_after || sa < 0.0) sa = 0.0;
    S_alt = sa;
    if (yq) { L_alt = 0; return 0; }
    const R g = source_term<R>(ls, tr, q);
    const R la = log_col<R>(znq, col_prob<R>(tr, (R)sa, g));
    const R lc = haveL ? Lq : log_col<R>(znq, col_prob<R>(tr, (R)Sq, g));
    L_alt = la;
    return ldiff<R>(la, lc);
}
// own-cell term of candidate k (z_t = z_t+1 = 1): y=1 -> log(1-E) ; y=0 -> log E + log C_k
template <typename R>
__device__ __forceinline__ R flip_own(const Landscape<R> &ls, const Trans<R> &tr, int k, int cur, double Sk)
{
    const R l1 = tr.log1mE;
    const R l0 = tr.logE + Num<R>::logv(col_prob<R>(tr, (R)Sk, source_term<R>(ls, tr, k)));
    return cur ? ldiff<R>(l0, l1) : ldiff<R>(l1, l0);
}

template <typename R, int GEOM>
__global__ void k_flip_delta(Landscape<R> ls, const mp_params *__restrict__ par, const R *__restrict__ aw,
                             const uint8_t *__restrict__ era, const uint8_t *__restrict__ z, const uint8_t *__restrict__ y,
                             const double *__restrict__ S, int T, int c, int t, int k, double *__restrict__ out)
{
    __shared__ double scratch[32];
    const int n = ls.n, ntrans = T - 1;
    const Trans<R> tr = make_trans<R>(par[c], era ? era[t] : 0);
    const uint8_t *yt = y + ((size_t)c * ntrans + t) * n, *zn = z + ((size_t)c * T + t + 1) * n;
    const double *St = S + ((size_t)c * ntrans + t) * n;
    const int cur = yt[k];
    int nocc = 0;
    for (int q = threadIdx.x; q < n; q += blockDim.x) nocc += yt[q];
    nocc = (int)(block_sum((double)nocc, scratch) + 0.5);
    __syncthreads();
    const bool zero_after = (nocc + (cur ? -1 : 1)) == 0;
    R kx = 0, ky = 0;
    if (GEOM == MP_GEOM_COORDS) { kx = ls.px[k]; ky = ls.py[k]; }
    const R awk = aw[(size_t)c * n + k];
    double acc = 0.0;
    for (int q = threadIdx.x; q < n; q += blockDim.x) {
        if (q == k) { acc += (double)flip_own<R>(ls, tr, k, cur, St[k]); continue; }
        double sa; R la;
        acc += (double)flip_pair<R, GEOM>(ls, tr, awk, k, kx, ky, q, cur, zero_after, St[q], yt[q], zn[q], (R)0, false, sa, la);
    }
    const double tot = block_sum(acc, scratch);
    if (threadIdx.x == 0) *out = isnan(tot) ? -INFINITY : tot;
}

// One CTA per (chain, transition): S_t (FP64), the cached log-terms L (R) and the cell flags live
// in shared memory for the whole scan.  Candidates (z_t = z_t+1 = 1) are visited in patch order;
// each visit evaluates the N-wide rank-1 change, reduces it in a fixed order, and every thread
// takes the same decision from logit(u) < delta with u = Philox(seed, chain, sweep, RK_Y, k, t).
template <typename R, int GEOM, int NT>
__global__ void __launch_bounds__(NT, 1)
k_sweep_y(SamplerDev sd, const uint32_t *__restrict__ sweep_p /* device-resident sweep counter (k_advance) */, Landscape<R> ls, const mp_params *__restrict__ par, const R *__restrict__ aw,
          const uint8_t *__restrict__ era, const uint8_t *__restrict__ z, uint8_t *__restrict__ y, double *__restrict__ S, int T,
          const int *__restrict__ order /* visiting order of the scan: slot -> patch (oracle: spom_scan_order) */,
          unsigned long long *__restrict__ stats,
          unsigned char *__restrict__ work /* landscapes beyond one CTA's shared memory: per-task scratch in global memory (L2 resident), else nullptr */,
          size_t work_stride)
{
    const uint32_t sweep = *sweep_p;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = ls.n, ntrans = T - 1, tid = threadIdx.x, nthr = blockDim.x;
    const int c = blockIdx.x / ntrans, t = blockIdx.x - c * ntrans;
    // every thread reads and writes only its own targets q = tid, tid + nthr, ...; the candidate's own cell is read by all
    // threads but written once, before the block barrier that precedes its visit -- so global scratch needs no more fences
    double *sS = reinterpret_cast<double *>(work ? work + (size_t)blockIdx.x * work_stride : smem_raw);
    R *sL = reinterpret_cast<R *>(sS + n);
    uint8_t *sF = reinterpret_cast<uint8_t *>(sL + n);        // bit0 y, bit1 z_t, bit2 z_t+1
    __shared__ double warp_part[2][32];
    __shared__ double thr_slot[2];
    __shared__ double scratch[32];

    const Trans<R> tr = make_trans<R>(par[c], era ? era[t] : 0);
    uint8_t *yt = y + ((size_t)c * ntrans + t) * n;
    const uint8_t *zt = z + ((size_t)c * T + t) * n, *zn = zt + n;
    double *St = S + ((size_t)c * ntrans + t) * n;
    const R *awc = aw + (size_t)c * n;

    int nocc_loc = 0;
    for (int q = tid; q < n; q += nthr) {
        const int yq = yt[q] != 0, znq = zn[q] != 0;
        const double s = St[q];
        sS[q] = s;
        sF[q] = (uint8_t)(yq | ((zt[q] != 0) << 1) | (znq << 2));
        sL[q] = yq ? (R)0 : log_col<R>(znq, col_prob<R>(tr, (R)s, source_term<R>(ls, tr, q)));
        nocc_loc += yq;
    }
    int nocc = (int)(block_sum((double)nocc_loc, scratch) + 0.5);
    __syncthreads();

    const uint32_t gchain = (uint32_t)(sd.chain_offset + c);
    int it = 0;
    for (int sl = 0; sl < n; sl++) {
        const int k = order[sl];
        const int fk = sF[k];
        if ((fk & 6) != 6) continue;                    // candidate iff z_t[k] = z_t+1[k] = 1
        const int par_i = it & 1; it++;
        const int cur = fk & 1;
        const bool zero_after = (nocc + (cur ? -1 : 1)) == 0;
        if (tid == 0) thr_slot[par_i] = logit_u(rng(sd.seed, gchain, sweep, RK_Y, (uint32_t)k, (uint32_t)t).x);
        R kx = 0, ky = 0;
        if (GEOM == MP_GEOM_COORDS) { kx = ls.px[k]; ky = ls.py[k]; }
        const R awk = awc[k];
        double acc = 0.0;
        for (int q = tid; q < n; q += nthr) {
            if (q == k) { acc += (double)flip_own<R>(ls, tr, k, cur, sS[k]); continue; }
            double sa; R la;
            const int fq = sF[q];
            acc += (double)flip_pair<R, GEOM>(ls, tr, awk, k, kx, ky, q, cur, zero_after, sS[q], fq & 1, (fq >> 2) & 1,
                                              sL[q], true, sa, la);
        }
        // fixed-order block reduction; every warp redoes the final tree so all threads agree
        const int lane = tid & 31, wid = tid >> 5, nw = (nthr + 31) >> 5;
        acc = warp_sum(acc);
        if (lane == 0) warp_part[par_i][wid] = acc;
        __syncthreads();
        double tot = warp_sum(lane < nw ? warp_part[par_i][lane] : 0.0);
        if (isnan(tot)) tot = -INFINITY;
        const bool flip = thr_slot[par_i] < tot;
        if (flip) {
            // recompute and commit: each thread rewrites the (S, L) of its own targets
            for (int q = tid; q < n; q += nthr) {
                if (q == k) { sF[k] = (uint8_t)(fk ^ 1);
                              sL[k] = cur ? log_col<R>(1, col_prob<R>(tr, (R)sS[k], source_term<R>(ls, tr, k))) : (R)0;
                              continue; }
                double sa; R la;
                const int fq = sF[q];
                flip_pair<R, GEOM>(ls, tr, awk, k, kx, ky, q, cur, zero_after, sS[q], fq & 1, (fq >> 2) & 1, sL[q], true, sa, la);
                sS[q] = sa;
                if (!(fq & 1)) sL[q] = la;
            }
            nocc += cur ? -1 : 1;
        }
    }
    __syncthreads();
    for (int q = tid; q < n; q += nthr) { St[q] = sS[q]; yt[q] = sF[q] & 1; }
    if (stats && tid == 0) atomicAdd(&stats[MP_CNT_SCAN_DENSE], (unsigned long long)it * (unsigned long long)n);
}

// ------------------------------------------------------------------ forward simulator
// Forward simulator (future.c:359-386 loops over simulations; simpij :64-110 is one year): survive iff u > E (:78),
// colonise iff u < C (:100).  One year = two launches over all trajectories:
//   k_sim_ext   one CTA per trajectory: extinction draws and the ORDERED list of the surviving sources (ascending patch
//               number, the order in which simpij and the CPU twin accumulate S)
//   k_sim_col   grid (target tiles, trajectories): S of 128 targets from the survivor list staged through shared memory
//               (coordinates and A_l^b, precomputed once per parameter set by k_area_weights), then the colonisation draws
// so a single large landscape spreads over the whole GPU (synth.make_workload_large generates cfg5 with it).
static __global__ void __launch_bounds__(256)
k_sim_init(const uint8_t *__restrict__ z0_all, int per_sim, int n, int nyears, uint8_t *__restrict__ zc, uint8_t *__restrict__ z_out,
           int32_t *__restrict__ occ_out)
{
    __shared__ double scratch[32];
    const uint8_t *z0 = z0_all + (per_sim ? (size_t)blockIdx.x * n : 0);
    int cnt = 0;
    for (int k = threadIdx.x; k < n; k += blockDim.x) {
        const uint8_t v = z0[k] != 0;
        zc[(size_t)blockIdx.x * n + k] = v; cnt += v;
        if (z_out) z_out[(size_t)blockIdx.x * (nyears + 1) * n + k] = v;
    }
    cnt = (int)(block_sum((double)cnt, scratch) + 0.5);
    if (threadIdx.x == 0 && occ_out) occ_out[(size_t)blockIdx.x * (nyears + 1)] = cnt;
}
template <typename R>
__global__ void __launch_bounds__(1024)
k_sim_ext(const mp_params *__restrict__ pars, int per_sim, int n, uint64_t seed, uint32_t sim0, int t, int era_all,
          const uint8_t *__restrict__ zc, uint8_t *__restrict__ yc, int *__restrict__ list, int *__restrict__ nlist)
{
    __shared__ int s_cnt[1024];
    const int tid = threadIdx.x;
    const uint32_t sim = sim0 + blockIdx.x;
    const Trans<R> tr = make_trans<R>(pars[per_sim ? blockIdx.x : 0], era_all);
    const uint8_t *z = zc + (size_t)blockIdx.x * n;
    uint8_t *y = yc + (size_t)blockIdx.x * n;
    const int per = (n + 1023) / 1024, k0 = min(n, tid * per), k1 = min(n, k0 + per);
    int cnt = 0;
    for (int k = k0; k < k1; k++) {
        const uint4 r = rng(seed, sim, (uint32_t)t, RK_SIM_EXT, (uint32_t)k, 0);
        const uint8_t v = z[k] && (u01(r.x) > (double)tr.E);
        y[k] = v; cnt += v;
    }
    s_cnt[tid] = cnt;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {                  // inclusive Hillis-Steele scan
        const int v = tid >= o ? s_cnt[tid - o] : 0;
        __syncthreads();
        s_cnt[tid] += v;
        __syncthreads();
    }
    int off = s_cnt[tid] - cnt;
    int *out = list + (size_t)blockIdx.x * n;
    for (int k = k0; k < k1; k++) if (y[k]) out[off++] = k;
    if (tid == 1023) nlist[blockIdx.x] = s_cnt[1023];
}
template <typename R, int GEOM>
__global__ void __launch_bounds__(128)
k_sim_col(Landscape<R> ls, const mp_params *__restrict__ pars, int per_sim, const R *__restrict__ aw /* [parameter set][n] */,
          const uint8_t *__restrict__ yc, const int *__restrict__ list, const int *__restrict__ nlist, uint64_t seed, uint32_t sim0,
          int t, int nyears, int era_all, uint8_t *__restrict__ zc, uint8_t *__restrict__ z_out, int32_t *__restrict__ occ_out)
{
    __shared__ int s_l[128];
    __shared__ R s_x[128], s_y[128], s_a[128];
    const int n = ls.n, tid = threadIdx.x, k = blockIdx.x * 128 + tid, si = blockIdx.y;
    const uint32_t sim = sim0 + si;
    const mp_params p = pars[per_sim ? si : 0];
    const Trans<R> tr = make_trans<R>(p, era_all);
    const R apre = alpha_pre<R>(p.alpha);
    const R *awp = aw + (per_sim ? (size_t)si * n : 0);
    const int *src = list + (size_t)si * n, ns = nlist[si];
    const int kq = min(k, n - 1);
    R kx = 0, ky = 0;
    if (GEOM == MP_GEOM_COORDS) { kx = ls.px[kq]; ky = ls.py[kq]; }
    double s = 0.0;
    for (int j0 = 0; j0 < ns; j0 += 128) {
        __syncthreads();
        if (j0 + tid < ns) {
            const int l = src[j0 + tid];
            s_l[tid] = l; s_a[tid] = awp[l];
            if (GEOM == MP_GEOM_COORDS) { s_x[tid] = ls.px[l]; s_y[tid] = ls.py[l]; }
        }
        __syncthreads();
        const int m = min(128, ns - j0);
        for (int j = 0; j < m; j++) {                     // ascending l: the accumulation order of simpij / the CPU twin
            const int l = s_l[j];
            if (l == kq) continue;
            s += (double)pair_weight<R, GEOM>(ls, apre, s_a[j], kq, l, kx, ky, GEOM == MP_GEOM_COORDS ? s_x[j] : (R)0, GEOM == MP_GEOM_COORDS ? s_y[j] : (R)0);
        }
    }
    int v = 0;
    if (k < n) {
        const R C = col_prob<R>(tr, (R)s, source_term<R>(ls, tr, k));
        const uint4 r = rng(seed, sim, (uint32_t)t, RK_SIM_COL, (uint32_t)k, 0);
        v = yc[(size_t)si * n + k] ? 1 : (u01(r.x) < (double)C);
        zc[(size_t)si * n + k] = (uint8_t)v;              // zc is only read through yc in this launch
        if (z_out) z_out[((size_t)si * (nyears + 1) + t + 1) * n + k] = (uint8_t)v;
    }
    const int c2 = __reduce_add_sync(0xffffffffu, v);
    if ((tid & 31) == 0 && occ_out && c2) atomicAdd(&occ_out[(size_t)si * (nyears + 1) + t + 1], c2);
}

// ------------------------------------------------------------------ posterior-predictive forecast (mp_forecast) and replicates (mp_ppc)
// nrep trajectories per chain from the chain's own z[c][t0] and parameters, states laid out [chain][replicate][patch]
// (t0 = T-1 for the forecast, 0 for the replicates of the data).
// Trajectory (c, r) is simulation number sim0 + c * nrep + r of mp_simulate_ensemble: the same Philox draws per patch number.
// One year = k_fc_ext, then S of every (chain, replicate) from k_conn with the replicates in place of the years (k_pack_sources
// packs 32 replicates per record word), then k_fc_col.
//   k_fc_init  grid (patch tiles, chains): start states, year-0 counts and incidence
static __global__ void __launch_bounds__(256)
k_fc_init(const uint8_t *__restrict__ z, int T, int t0, int n, int nrep, int nyears, uint8_t *__restrict__ zc, int32_t *__restrict__ occ,
          uint32_t *__restrict__ inc)
{
    __shared__ int s_cnt;
    const int c = blockIdx.y, k = blockIdx.x * 256 + threadIdx.x;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    int v = 0;
    if (k < n) {
        v = z[((size_t)c * T + t0) * n + k] != 0;
        for (int r = 0; r < nrep; r++) zc[((size_t)c * nrep + r) * n + k] = (uint8_t)v;
        if (inc && v) atomicAdd(&inc[k], (uint32_t)nrep);
    }
    const int w = __reduce_add_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && w) atomicAdd(&s_cnt, w);
    __syncthreads();
    if (occ && s_cnt)
        for (int r = threadIdx.x; r < nrep; r += blockDim.x) atomicAdd(&occ[((size_t)c * nrep + r) * (nyears + 1)], s_cnt);
}
//   k_fc_ext   grid (patch tiles, replicates, chains): survive iff u > E, u keyed by (sim, year, patch number) as in k_sim_ext
template <typename R>
__global__ void __launch_bounds__(256)
k_fc_ext(const mp_params *__restrict__ pars, int n, int nrep, uint64_t seed, uint32_t sim0, int t, int era_all,
         const uint8_t *__restrict__ zc, uint8_t *__restrict__ yc)
{
    const int k = blockIdx.x * 256 + threadIdx.x, r = blockIdx.y, c = blockIdx.z;
    if (k >= n) return;
    const size_t i = ((size_t)c * nrep + r) * n + k;
    uint8_t v = 0;
    if (zc[i]) {
        const Trans<R> tr = make_trans<R>(pars[c], era_all);
        const uint4 u = rng(seed, sim0 + (uint32_t)c * (uint32_t)nrep + (uint32_t)r, (uint32_t)t, RK_SIM_EXT, (uint32_t)k, 0);
        v = u01(u.x) > (double)tr.E;
    }
    yc[i] = v;
}
//   k_fc_col   grid (patch tiles, chains): one thread per (chain, patch) runs the colonisation draws of all replicates
//              (u < C as in k_sim_col), writes next year's z, adds the occupied count of every trajectory (one shared-memory
//              atomic per warp, one global atomic per CTA and replicate) and the patch's count over the replicates to incidence
template <typename R>
__global__ void __launch_bounds__(256)
k_fc_col(Landscape<R> ls, const mp_params *__restrict__ pars, int nrep, uint64_t seed, uint32_t sim0, int t, int nyears, int era_all,
         const double *__restrict__ S, const uint8_t *__restrict__ yc, uint8_t *__restrict__ zc, int32_t *__restrict__ occ,
         uint32_t *__restrict__ inc)
{
    __shared__ int s_cnt[32];
    const int n = ls.n, c = blockIdx.y, tid = threadIdx.x, k = blockIdx.x * 256 + tid;
    const Trans<R> tr = make_trans<R>(pars[c], era_all);
    const R g = k < n ? source_term<R>(ls, tr, k) : (R)0;
    uint32_t mine = 0;
    for (int r0 = 0; r0 < nrep; r0 += 32) {
        const int nr = min(32, nrep - r0);
        if (tid < 32) s_cnt[tid] = 0;
        __syncthreads();
        for (int j = 0; j < nr; j++) {
            const int r = r0 + j;
            int v = 0;
            if (k < n) {
                const size_t i = ((size_t)c * nrep + r) * n + k;
                if (yc[i]) v = 1;
                else {
                    const R C = col_prob<R>(tr, (R)S[i], g);
                    const uint4 u = rng(seed, sim0 + (uint32_t)c * (uint32_t)nrep + (uint32_t)r, (uint32_t)t, RK_SIM_COL, (uint32_t)k, 0);
                    v = u01(u.x) < (double)C;
                }
                zc[i] = (uint8_t)v;
            }
            mine += v;
            const int w = __reduce_add_sync(0xffffffffu, v);
            if ((tid & 31) == 0 && w) atomicAdd(&s_cnt[j], w);
        }
        __syncthreads();
        if (occ && tid < nr && s_cnt[tid]) atomicAdd(&occ[((size_t)c * nrep + r0 + tid) * (nyears + 1) + t + 1], s_cnt[tid]);
        __syncthreads();
    }
    if (inc && mine) atomicAdd(&inc[(size_t)(t + 1) * n + k], mine);
}

//   k_ppc_obs  grid (patch tiles, chains): the observation of year t of every replicate, after k_fc_init (t = 0) and after
//              each k_fc_col (t + 1).  One thread per (chain, patch) runs all replicates of the patch.  A cell missing in obs
//              stays missing; otherwise rep = z, with detection z && u < p, u keyed by (sim, year, RK_PPC_DET, patch number).
//              The record word of a (chain, replicate, patch) holds the replicate's previous observation (bit 0) and its
//              number of years observed occupied D (bits 1-31).  detected / colonised / extinct of every (trajectory, year):
//              one shared-memory atomic per warp, one global atomic per CTA, replicate and statistic.  In the last year each
//              thread adds to patch_ge / patch_gt its replicates with D >= / > the observed D of the patch.
static __global__ void __launch_bounds__(256)
k_ppc_obs(const mp_params *__restrict__ pars, const int8_t *__restrict__ obs, int T, int n, int nrep, uint64_t seed, uint32_t sim0,
          int t, int detect, const uint8_t *__restrict__ zc, uint32_t *__restrict__ rec, int32_t *__restrict__ stats,
          uint32_t *__restrict__ patch_ge, uint32_t *__restrict__ patch_gt)
{
    __shared__ int s_cnt[32 * MP_NPPC];
    const int c = blockIdx.y, tid = threadIdx.x, k = blockIdx.x * 256 + tid;
    const bool live = k < n, last = t == T - 1;
    const int o = live ? obs[(size_t)t * n + k] : -1;
    const bool both = o >= 0 && t > 0 && obs[(size_t)(t - 1) * n + k] >= 0;   // observed in t-1 and t: a transition to count
    const double p = pars[c].p;
    uint32_t dobs = 0, ge = 0, gt = 0;
    if (last && live)
        for (int s = 0; s < T; s++) dobs += obs[(size_t)s * n + k] == 1;
    for (int r0 = 0; r0 < nrep; r0 += 32) {
        const int nr = min(32, nrep - r0);
        if (tid < 32 * MP_NPPC) s_cnt[tid] = 0;
        __syncthreads();
        for (int j = 0; j < nr; j++) {
            const int r = r0 + j;
            int det = 0, col = 0, ext = 0;
            if (live) {
                const size_t i = ((size_t)c * nrep + r) * n + k;
                uint32_t w = t > 0 ? rec[i] : 0u;
                if (o >= 0) {
                    int v = zc[i];
                    if (v && detect) {
                        const uint4 u = rng(seed, sim0 + (uint32_t)c * (uint32_t)nrep + (uint32_t)r, (uint32_t)t, RK_PPC_DET, (uint32_t)k, 0);
                        v = u01(u.x) < p;
                    }
                    const int prev = (int)(w & 1u);
                    det = v; col = both && !prev && v; ext = both && prev && !v;
                    w = (((w >> 1) + (uint32_t)v) << 1) | (uint32_t)v;
                }
                if (last) { ge += (w >> 1) >= dobs; gt += (w >> 1) > dobs; }
                else rec[i] = w;
            }
            const int a = __reduce_add_sync(0xffffffffu, det), b = __reduce_add_sync(0xffffffffu, col),
                      e = __reduce_add_sync(0xffffffffu, ext);
            if ((tid & 31) == 0) {
                if (a) atomicAdd(&s_cnt[j * MP_NPPC + 0], a);
                if (b) atomicAdd(&s_cnt[j * MP_NPPC + 1], b);
                if (e) atomicAdd(&s_cnt[j * MP_NPPC + 2], e);
            }
        }
        __syncthreads();
        if (tid < nr * MP_NPPC && s_cnt[tid]) {
            const int j = tid / MP_NPPC, s = tid - j * MP_NPPC;
            atomicAdd(&stats[(((size_t)c * nrep + r0 + j) * T + t) * MP_NPPC + s], s_cnt[tid]);
        }
        __syncthreads();
    }
    if (last && live) {
        if (ge) atomicAdd(&patch_ge[k], ge);
        if (gt) atomicAdd(&patch_gt[k], gt);
    }
}

// ------------------------------------------------------------------ peak probes (roofline denominators)
__global__ void k_probe_mufu(float *out, int iters)
{
    float a = 0.5f + 1e-6f * threadIdx.x, b = 0.25f + 1e-6f * threadIdx.x, c = 0.125f, d = 0.75f;
    for (int i = 0; i < iters; i++) {
        a = Num<float>::ex2(-a); b = Num<float>::ex2(-b); c = Num<float>::ex2(-c); d = Num<float>::ex2(-d);
    }
    if (a + b + c + d == 12345.f) out[0] = a;
}
__global__ void k_probe_ffma(float *out, int iters)
{
    float a = 1.0f + threadIdx.x, b = 2.0f, c = 3.0f, d = 4.0f, e = 5.f, f = 6.f, g = 7.f, h = 8.f;
    const float m = 0.999f, s = 1e-3f;
    for (int i = 0; i < iters; i++) {
        a = fmaf(a, m, s); b = fmaf(b, m, s); c = fmaf(c, m, s); d = fmaf(d, m, s);
        e = fmaf(e, m, s); f = fmaf(f, m, s); g = fmaf(g, m, s); h = fmaf(h, m, s);
    }
    if (a + b + c + d + e + f + g + h == 12345.f) out[0] = a;
}
__global__ void k_probe_dadd(double *out, int iters)
{
    double a = 1.0 + threadIdx.x, b = 2.0, c = 3.0, d = 4.0, e = 5., f = 6., g = 7., h = 8.;
    const double s = 1e-3;
    for (int i = 0; i < iters; i++) { a += s; b += s; c += s; d += s; e += s; f += s; g += s; h += s; }
    if (a + b + c + d + e + f + g + h == 12345.) out[0] = a;
}
__global__ void k_probe_copy(const float4 *__restrict__ in, float4 *__restrict__ out, size_t n4)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) out[i] = in[i];
}

}  // namespace mp
