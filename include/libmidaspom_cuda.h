/* libmidaspom_cuda.h -- C ABI of the B200-native SPOM likelihood / MCMC engine.
 *
 * This is the drop-in boundary for ONE hot path of nalcala/MIDASPOM: the stochastic patch
 * occupancy model (SPOM) log-likelihood and its connectivity term.  The reference has no
 * plugin/FFI boundary (each program is one C translation unit); the entry points below sit on its
 * function-level seams and keep its conventions: plain C, caller-owned flat host arrays, years
 * major / patches minor (piobs[i][j], main_MIDASPOM.c:152-161), scalars by value.  Unlike the
 * reference they return an int status (0 = ok, <0 = error, text via mp_last_error) and never abort.
 *
 * Reference code each entry point replaces (paths under /root/reference/sources/):
 *   mp_set_landscape_linear   main_MIDASPOM.c:177-188          kernel matrix M[i][j]=exp(-a|i-j|d) (flag -d);
 *                             never materialised here: weights are evaluated on the fly
 *   mp_set_landscape_coords / _dense                            (extension: general d_ij, areas A_j^b)
 *   mp_set_observations       main_MIDASPOM.c:138-167           piobs table (-1/0/1), T x N
 *   mp_connectivity           main_MIDASPOM.c:350-358           S_k = sum_{l!=k} M[l][k] y_l  (scalar triple loop)
 *                             dieoff.c:73-79, loss.c:74-80,93-101, future.c:89-97
 *   mp_loglik                 main_MIDASPOM.c:18-50 (compPePc), dieoff.c:51-83 (pije/pijc),
 *                             loss.c:86-105 (pijcsource): the per-patch Bernoulli factors, summed as logs
 *   mp_flip_delta             (no counterpart) rank-1 incremental form of the same terms
 *   mp_sweep / mp_get_draws   replaces the (e,c) grid loops main_MIDASPOM.c:341-395 by data-augmented
 *                             Gibbs/Metropolis chains; MIDASPOM_MPI's static row split
 *                             (main_MIDASPOM_MPI.c:361-372,483-505) becomes chain sharding (chain_offset)
 *   mp_set_era / mp_params.K,Ksrc,dsrc   dieoff.c:56-57,78 ; loss.c:93-101,365 ; future.c:67,90-97
 *   mp_simulate               future.c:64-110 (simpij) + :359-386 (simulation loop)
 *   mp_forecast               future.c:359-386 at large N: the simulation loop started from the sampler's own chains
 *   mp_set_summaries / mp_get_summaries   (no counterpart) posterior occupancy, survival and connectivity of every patch-year
 *   mp_set_waic / mp_get_waic  Rscript/hypothesis_test.R at large N: pointwise predictive densities for WAIC
 *   mp_ppc                    (no counterpart) posterior-predictive replicates of the observation table from the chains
 *   mp_capacity               (no counterpart) metapopulation capacity and patch values of the landscape per parameter set
 *   mp_set_sources / mp_get_sources   (no counterpart) colonisations attributed to their source patches and distances
 *
 * All device memory is owned by the engine handle; host buffers are owned by the caller.  One
 * handle per GPU / host thread (thread-compatible, not thread-safe).  There is no CPU fallback:
 * every entry point fails with MP_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef LIBMIDASPOM_CUDA_H
#define LIBMIDASPOM_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MP_ABI_VERSION 1

enum { MP_OK = 0, MP_ERR_ARG = -1, MP_ERR_CUDA = -2, MP_ERR_STATE = -3, MP_ERR_UNSUPPORTED = -4 };
enum { MP_FP32 = 0, MP_FP64 = 1 };                       /* arithmetic of the weight / log terms */
enum { MP_GEOM_LINEAR = 0, MP_GEOM_COORDS = 1, MP_GEOM_DENSE = 2 };

#define MP_NDRAW 11  /* per (sweep, chain): e, c, alpha, b, p, loglik, #y=1, #z=1, K, Ksrc, dsrc */
#define MP_NLSIG 8   /* log proposal scales: e, c, alpha, b, p, K, Ksrc, dsrc */
#define MP_NPART 4   /* loglik parts: extinction, colonisation, year-0 prior, detection */

typedef struct mp_engine mp_engine;

typedef struct {
    int32_t  n_patches;      /* N */
    int32_t  n_years;        /* T (rows of the observation table) */
    int32_t  n_chains;       /* chains resident on this GPU */
    int32_t  chain_offset;   /* global id of local chain 0 (RNG streams are keyed by global id) */
    int32_t  precision;      /* MP_FP32 | MP_FP64 */
    int32_t  device;         /* CUDA ordinal */
    int32_t  detect;         /* 0: perfect detection (reference) ; 1: obs=0 hides z=1 w.p. 1-p */
    int32_t  max_draws;      /* capacity (sweeps) of the device draw buffer */
    uint64_t seed;
    double   prior_occ;      /* flag -p: year-0 prior occupancy of latent cells (float in the reference) */
} mp_config;

/* e, c: flags/grid axes of the reference; alpha = 1/(flag -m); b: area exponent; p: detection;
 * K: pre-event scaling (E=min(1,e/K), C=min(1,c*(K*S+...))); Ksrc, dsrc: external source size and
 * distance unit (source term exp(-alpha*u_k*dsrc)*Ksrc, u_k = k+1 by default, loss.c:365). */
typedef struct { double e, c, alpha, b, p, K, Ksrc, dsrc; } mp_params;

typedef struct {
    double  e_min, e_max, c_min, c_max, alpha_min, alpha_max, b_min, b_max, p_min, p_max;
    double  K_min, K_max, Ksrc_min, Ksrc_max, dsrc_min, dsrc_max;   /* variant parameters (dieoff.c:283-286, loss.c:319-322 grids) */
    int32_t sample_e, sample_c, sample_alpha, sample_b, sample_p;
    int32_t n_e_steps, n_c_steps;   /* Metropolis sub-steps per sweep */
    int32_t n_adapt;                /* sweeps during which proposal scales adapt */
    int32_t update_z, update_y;     /* Gibbs updates of latent occupancy / intermediate state */
    int32_t sample_K, sample_Ksrc, sample_dsrc;   /* Metropolis on the pre-event scaling / external source (log-uniform K, Ksrc; uniform dsrc) */
    int32_t n_v_steps;              /* sub-steps per sweep for each sampled variant parameter */
} mp_sampler_config;

/* kernel categories for mp_get_timing */
enum { MP_K_CONN = 0, MP_K_COL = 1, MP_K_SWEEP_Y = 2, MP_K_SWEEP_Z = 3, MP_K_SMALL = 4, MP_K_SIM = 5, MP_K_NCAT = 6 };
/* device buffers for mp_device_ptr (zero-copy hand-off to NCCL / torch) */
enum { MP_BUF_DRAWS = 0, MP_BUF_Z = 1, MP_BUF_Y = 2, MP_BUF_S = 3, MP_BUF_PARAMS = 4, MP_BUF_S_PROP = 5 };

const char *mp_version(void);
int mp_device_count(void);

int mp_create(const mp_config *cfg, mp_engine **out);
int mp_destroy(mp_engine *h);
const char *mp_last_error(const mp_engine *h);   /* h may be NULL: error of the last failed mp_create */

/* ---- landscape (replaces the dense kernel matrix M) ---- */
int mp_set_landscape_linear(mp_engine *h, double spacing, const double *area /* N or NULL */);
int mp_set_landscape_coords(mp_engine *h, const double *x, const double *y, const double *area);
int mp_set_landscape_dense(mp_engine *h, const double *dist /* N*N, [source][target] */, const double *area);
int mp_set_source_units(mp_engine *h, const double *src_unit /* N or NULL => k+1 */);
/* Order in which the y scan visits the patches of a year (slot -> patch): the Morton order of planar
 * coordinates, index order for linear and dense landscapes (oracle: spom_scan_order). */
int mp_get_scan_order(mp_engine *h, int32_t *order /* N */);
/* Block grid of the y scan (planar coordinates only; no reference counterpart -- the reference has no sampler).
 * The bounding box of the patches is cut into nx x ny cells and the cells are coloured k x k periodically.  The scan
 * then visits the patches colour by colour, block by block, in Morton order inside a block (oracle: spom_scan_order
 * with blk_nx, blk_ny, blk_k -- any fixed order is a valid Gibbs scan).  The FP32 engine scans the blocks of one colour
 * CONCURRENTLY, one cluster per (chain, year, block), with the block's own patches and every patch within `halo` of
 * its cell as targets: same-colour cells must lie farther apart than 2 halo ((k - 1) x cell width > 2 halo, else
 * MP_ERR_ARG), so their target sets are disjoint.  Each sweep a (chain, year) is scanned by blocks only if the largest
 * dispersal weight at the halo distance is below 2^-36 of the year's smallest S -- the commit rule the whole-year culled
 * scan applies anyway -- and the year holds at least 64 occupied patches; otherwise that year falls back to the
 * whole-year scan in the same order.  nx * ny <= 1 switches the grid off.  The FP64 engine only takes the order. */
int mp_set_scan_blocks(mp_engine *h, int nx, int ny, int k, double halo);

/* ---- data ---- */
int mp_set_observations(mp_engine *h, const int8_t *obs /* T*N, -1/0/1 */);
int mp_set_era(mp_engine *h, const uint8_t *era /* T-1 flags or NULL */);

/* ---- chain state ---- */
int mp_set_params(mp_engine *h, const mp_params *par /* n_chains */);
int mp_get_params(mp_engine *h, mp_params *par);
int mp_set_state(mp_engine *h, const uint8_t *z /* C*T*N */, const uint8_t *y /* C*(T-1)*N */);
int mp_get_state(mp_engine *h, uint8_t *z, uint8_t *y);
int mp_set_scales(mp_engine *h, const double *lsig /* C*MP_NLSIG */);
int mp_get_scales(mp_engine *h, double *lsig);

/* ---- likelihood ---- */
/* recompute S from the current y and parameters; S_out (host, C*(T-1)*N, nullable).  FP64 engines: 1e-9 path.  FP32 engines: the
 * evaluation form of k_conn (or the tensor-core path, see mp_get_conn_path), inside the FP32 path's 1e-5 */
int mp_connectivity(mp_engine *h, double *S_out);
int mp_get_connectivity(mp_engine *h, double *S_out);   /* copy of the resident S (no recompute) */
/* complete-data log-likelihood per chain (recomputes S); parts: C*MP_NPART, nullable */
int mp_loglik(mp_engine *h, double *ll, double *parts);
/* one-call form: upload parameters and state, evaluate, download (host buffers in and out) */
int mp_loglik_host(mp_engine *h, const mp_params *par, const uint8_t *z, const uint8_t *y, double *ll, double *parts);
/* log-odds of flipping y[chain][t][k] by the rank-1 update of the resident S */
int mp_flip_delta(mp_engine *h, int chain, int t, int k, double *dll);

/* ---- sampler ---- */
int mp_init_chains(mp_engine *h, const mp_sampler_config *sc, int disperse);
int mp_set_sampler(mp_engine *h, const mp_sampler_config *sc);
int mp_sweep(mp_engine *h, int nsweeps);            /* asynchronous on the engine stream */
int mp_synchronize(mp_engine *h);
/* One chain sharded over several GPUs (large N): every rank holds a full replica and runs the four phases of
 * a sweep with a collective in between (midaspom_b200/distributed.py: ShardedChain).
 *   mp_set_shard: this engine evaluates the connectivity of the targets [conn_lo, conn_hi) only (conn_hi < 0: all;
 *     positions in the Morton order of the patches on landscapes with positions, patch numbers otherwise; multiples
 *     of 256 except for the last rank) and scans the (chain, year) tasks task_first, task_first + task_stride, ... only.
 *     The other targets' columns of S / S_prop are left zero so that a sum over ranks assembles them.
 *   mp_sweep_phase: 0 proposal + connectivity (sum S / S_prop over ranks afterwards; flags_out bit 0: resident S
 *     recomputed, bit 1: proposal computed), 1 Metropolis decisions + z update, 2 y scan of the owned tasks
 *     (exchange the owned rows of y and S afterwards), 3 e/p update + record.  mp_sweep == the four phases. */
int mp_set_shard(mp_engine *h, int conn_lo, int conn_hi, int task_first, int task_stride);
int mp_sweep_phase(mp_engine *h, int phase, int *flags_out);
/* ---- several GPUs behind the C ABI (NCCL; replaces MPI_Init / the row split / the MPI_Send-MPI_Recv gather of
 * main_MIDASPOM_MPI.c:344-372,483-505).  One process per GPU: rank 0 calls mp_comm_unique_id, ships the MP_COMM_ID_BYTES
 * to the other ranks by whatever launcher it runs under, and every rank calls mp_comm_init.  One process driving several
 * engines (one per device): mp_comm_init_all.  NCCL is loaded at the first of these calls (MP_ERR_UNSUPPORTED if absent).
 *   mp_gather_draws   every rank's draws [first, first + count): out[rank][sweep][chain][MP_NDRAW], same on every rank
 *                     (independent chains per rank, chain_offset = rank x n_chains)
 *   mp_sweep_sharded  nsweeps iterations of ONE set of chains replicated on every rank: connectivity split by target
 *                     patches (all-gather of the owned columns of S / S_prop), y scan split by (chain, year) tasks
 *                     (broadcast of the owned rows of y and S), decisions replicated; equals mp_sweep on one engine bit
 *                     for bit.  Everything is enqueued on the engine stream; no host synchronisation inside a sweep.
 *                     In a single process call it for every engine of the communicator between mp_comm_group_begin /
 *                     mp_comm_group_end is NOT needed: use mp_sweep_sharded_all instead. */
#define MP_COMM_ID_BYTES 128
int mp_comm_unique_id(void *id128);
int mp_comm_init(mp_engine *h, int nranks, int rank, const void *id128);
int mp_comm_init_all(mp_engine **engines, int n);
int mp_comm_destroy(mp_engine *h);
int mp_comm_rank(mp_engine *h);
int mp_comm_size(mp_engine *h);
const char *mp_comm_last_error(void);
int mp_gather_draws(mp_engine *h, int first, int count, double *out /* nranks*count*C*MP_NDRAW */);
int mp_gather_draws_all(mp_engine **engines, int n, int first, int count, double *out);   /* one process, all engines: one NCCL group */
int mp_sweep_sharded(mp_engine *h, int nsweeps);
int mp_sweep_sharded_all(mp_engine **engines, int n, int nsweeps);
int mp_num_draws(mp_engine *h);
int mp_get_draws(mp_engine *h, int first, int count, double *out /* count*C*MP_NDRAW */);
int mp_reset_draws(mp_engine *h);
int mp_sweep_index(mp_engine *h);
/* Posterior summaries of the latent state (no reference counterpart: the reference marginalises the missing cells away),
 * accumulated on the device at the end of every qualifying sweep, summed over this engine's chains.  first_sweep: the first
 * sweep index (as mp_sweep_index counts) that is accumulated; thin: every thin-th sweep from there.  thin = 0 switches the
 * summaries off and frees them.  Setting them zeroes every array.  A sweep adds the state it ends with: z, y, S after the
 * y scan and the parameters after the e/p update.  The sweep counter is read on the device, so captured sweeps replay
 * unchanged; without summaries a sweep launches exactly what it launched before.  One kernel per qualifying sweep, counted
 * under MP_K_SMALL.  Device memory: T N 12 + (T-1) N 12 bytes.
 * mp_forecast, mp_connectivity, mp_loglik, mp_loglik_host, mp_simulate* and mp_flip_delta leave the sums unchanged.
 * mp_sweep_sharded[_all] ranks hold identical sums (phase 3 runs replicated); chain-sharded engines (chain_offset) add theirs.
 * MP_ERR_ARG: first_sweep < 0 or thin < 0. */
int mp_set_summaries(mp_engine *h, int first_sweep, int thin);
/* Copy (and with reset != 0 zero) the sums.  Every output is nullable.  Synchronous, after any queued sweeps.
 *   nsamples   accumulated sweeps x n_chains
 *   z_count    T*N      uint32   number of samples with z_tk = 1
 *   z_prob     T*N      double   sum of P(z_tk = 1 | y, theta, obs) (Rao-Blackwellised: the log-odds of k_update_z, in the
 *                                engine's precision; 1 for cells an adjacent y = 1 forces; the indicator for cells the data fix;
 *                                0 where the log-odds is NaN, as the Gibbs draw)
 *   y_count    (T-1)*N  uint32   number of samples with y_tk = 1 (patch occupied and survived extinction in t -> t+1)
 *   S_sum      (T-1)*N  double   sum of the connectivity S_tk
 * Extinctions in t -> t+1 = z_count[t] - y_count[t]; colonisations = z_count[t+1] - y_count[t].
 * MP_ERR_STATE: summaries not set.  mp_sweep (and the sharded and phase forms) refuses with MP_ERR_STATE, before launching,
 * when the queued sweeps could push nsamples past 2^32 - 1, the limit of the uint32 counts. */
int mp_get_summaries(mp_engine *h, int64_t *nsamples, uint32_t *z_count, double *z_prob, uint32_t *y_count,
                     double *S_sum, int reset);
/* Pointwise predictive densities of the observations for WAIC (no reference counterpart: the large-N counterpart of the
 * model comparison of Rscript/hypothesis_test.R), accumulated on the device at the end of every qualifying sweep, summed
 * over this engine's chains.  first_sweep / thin as for mp_set_summaries; thin = 0 switches them off and frees them;
 * setting them zeroes the sums, and so does mp_set_observations while they are on.  For every observed cell (obs 0 or 1,
 * year 0 included) a sample adds the density p of the observation given the chain's state of the previous year:
 *   pi = p0 (year 0);  pi = s + (1 - s) C_{t-1,k},  s = z_{t-1,k} (1 - E_{t-1})  (t >= 1, E and C of transition t-1,
 *        C from the S the sweep ends with)
 *   p  = q pi (obs 1),  1 - q pi (obs 0),  q = p (detection on) or 1
 * This is a conditional predictive: values compare only between fits to the same observations and prior_occ.
 * One kernel per qualifying sweep, counted under MP_K_SMALL; without WAIC a sweep launches exactly what it launched before.
 * Device memory: T N 24 + 8 bytes.  mp_forecast, mp_connectivity, mp_loglik, mp_loglik_host, mp_simulate* and mp_flip_delta
 * leave the sums unchanged.  mp_sweep_sharded[_all] ranks hold identical sums; chain-sharded engines add theirs.
 * MP_ERR_ARG: first_sweep < 0 or thin < 0.  MP_ERR_STATE: switched on before mp_set_observations. */
int mp_set_waic(mp_engine *h, int first_sweep, int thin);
/* Copy (and with reset != 0 zero) the sums.  Every output is nullable; each array is T*N, 0 in cells that are not
 * observations.  Synchronous, after any queued sweeps.
 *   nsamples    accumulated sweeps x n_chains (S)
 *   lik_sum     L_i = sum of p
 *   loglik_sum  G_i = sum of log p
 *   loglik_sq   Q_i = sum of (log p)^2
 * Reduction (Watanabe 2010; Vehtari, Gelman and Gabry 2017), over the observed cells i, after adding the arrays of
 * chain-sharded engines:  lppd_i = log(L_i / S),  p_waic_i = max(0, (Q_i - G_i^2 / S) / (S - 1)) (needs S >= 2),
 * elpd_i = lppd_i - p_waic_i;  elpd_waic = sum_i elpd_i, waic = -2 elpd_waic.  Two fits A, B to the same observations:
 * delta = sum_i (elpd_i^A - elpd_i^B), se = sqrt(n_obs var_i(elpd_i^A - elpd_i^B)).
 * MP_ERR_STATE: WAIC sums not set. */
int mp_get_waic(mp_engine *h, int64_t *nsamples, double *lik_sum, double *loglik_sum, double *loglik_sq, int reset);
/* Attribution of every colonisation to its source patches (no reference counterpart), accumulated on the device at the end
 * of every qualifying sweep, summed over this engine's chains.  first_sweep / thin as for mp_set_summaries; thin = 0 switches
 * them off and frees them; setting them zeroes every array.  For a sample (chain after a qualifying sweep, its final z, y,
 * resident S and parameters) and transition t = 0 .. T-2:
 *   event        target k with y_tk = 0 and z_{t+1,k} = 1 (the cells whose likelihood term is log C_tk)
 *   pressure     P_tk = K_t S_tk + Ksrc_t g_k (K_t, Ksrc_t, g_k as in C_tk; P = S without era flags)
 *   shares       source l (y_tl = 1): rho_tkl = K_t w(k<-l) / P_tk;  external: rho_tk,ext = Ksrc_t g_k / P_tk; they sum to 1
 *   unattributed an event with P_tk = 0 (an initial or impossible state): counted, not attributed
 * rho is the share of the colonisation pressure, not an observed causal link: read it as "which source colonised k" only under
 * independent propagule contributions.  nbins > 0 adds a histogram of rho over the source-target distance d (pair_distance's
 * value in the landscape's unit): bins [b w, (b + 1) w), the last bin open (d >= (nbins - 1) w); nbins = 0: no histogram,
 * bin_width ignored.  Per transition, sum_l src_sum + ext_sum = events - unattributed up to the difference between the
 * resident S and a fresh sum of the same weights; sum_b dist_hist = sum_l src_sum up to the histogram's fixed point (each pair
 * is rounded to 2^-40).  Three kernels per qualifying sweep (no floating-point atomics: bit-identical sums), counted under
 * MP_K_SMALL; without sources a sweep launches exactly what it launched before.  The work is events x sources per (chain,
 * transition), without culling.  Device memory: C (T-1) N (2 r + 8) + (T-1) N 8 + C (T-1) 24 + (T-1)(16 nbins + 24) + 8 bytes
 * (each part rounded up to 256), r = 16 (FP32) or 32 (FP64) the record size.  mp_forecast, mp_ppc, mp_capacity, mp_connectivity,
 * mp_loglik[_host], mp_simulate* and mp_flip_delta leave the sums unchanged.  mp_sweep_sharded[_all] ranks hold identical sums
 * (phase 3 runs replicated there); chain-sharded engines add theirs.
 * MP_ERR_ARG: first_sweep < 0, thin < 0, nbins < 0 or > 4096, or nbins > 0 with bin_width not finite and > 0. */
int mp_set_sources(mp_engine *h, int first_sweep, int thin, int nbins, double bin_width);
/* Copy (and with reset != 0 zero) the sums.  Every output is nullable.  Synchronous, after any queued sweeps.
 *   nsamples   accumulated sweeps x n_chains
 *   events     (T-1)*2: events[t] at t, unattributed[t] at (T-1) + t
 *   src_sum    (T-1)*N, patch order: sum over samples and events of rho_tkl (expected colonisations patch l seeded in t -> t+1)
 *   ext_sum    T-1: sum of rho_tk,ext
 *   dist_hist  (T-1)*nbins: sum of rho_tkl over the pairs in each distance bin (untouched without a histogram)
 * MP_ERR_STATE: source sums not set. */
int mp_get_sources(mp_engine *h, int64_t *nsamples, uint64_t *events, double *src_sum, double *ext_sum, double *dist_hist, int reset);

/* ---- forward simulator ---- */
/* nsims independent trajectories of nyears from z0 (N bytes); era_all != 0 applies K/Ksrc every
 * year (future.c).  z_out (nullable): nsims*(nyears+1)*N ; occupied_out (nullable): nsims*(nyears+1) counts */
int mp_simulate(mp_engine *h, const mp_params *par, const uint8_t *z0, int nyears, int nsims, uint64_t seed,
                int era_all, uint8_t *z_out, int32_t *occupied_out);
/* same, with one parameter set and one start state per trajectory (future.c:359-381 draws (e,c) from
 * the posterior table and a completion of the last survey for every simulation) */
int mp_simulate_ensemble(mp_engine *h, const mp_params *par_per_sim /* nsims */, const uint8_t *z0_per_sim /* nsims*N */,
                         int nyears, int nsims, uint64_t seed, int era_all, uint8_t *z_out, int32_t *occupied_out);
/* Posterior-predictive forecast from the chains' current state (large-N counterpart of MIDASPOM_future.out,
 * future.c:359-386).  Chain c starts nrep trajectories from its own latent occupancy of the last survey year,
 * z[c][T-1], with its own resident parameters, and simulates nyears years of simpij (future.c:64-110).
 * Trajectory (c, r) draws from the Philox streams that mp_simulate_ensemble gives simulation number
 * (chain_offset + c) * nrep + r under `seed`, so results do not depend on how chains are sharded.
 * scenario (nullable): {K, Ksrc, dsrc}.  Replaces the chains' K, Ksrc, dsrc and applies them in every forecast year
 *   (era_all of mp_simulate; the reference's -D, -S, -s).  NULL: plain model.
 * occupied_out  (nullable): n_chains * nrep * (nyears+1) int32, occupied patches per trajectory (year 0 = start).
 * incidence_out (nullable): (nyears+1) * N uint32, the number of this engine's trajectories with patch k occupied in year t.
 * Leaves all sampler state as it was: chain state, S and its validity flags, draws, sweep counter, scales, captured graphs.
 * Synchronous, on the engine stream after any queued sweeps.
 * One year: extinction draws, then the connectivity of every (chain, replicate) by k_conn with the replicates in place of the
 * years (one weight per (target, source) pair and chain, shared by the chain's replicates; FP64 accumulation; FP32 engines on
 * landscapes with positions skip source tiles whose weights add less than 2^-32 to any c K S, MP_CONN_CULL=0 disables),
 * then the colonisation draws.  Counted under MP_K_SIM and in MP_CNT_CONN_*; mp_set_shard does not apply (every target).
 * Device memory: one arena per call of about C nrep N (8 + 2 + 0.5 (FP32) | 1 (FP64)) bytes -- S, the current and surviving
 * states, the source records -- plus C N (8 | 4) bytes of area weights and the outputs.
 * MP_ERR_ARG: nyears < 1, nrep < 1 or > 65535, (chain_offset + n_chains) * nrep >= 2^32, scenario K <= 0.
 * MP_ERR_STATE: no landscape, no chain state, a chain with alpha <= 0. */
int mp_forecast(mp_engine *h, int nyears, int nrep, uint64_t seed, const double *scenario,
                int32_t *occupied_out, uint32_t *incidence_out);
/* Posterior-predictive check of the fit (no reference counterpart): nrep replicates per chain of the whole observation table,
 * simulated from the chain's own imputed year 0 and resident parameters under the fit's own era flags, observed through the
 * table's missing-cell mask and, with detection on, the chain's p (DESIGN.md §2 defines every step and statistic).
 * Trajectory (c, r) is simulation number (chain_offset + c) * nrep + r under `seed`, the numbering of mp_forecast, so results do
 * not depend on how chains are sharded.  Statistics, integers per (chain, replicate, year t):
 *   0 detected   observed cells with rep_tk = 1
 *   1 colonised  cells observed in t-1 and t with rep 0 -> 1 (0 in year 0)
 *   2 extinct    cells observed in t-1 and t with rep 1 -> 0 (0 in year 0)
 * stats_out      (nullable): n_chains * nrep * T * MP_NPPC int32, [chain][replicate][year][statistic]
 * obs_stats_out  (nullable): T * MP_NPPC int32, the same statistics of the observation table itself
 * patch_ge / patch_gt (nullable): N uint32 each, the number of this engine's replicates whose count of years observed occupied,
 *   D_k = sum_t [rep_tk = 1], is >= / > that of the observations, sum_t [obs_tk = 1].  Chain-sharded engines add theirs.
 * Replicates start from the chains' imputed year 0, so without detection their year 0 reproduces the observed cells exactly: the
 * check concerns years 1 .. T-1.
 * Leaves all sampler state as it was: chain state, S and its validity flags, draws, sweep counter, scales, captured graphs, the
 * summaries and the WAIC sums.  Synchronous, on the engine stream after any queued sweeps.  Each transition runs mp_forecast's
 * year (k_conn shared by a chain's replicates; FP32 engines on landscapes with positions cull it with the floor of DESIGN.md §5,
 * MP_CONN_CULL=0 disables), then one observation kernel per year.  Counted under MP_K_SIM and in MP_CNT_CONN_*; mp_set_shard does
 * not apply.  Device memory: one arena per call of mp_forecast's size plus C nrep N 4 bytes of per-replicate records and
 * C nrep T MP_NPPC 4 bytes of statistics.
 * MP_ERR_ARG: nrep < 1 or > 65535, (chain_offset + n_chains) * nrep >= 2^32.
 * MP_ERR_STATE: no observations, no landscape, no chain state, a chain with alpha <= 0. */
#define MP_NPPC 3   /* detected, colonised, extinct */
int mp_ppc(mp_engine *h, int nrep, uint64_t seed, int32_t *stats_out, int32_t *obs_stats_out, uint32_t *patch_ge,
           uint32_t *patch_gt);
/* Metapopulation capacity of the landscape (Hanski & Ovaskainen 2000) and patch values (Ovaskainen & Hanski 2001), one eigenproblem
 * per parameter set (no reference counterpart; DESIGN.md §2 defines the quantities).  lambda_M is the largest eigenvalue of the
 * symmetric M~_kl = sqrt(a_k a_l) exp(-alpha d_kl) (k != l), M~_kk = 0, a = A^b; only alpha and b of a set are read.  LOBPCG with
 * block size 1 from the all-ones vector over the kept patches, stopped when ||M~x - theta x|| / theta <= rtol.
 *   par        nsets parameter sets; NULL: the chains' resident parameters (nsets = n_chains), after any queued sweeps
 *   keep       (nullable) N flags in patch order: 0 removes the patch as source and target (the principal submatrix)
 *   out3       nsets*3: lambda (Rayleigh quotient of the returned vector: a lower bound of lambda_M), relative residual
 *              ||M~x - lambda x|| / lambda, relative bound of the culled weights (||E||_2 / lambda; 0 when nothing is culled)
 *   iters_out  (nullable) nsets iterations; a set that has not converged after max_iter reports max_iter and a residual above rtol
 *              (not an error)
 *   value_out  (nullable) nsets*N patch values V_k = x_k^2 / ||x||^2 in patch order (sum 1; 0 on removed patches); removing patch k
 *              changes lambda_M by about -2 lambda V_k
 *   value_sum  (nullable) N: the values summed over the sets
 * Synchronous, on the engine stream after any queued sweeps.  Leaves everything as it was: chain state, S and its validity flags,
 * draws, sweep counter, scales, captured graphs, summaries and WAIC sums.  Kernels are counted under MP_K_SIM, the (32 target x 32
 * source) tiles of the products in MP_CNT_CONN_EXEC / MP_CNT_CONN_TOTAL; mp_set_shard does not apply.  FP32 engines on landscapes
 * with positions skip tiles whose largest weight is below 2^-30 theta0 / N (theta0: the Rayleigh quotient of the start vector under
 * an unculled product), MP_CONN_CULL=0 disables; the FP64 engine never culls.  A set's results depend only on its (alpha, b), the
 * landscape, keep, rtol and max_iter, bit for bit: not on nsets, the other sets, the batching or chain_offset.
 * Device memory: one arena per call of about min(nsets, ~1 GB worth) x N x (48 + 4 | 8) bytes; more sets run in batches.
 * MP_ERR_ARG: nsets < 1, rtol <= 0, max_iter < 1, alpha <= 0, fewer than 2 kept patches, par = NULL with nsets != n_chains.
 * MP_ERR_STATE: no landscape, par = NULL before any chain parameters are set.
 * MP_ERR_UNSUPPORTED: a dense landscape whose distance matrix is not symmetric. */
int mp_capacity(mp_engine *h, int nsets, const mp_params *par, const uint8_t *keep, double rtol, int max_iter, double *out3,
                int32_t *iters_out, double *value_out, double *value_sum);

/* ---- exact small-n engine: the reference's own algorithm (state enumeration on an (e,c) grid) ----
 * Replaces the whole hot loop of MIDASPOM.out, main_MIDASPOM.c:198-290 (state tables) and :341-395
 * (compPePc, Pe.Pc, forward recursion): loglik_out[ie*nstep+ic] = log L(e_ie, c_ic) on the grid
 * ecmin + i*(ecmax-ecmin)/(nstep-1); ltot_out (nullable) = the "Total log-likelihood" of :414-425;
 * state_info (nullable, 4 ints) = variable patches, enumerated states, short-list states, max states/year.
 * Linear habitat only (flags -m -> a = 1/m, -d, -p, -s, -l, -u).  At most 24 variable patches, 12 missing cells in one
 * year and 4,096 distinct observation-compatible rows (P is formed in 32 x 32 tiles, the grid in batches of <= 2 GB). */
int mp_exact_posterior(int device, const int8_t *obs, int n_years, int n_patches, double a, double d, double prior_occ,
                       int nstep, double ecmin, double ecmax, double *loglik_out, double *ltot_out, int *state_info);
/* MIDASPOM_dieoff.out (variant 1, main_MIDASPOM_dieoff.c:307-351) / MIDASPOM_loss.out (variant 2,
 * main_MIDASPOM_loss.c:345-386): likelihood of the FIRST survey row after ts pre-event + tdis post-event
 * unobserved years, on the log-spaced K grid (x the d_L grid for loss).  lik_out: nstepK (dieoff) or
 * nstepK*nstepd (loss) raw likelihoods, in the layout the reference writes.  At most 16 patches (the reference's own
 * 2^n x 2^n matrices stop fitting memory at 15); up to 13 the state vectors stay in shared memory. */
int mp_exact_variant(int device, int variant, const int8_t *first_row, int n_patches, double a, double d, double prior_occ,
                     double eB, double cB, int ts, int tdis, int nstepK, double Kmin, double Kmax, int nstepd, double dmin,
                     double dmax, double *lik_out);
const char *mp_exact_last_error(void);

/* ---- plumbing ---- */
int mp_device_ptr(mp_engine *h, int which, void **ptr, size_t *bytes);
/* the cudaStream_t every kernel of this engine is launched on (for CUDA-event timing by the caller) */
int mp_get_stream(mp_engine *h, void **stream);
int mp_set_timing(mp_engine *h, int enabled);
/* accumulated since the last call with reset != 0: ms[MP_K_NCAT], launches[MP_K_NCAT] */
int mp_get_timing(mp_engine *h, double *ms, int64_t *launches, int reset);
/* Work actually executed by the hot kernels since the last reset (always on: warp-local counts, one atomic per warp and
 * launch).  Used by bench.py so that roofline fractions count executed work, not the dense algorithm's:
 *   MP_CNT_SCAN_TRIPS    warp-trips of the culled y scan (one trip = one exchange of SP candidate sums; with the branch sum of
 *                        the 512-thread tasks, the exchange also carries "candidate 2 given candidate 1 accepted")
 *   MP_CNT_SCAN_EXEC     (candidate, group of 32 targets) evaluations executed, speculative ones included; the branch sum
 *                        evaluates no weights of its own and adds nothing here
 *   MP_CNT_SCAN_RETIRED  the part of MP_CNT_SCAN_EXEC that belongs to candidates decided in their trip (with the branch sum:
 *                        both candidates of a trip unless the second one is deferred)
 *   MP_CNT_SCAN_COMMIT   (accepted flip, group of 32 targets) rank-1 updates of S
 *   MP_CNT_SCAN_DENSE    (candidate, target) pairs of the unculled scans (k_sweep_y_fast, k_sweep_y)
 *   MP_CNT_CONN_EXEC     (group of 32 targets, group of 32 sources) tiles of k_conn evaluated
 *   MP_CNT_CONN_TOTAL    the same, culled ones included
 *   MP_CNT_GEMM_TILES    128 x 128 x 64 tensor-core tiles issued by the fixed-(alpha, b) connectivity path
 *   MP_CNT_SCAN_BLOCKS   block tasks of the y scan executed (mp_set_scan_blocks; 0: every year was scanned as a whole) */
enum { MP_CNT_SCAN_TRIPS = 0, MP_CNT_SCAN_EXEC = 1, MP_CNT_SCAN_RETIRED = 2, MP_CNT_SCAN_COMMIT = 3, MP_CNT_SCAN_DENSE = 4,
       MP_CNT_CONN_EXEC = 5, MP_CNT_CONN_TOTAL = 6, MP_CNT_GEMM_TILES = 7, MP_CNT_SCAN_BLOCKS = 8, MP_CNT_N = 9 };
int mp_get_work_counters(mp_engine *h, uint64_t *out /* MP_CNT_N */, int reset);
/* which kernel evaluated the connectivity last: 0 = k_conn (per-chain parameters; the sampler's own S with the year contraction
 * in FP64, the evaluation calls mp_connectivity / mp_loglik / mp_loglik_host of an FP32 engine with FP32 partial sums per 32
 * sources joined in FP64, ~1e-7 of every S -- the sweep after such a call recomputes the resident S), 1 = the tensor-core
 * contraction k_conn_gemm (FP32 engines; taken by mp_connectivity / mp_loglik / mp_loglik_host when every chain holds the
 * same alpha and b as uploaded by mp_set_params, the matrix form c*M%*%pti of Rscript/simuls_traj.R:16,203,214) */
int mp_get_conn_path(mp_engine *h);
/* launch geometry of the last y scan: out4 = threads per (chain, year) task, CTAs per cluster, candidates evaluated per
 * trip (1 + speculative), 1 if the spatially culled kernel ran, 2 if it ran block by block (mp_set_scan_blocks; the first
 * three numbers then describe a block task) (0: k_sweep_y_fast; all 0: the generic FP64 k_sweep_y) */
int mp_get_scan_geometry(mp_engine *h, int *out4);
/* micro-benchmarks on the engine's device: out[0] MUFU.EX2 Gop/s, out[1] FP32 FMA GFMA/s,
 * out[2] FP64 add Gop/s, out[3] device copy GB/s (read+write) */
int mp_probe_peaks(mp_engine *h, double *out4);

#ifdef __cplusplus
}
#endif
#endif /* LIBMIDASPOM_CUDA_H */
