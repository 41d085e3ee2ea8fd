/* driver/midaspom.c -- command-line driver with the flags and file formats of MIDASPOM.out
 * (reference: sources/main_MIDASPOM.c), calling the B200 engine through the C ABI
 * (include/libmidaspom_cuda.h) where the reference has its grid loops, compPePc and cblas_dgemm
 * (main_MIDASPOM.c:341-395).
 *
 *   midaspom -m 400 -d 100 -i occupancies.txt -o posterior.txt          (same flags: m p d i o s l u)
 *
 * Default mode = the reference's computation: exact likelihood on the s x s grid of (e, c)
 * (mp_exact_posterior), trapezoid normalisation, table written with "%.20lf\t".
 * Extra flags (letters the reference does not use) select the sampler instead of the grid:
 *   -n SWEEPS   run data-augmented MCMC (mp_sweep) and histogram the (e, c) draws onto the same
 *               s x s grid, so the reference's R scripts read the file unchanged
 *   -c CHAINS   chains (default 8)      -b BURNIN  sweeps discarded (default SWEEPS/5)
 *   -r SEED     Philox seed (default 1) -g DEVICE  CUDA ordinal (default 0)
 *   -t FILE     also write the raw draws (one row per sweep and chain)
 *   -O FILE     also write the posterior occupancy of every patch-year after the burn-in (mp_set_summaries): the T x N
 *               table of P(z_tk = 1 | data), rows = years and columns = patches as in the input, "%.20lf\t" like -o
 *   -G 0,1,2,3  run the chains on several GPUs: the drop-in for `mpirun -np 4 MIDASPOM_MPI.out` (run_examples_MPI.sh:8).
 *               Where MIDASPOM_MPI splits the rows of the (e, c) grid over ranks and rank 0 collects them with MPI_Send /
 *               MPI_Recv (main_MIDASPOM_MPI.c:361-372,483-505), the chains are split over the listed devices (device g
 *               holds the global chains g*C/G ... ), sweep concurrently, and one NCCL all-gather inside the library
 *               (mp_comm_init_all + mp_gather_draws_all) brings the draws together.  Needs -n.
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>

#include "../include/libmidaspom_cuda.h"
#include "mp_io.h"

static int run_grid(const int8_t *obs, int tmax, int n, double a, double d, float prioroc, int nstep, double ecmin,
                    double ecmax, int device, const char *fout)
{
    double *lik = (double *)malloc((size_t)nstep * nstep * sizeof(double));
    double ltot = 0.0;
    int info[4];
    printf("Starting parallel likelihood computation\n");
    int rc = mp_exact_posterior(device, obs, tmax, n, a, d, prioroc, nstep, ecmin, ecmax, lik, &ltot, info);
    if (rc != MP_OK) { fprintf(stderr, "mp_exact_posterior failed (%d): %s\n", rc, mp_exact_last_error()); free(lik); return 2; }
    printf("Number of states to compute: %d\n", info[1]);
    for (int ie = 0; ie < nstep; ie++) printf("%.2f%% done\n", ((float)ie + 1) * 100.0 / nstep);
    printf("end likelihood computation\n");
    printf("Total log-likelihood=%.5lf\n", ltot);
    printf("Writing output in file %s... ", fout);
    for (long i = 0; i < (long)nstep * nstep; i++) lik[i] = exp(lik[i] - ltot);     /* main_MIDASPOM.c:432 */
    rc = mp_write_table(fout, lik, nstep, nstep);
    free(lik);
    if (rc) return 3;
    printf("done\n");
    return 0;
}

#define MAXDEV 16
static int run_mcmc(const int8_t *obs, int tmax, int n, double a, double d, float prioroc, int nstep, double ecmin,
                    double ecmax, const int *devices, int ndev, const char *fout, int nsweeps, int nchains, int burn, unsigned long long seed,
                    const char *fdraws, const char *focc)
{
    const int cpg = nchains / ndev;                                   /* chains per GPU (main checked divisibility) */
    mp_engine *hs[MAXDEV] = { NULL };
    int rc = 2;
    mp_sampler_config sc;
    memset(&sc, 0, sizeof sc);
    sc.e_min = ecmin; sc.e_max = ecmax; sc.c_min = ecmin; sc.c_max = ecmax;     /* uniform prior on the grid's square (:312-319) */
    sc.alpha_min = a; sc.alpha_max = a; sc.b_min = 0; sc.b_max = 0; sc.p_min = 1; sc.p_max = 1;
    sc.sample_e = 1; sc.sample_c = 1; sc.n_e_steps = 4; sc.n_c_steps = 2; sc.n_adapt = burn; sc.update_z = 1; sc.update_y = 1;
    mp_params *par = (mp_params *)calloc((size_t)cpg, sizeof(mp_params));
    for (int c = 0; c < cpg; c++) { par[c].e = 0.5 * (ecmin + ecmax); par[c].c = 0.5 * (ecmin + ecmax); par[c].alpha = a; par[c].p = 1; par[c].K = 1; }
    /* draws of all chains, [sweep][global chain][MP_NDRAW]; gathered per device as [device][sweep][local chain] first */
    double *gath = (double *)malloc((size_t)nsweeps * nchains * MP_NDRAW * sizeof(double));
    double *draws = (double *)malloc((size_t)nsweeps * nchains * MP_NDRAW * sizeof(double));
    double *dens = (double *)calloc((size_t)nstep * nstep, sizeof(double));
    double *occ = focc ? (double *)calloc((size_t)tmax * n * 2, sizeof(double)) : NULL;   /* sum over devices, one device's sums */
    for (int g = 0; g < ndev; g++) {
        mp_config cfg;
        memset(&cfg, 0, sizeof cfg);
        cfg.n_patches = n; cfg.n_years = tmax; cfg.n_chains = cpg; cfg.chain_offset = g * cpg; cfg.precision = MP_FP64; cfg.device = devices[g];
        cfg.max_draws = nsweeps; cfg.seed = seed; cfg.prior_occ = prioroc;
        if (mp_create(&cfg, &hs[g]) != MP_OK) { fprintf(stderr, "mp_create (device %d): %s\n", devices[g], mp_last_error(NULL)); goto out; }
        if (mp_set_landscape_linear(hs[g], d, NULL) || mp_set_source_units(hs[g], NULL) || mp_set_observations(hs[g], obs) ||
            mp_set_params(hs[g], par) || mp_init_chains(hs[g], &sc, 1) || (focc && mp_set_summaries(hs[g], burn, 1))) {
            fprintf(stderr, "setup: %s\n", mp_last_error(hs[g])); goto out;
        }
    }
    if (ndev > 1 && mp_comm_init_all(hs, ndev)) { fprintf(stderr, "mp_comm_init_all: %s %s\n", mp_last_error(hs[0]), mp_comm_last_error()); goto out; }
    printf("Starting MCMC: %d chains x %d sweeps (%d burn-in) on %d GPU%s\n", nchains, nsweeps, burn, ndev, ndev > 1 ? "s" : "");
    for (int g = 0; g < ndev; g++)                                    /* asynchronous: the devices sweep concurrently */
        if (mp_sweep(hs[g], nsweeps)) { fprintf(stderr, "sweep: %s\n", mp_last_error(hs[g])); goto out; }
    for (int g = 0; g < ndev; g++) if (mp_synchronize(hs[g])) { fprintf(stderr, "sweep: %s\n", mp_last_error(hs[g])); goto out; }
    if (ndev > 1) {
        if (mp_gather_draws_all(hs, ndev, 0, nsweeps, gath)) { fprintf(stderr, "gather: %s\n", mp_last_error(hs[0])); goto out; }
        for (int g = 0; g < ndev; g++)
            for (int s = 0; s < nsweeps; s++)
                memcpy(draws + ((size_t)s * nchains + (size_t)g * cpg) * MP_NDRAW, gath + (((size_t)g * nsweeps + s) * cpg) * MP_NDRAW,
                       (size_t)cpg * MP_NDRAW * sizeof(double));
    } else if (mp_get_draws(hs[0], 0, nsweeps, draws)) { fprintf(stderr, "draws: %s\n", mp_last_error(hs[0])); goto out; }
    {
        /* histogram on the reference's grid: node i collects draws within half a window, edge nodes half
         * as wide -- the cells the trapezoid weights of :418-421 stand for */
        const double win = (ecmax - ecmin) / (nstep - 1);
        double me = 0, mc = 0; long cnt = 0;
        for (int s = burn; s < nsweeps; s++)
            for (int c = 0; c < nchains; c++) {
                const double *dr = draws + ((size_t)s * nchains + c) * MP_NDRAW;
                int ie = (int)floor((dr[0] - ecmin) / win + 0.5), ic = (int)floor((dr[1] - ecmin) / win + 0.5);
                ie = ie < 0 ? 0 : (ie > nstep - 1 ? nstep - 1 : ie);
                ic = ic < 0 ? 0 : (ic > nstep - 1 ? nstep - 1 : ic);
                dens[(size_t)ie * nstep + ic] += 1.0; me += dr[0]; mc += dr[1]; cnt++;
            }
        for (int i = 0; i < nstep; i++)
            for (int j = 0; j < nstep; j++) {
                double w = win * win;
                if (i == 0 || i == nstep - 1) w *= 0.5;
                if (j == 0 || j == nstep - 1) w *= 0.5;
                dens[(size_t)i * nstep + j] /= (double)cnt * w;        /* density: trapezoid sum * win^2 == 1 */
            }
        printf("posterior means: e=%.5lf c=%.5lf (%ld draws)\n", me / cnt, mc / cnt, cnt);
    }
    printf("Writing output in file %s... ", fout);
    if (mp_write_table(fout, dens, nstep, nstep)) goto out;
    printf("done\n");
    if (focc) {
        /* Rao-Blackwellised occupancy, summed over the devices' chains (each device holds its own chains' sums) */
        const size_t cells = (size_t)tmax * n;
        int64_t ns = 0;
        for (int g = 0; g < ndev; g++) {
            int64_t nsg = 0;
            if (mp_get_summaries(hs[g], &nsg, NULL, occ + cells, NULL, NULL, 0)) { fprintf(stderr, "summaries: %s\n", mp_last_error(hs[g])); goto out; }
            for (size_t i = 0; i < cells; i++) occ[i] += occ[cells + i];
            ns += nsg;
        }
        for (size_t i = 0; i < cells; i++) occ[i] = ns > 0 ? occ[i] / (double)ns : 0.0;
        printf("Writing posterior occupancy (%lld samples) in file %s... ", (long long)ns, focc);
        if (mp_write_table(focc, occ, tmax, n)) goto out;
        printf("done\n");
    }
    if (fdraws) {
        FILE *f = fopen(fdraws, "wb");
        if (f) {
            fprintf(f, "sweep\tchain\te\tc\talpha\tb\tp\tloglik\tny1\tnz1\n");
            for (int s = 0; s < nsweeps; s++)
                for (int c = 0; c < nchains; c++) {
                    const double *dr = draws + ((size_t)s * nchains + c) * MP_NDRAW;
                    fprintf(f, "%d\t%d\t%.10g\t%.10g\t%.10g\t%.10g\t%.10g\t%.10g\t%.0f\t%.0f\n", s, c, dr[0], dr[1], dr[2], dr[3], dr[4], dr[5], dr[6], dr[7]);
                }
            fclose(f);
        }
    }
    rc = 0;
out:
    free(par); free(draws); free(gath); free(dens); free(occ);
    for (int g = 0; g < ndev; g++) if (hs[g]) mp_destroy(hs[g]);
    return rc;
}

int main(int argc, char **argv)
{
    printf("------ MIDASPOM on B200 (midaspom_b200; model and formats of MIDASPOM beta, Alcala, Cole & Rosenberg) ------\n");
    float prioroc = 0.5f;                 /* defaults of main_MIDASPOM.c:66-73 */
    const char *fname = "input.txt", *fout = "posterior.txt", *fdraws = NULL, *focc = NULL;
    double d = 100, a = 1.0 / 400, ecmin = 0.0, ecmax = 1.0;
    int nstep = 101, nsweeps = 0, nchains = 8, burn = -1, device = 0, c;
    unsigned long long seed = 1;
    int devices[MAXDEV], ndev = 0;
    opterr = 0;
    while ((c = getopt(argc, argv, "m:p:d:i:o:s:l:u:n:c:b:r:g:t:G:O:")) != -1)
        switch (c) {
        case 'm': a = 1.0 / atof(optarg); break;
        case 'p': prioroc = (float)atof(optarg); break;
        case 'd': d = atof(optarg); break;
        case 'i': fname = optarg; break;
        case 'o': fout = optarg; break;
        case 's': nstep = atoi(optarg); break;
        case 'l': ecmin = atof(optarg); break;
        case 'u': ecmax = atof(optarg); break;
        case 'n': nsweeps = atoi(optarg); break;
        case 'c': nchains = atoi(optarg); break;
        case 'b': burn = atoi(optarg); break;
        case 'r': seed = strtoull(optarg, NULL, 10); break;
        case 'g': device = atoi(optarg); break;
        case 't': fdraws = optarg; break;
        case 'O': focc = optarg; break;
        case 'G':
            for (char *tok = strtok(optarg, ","); tok && ndev < MAXDEV; tok = strtok(NULL, ",")) devices[ndev++] = atoi(tok);
            break;
        default: fprintf(stderr, "Unknown option `-%c'.\n", optopt); return 1;
        }
    if (nstep < 2) { fprintf(stderr, "-s must be at least 2\n"); return 1; }
    if (ndev == 0) { devices[0] = device; ndev = 1; }
    if (focc && nsweeps <= 0) { fprintf(stderr, "-O needs -n SWEEPS (the occupancy comes from the chains)\n"); return 1; }
    if (ndev > 1 && (nsweeps <= 0 || nchains % ndev)) { fprintf(stderr, "-G needs -n SWEEPS and a chain count divisible by the number of GPUs\n"); return 1; }
    const double win = (ecmax - ecmin) / (nstep - 1);
    printf("Parameters for numerical approximation of the posterior density:\n\tWindow size=%lf, number of steps=%d\n", win, nstep);
    time_t start = time(NULL);
    printf("Reading observations from file %s... ", fname);
    int8_t *obs = NULL; int n = 0, tmax = 0;
    if (mp_read_occupancy(fname, &obs, &n, &tmax)) return 1;
    printf("done\n");
    printf("Number of habitat patches: %d\nNumber of sampled years: %d\n", n, tmax);
    if (tmax < 2) { fprintf(stderr, "need at least two sampled years\n"); free(obs); return 1; }
    printf("Dispersal matrix:\n");                                                  /* main_MIDASPOM.c:180-195 */
    for (int i = 0; i < n && n <= 64; i++) {
        for (int j = 0; j < n; j++) printf("%.3f ", i == j ? 0.0 : exp(-a * abs(j - i) * d));
        printf("\n");
    }
    printf("Input occupancy data:\n");
    for (int i = 0; i < tmax; i++) {
        printf("Year %d: ", i);
        for (int j = 0; j < n && n <= 256; j++) printf("%d ", obs[(size_t)i * n + j]);
        printf("\n");
    }
    printf("Number of possible states per year:\n");
    for (int i = 0; i < tmax; i++) {
        int s1 = 0;
        for (int j = 0; j < n; j++) s1 += obs[(size_t)i * n + j] == -1;
        if (s1 < 31) printf("Year %d: %d\n", i, 1 << s1); else printf("Year %d: 2^%d\n", i, s1);
    }
    setbuf(stdout, NULL);
    int rc;
    if (nsweeps > 0) {
        if (burn < 0) burn = nsweeps / 5;
        rc = run_mcmc(obs, tmax, n, a, d, prioroc, nstep, ecmin, ecmax, devices, ndev, fout, nsweeps, nchains, burn, seed, fdraws, focc);
    } else rc = run_grid(obs, tmax, n, a, d, prioroc, nstep, ecmin, ecmax, devices[0], fout);
    free(obs);
    printf(" Total running time: %.2lf min\n", difftime(time(NULL), start) / 60.0);
    return rc;
}
