// mp_engine.cu -- host side of libmidaspom_cuda.so: the engine handle, device memory, kernel
// launch sequences and the extern "C" entry points declared in include/libmidaspom_cuda.h.
// No CPU fallback: without a usable sm_100 device every entry point returns MP_ERR_CUDA.
#include "mp_host.h"
#include "mp_kernels.cuh"
#include "mp_sweep_cull.cuh"   // k_build_candidates, CandRec, BlockTask, k_block_valid
#include "mp_comm.h"
#include "mp_capacity.cuh"
#include "mp_sources.cuh"

using namespace mp;

static thread_local std::string g_create_error;

// device copies of the sweep and draw counters (after the host changed them: mp_init_chains, mp_reset_draws)
static int push_counters(mp_engine *h)
{
    CK(cudaSetDevice(h->cfg.device));
    const uint32_t v[2] = { h->sweep, (uint32_t)h->ndraws };
    CK(cudaMemcpyAsync(h->d_ctr, v, sizeof v, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MP_OK;
}
// captured sweeps depend on everything a launch takes by value: drop them whenever a setter changes the engine
static void drop_graphs(mp_engine *h)
{
    for (int v = 0; v < 2; v++) { if (h->gexec[v]) { cudaGraphExecDestroy(h->gexec[v]); h->gexec[v] = nullptr; } h->gwarm[v] = false; }
}

static SamplerDev sampler_dev(const mp_engine *h)
{
    SamplerDev sd;
    sd.sc = h->sc; sd.seed = h->cfg.seed; sd.chain_offset = h->cfg.chain_offset; sd.detect = h->cfg.detect;
    sd.p0 = (double)(float)h->cfg.prior_occ;   // float in the reference (main_MIDASPOM.c:66,218)
    return sd;
}

// ------------------------------------------------------------------ launch helpers
template <typename R> static int launch_area_weights(mp_engine *h, int set)
{
    Timed tm(h, MP_K_SMALL);
    const int n = h->cfg.n_patches;
    dim3 grid((n + 255) / 256, h->cfg.n_chains);
    k_area_weights<R><<<grid, 256, 0, h->stream>>>(set ? h->d_prop : h->d_par, h->have_area ? h->d_area : nullptr,
                                                    (R *)h->d_aw[set], n);
    CK(cudaGetLastError());
    return MP_OK;
}
// source records of k_conn (scan order; year bits + coordinates + area constant) for the parameter sets in set_mask
template <typename R> static int launch_pack_sources(mp_engine *h, int set_mask)
{
    Timed tm(h, MP_K_SMALL);
    const int npad = conn_npad(h->cfg.n_patches);
    dim3 grid((npad + 255) / 256, h->cfg.n_chains, h->nwords);
    mp::Landscape<R> ls = view<R>(h);
    if (h->geom != MP_GEOM_COORDS) { ls.px = nullptr; ls.py = nullptr; }
    k_pack_sources<R><<<grid, 256, 0, h->stream>>>(ls, h->d_perm, (const R *)h->d_aw[0], (const R *)h->d_aw[1], h->d_y,
                                                    h->cfg.n_years - 1, h->nwords, set_mask, (SrcRec<R> *)h->d_srec);
    CK(cudaGetLastError());
    return MP_OK;
}
// k_conn over the buffers of `a` (sets [a.set_base, a.set_base + nsets), every chain of a.nchains).  a32: the evaluation form
// with the year contraction on the FP32 pipe (FP32 engines); otherwise the DFMA form.
template <typename R, int GEOM> static int launch_conn_args(mp_engine *h, const ConnArgs<R> &a, int nsets, bool a32)
{
    if (a.k_hi <= a.k_lo) return MP_OK;
    const int ny = a.ntrans;                          // year accumulators per target: next multiple of 4 (<= 32 per pass)
    // FP32 engines on landscapes with positions skip source tiles out of reach (see CONN_CULL_LOG2); FP64 never culls
    constexpr bool CAN_CULL = sizeof(R) == 4 && GEOM != MP_GEOM_DENSE;
    const bool cull = CAN_CULL && h->conn_cull && h->have_boxes;
    // CTA shape: 128 threads x 2 targets; with few CTAs per SM, 64 or 32 threads x 2 targets (2x / 4x the CTAs) balance the
    // unequal (culled) work better, and the FP32 engines go on to 32 threads x 1 target (8x the CTAs, 96 registers: cfg3 with
    // 8 chains 1.41 -> 1.25 ms per launch; no difference at cfg5).  Every shape gives bit-identical sums.  MP_CONN_SHAPE=1|2|3|4
    // forces a shape.
    const long long wide_ctas = (long long)((a.k_hi - a.k_lo + 255) / 256) * a.nchains * nsets;
    // shape 1: 128 threads, 2: 64 threads, 3: 32 threads (2 targets per thread each), 4: 32 threads x 1 target (FP32 engines)
    int shape = h->conn_shape ? h->conn_shape : wide_ctas >= 16LL * h->sm_count ? 1 : wide_ctas >= 4LL * h->sm_count ? 2 : 4;
    if (shape == 4 && (sizeof(R) != 4 || a32)) shape = 3;
    const int per_cta = shape == 1 ? 256 : shape == 2 ? 128 : shape == 3 ? 64 : 32;
    dim3 grid((a.k_hi - a.k_lo + per_cta - 1) / per_cta, a.nchains, nsets);
    if (sizeof(R) == 4 && a32) return mp_launch_conn32(h, &a, GEOM, ny, shape, cull ? 1 : 0, grid.x, grid.y, grid.z);
#define MP_CONN_T(NYB, NT) do { if (cull) k_conn<R, GEOM, NYB, CAN_CULL, 2, NT><<<grid, NT, 0, h->stream>>>(a);      \
                                else k_conn<R, GEOM, NYB, false, 2, NT><<<grid, NT, 0, h->stream>>>(a); } while (0)
#define MP_CONN_ONE(NYB) do { if constexpr (sizeof(R) == 4) { if (cull) k_conn<R, GEOM, NYB, CAN_CULL, 1, 32><<<grid, 32, 0, h->stream>>>(a);   \
                                                              else k_conn<R, GEOM, NYB, false, 1, 32><<<grid, 32, 0, h->stream>>>(a); } } while (0)
#define MP_CONN(NYB) do { if (shape == 1) MP_CONN_T(NYB, 128); else if (shape == 2) MP_CONN_T(NYB, 64); else if (shape == 3) MP_CONN_T(NYB, 32); \
                          else MP_CONN_ONE(NYB); } while (0)
    if (ny <= 4) MP_CONN(4); else if (ny <= 8) MP_CONN(8); else if (ny <= 12) MP_CONN(12); else if (ny <= 16) MP_CONN(16);
    else if (ny <= 20) MP_CONN(20); else if (ny <= 24) MP_CONN(24); else if (ny <= 28) MP_CONN(28); else MP_CONN(32);
#undef MP_CONN
#undef MP_CONN_ONE
#undef MP_CONN_T
    CK(cudaGetLastError());
    return MP_OK;
}
template <typename R, int GEOM> static int launch_conn_g(mp_engine *h, int set_base, int nsets, bool eval)
{
    Timed tm(h, MP_K_CONN);
    ConnArgs<R> a;
    a.ls = view<R>(h);
    a.par[0] = h->d_par; a.par[1] = h->d_prop;
    a.S[0] = h->d_S[0]; a.S[1] = h->d_S[1];
    a.rec = (const SrcRec<R> *)h->d_srec;
    a.ntrans = h->cfg.n_years - 1; a.nwords = h->nwords; a.nchains = h->cfg.n_chains; a.set_base = set_base;
    a.k_lo = h->conn_lo; a.k_hi = h->conn_hi < 0 ? h->cfg.n_patches : h->conn_hi;
    a.perm = h->d_perm; a.box32 = (const float4 *)h->d_tile_box;
    a.mlow = h->d_mlow; a.area_max = (float)h->area_max; a.area_min = (float)h->area_min;   // bounds: launch_conn_bounds
    a.stats = h->d_work;
    // Evaluation entry points of the FP32 engines (mp_connectivity, mp_loglik, mp_loglik_host): the year contraction on the FP32
    // pipe (FFMA2, FP32 partial sums per 32 sources joined in FP64; mp_conn32.cu), accurate to ~1e-7 of every S.  The sampler's
    // own S keeps the DFMA form: a weight the y scan later removes must cancel to the last bit even where S then falls
    // by orders of magnitude.  MP_CONN_ACC32=0 keeps the DFMA form everywhere.
    const bool a32 = sizeof(R) == 4 && eval && h->conn_acc32;
    if (a32 && a.k_hi > a.k_lo) h->S_exact = false;
    return launch_conn_args<R, GEOM>(h, a, nsets, a32);
}
// Culling bounds of k_conn: a lower bound of every target group's S, taken from the resident S BEFORE it is overwritten
// or zeroed (none before the first refresh: mlow = 0, nothing is skipped).
static int launch_conn_bounds(mp_engine *h)
{
    if (is64(h) || h->geom == MP_GEOM_DENSE || !h->conn_cull || !h->have_boxes) return MP_OK;
    Timed tm(h, MP_K_SMALL);
    k_group_min_S<<<dim3((h->cfg.n_patches + 31) / 32, h->cfg.n_chains), 32, 0, h->stream>>>(h->d_S[0], h->d_perm, h->cfg.n_patches,
                                                                                             h->cfg.n_years - 1, h->S_valid ? 1 : 0, h->d_mlow);
    CK(cudaGetLastError());
    return MP_OK;
}
// sets [set_base, set_base + nsets): 0 = resident parameters -> S, 1 = proposal -> S_prop
// eval: the call serves an evaluation entry point (FP32 engines may take the FP32 contraction), not the sampler's resident S
template <typename R> static int launch_conn(mp_engine *h, int set_base, int nsets, bool eval = false)
{
    if (nsets <= 0) return MP_OK;
    switch (h->geom) {
    case MP_GEOM_LINEAR: return launch_conn_g<R, MP_GEOM_LINEAR>(h, set_base, nsets, eval);
    case MP_GEOM_COORDS: return launch_conn_g<R, MP_GEOM_COORDS>(h, set_base, nsets, eval);
    default: return launch_conn_g<R, MP_GEOM_DENSE>(h, set_base, nsets, eval);
    }
}
// colonisation log-likelihood partials: set s uses parameters par_s, connectivity S_s, writes partial[s]
template <typename R>
static int launch_col(mp_engine *h, int nsets, const mp_params *p0, const double *S0, const mp_params *p1, const double *S1)
{
    Timed tm(h, MP_K_COL);
    ColArgs a;
    a.par[0] = p0; a.par[1] = p1; a.S[0] = S0; a.S[1] = S1;
    a.partial[0] = h->d_partial[0]; a.partial[1] = h->d_partial[1];
    dim3 grid(h->nblk_col, h->cfg.n_chains, nsets);
    k_col_ll<R><<<grid, COL_THREADS, 0, h->stream>>>(a, view<R>(h), h->d_z, h->d_y, h->have_era ? h->d_era : nullptr,
                                                     h->cfg.n_years);
    CK(cudaGetLastError());
    return MP_OK;
}
static int launch_counts(mp_engine *h)
{
    Timed tm(h, MP_K_SMALL);
    CK(cudaMemsetAsync(h->d_counts, 0, nC(h) * NCOUNT * sizeof(unsigned long long), h->stream));
    const long long cells = (long long)zcells(h);
    dim3 grid((unsigned)std::min<long long>((cells + 255) / 256, 1024), h->cfg.n_chains);
    k_counts<<<grid, 256, 0, h->stream>>>(h->d_obs, h->have_era ? h->d_era : nullptr, h->d_z, h->d_y, h->d_counts,
                                          h->cfg.n_patches, h->cfg.n_years, h->cfg.detect);
    CK(cudaGetLastError());
    return MP_OK;
}
template <typename R, int GEOM> static int launch_sweep_y_g(mp_engine *h)
{
    Timed tm(h, MP_K_SWEEP_Y);
    constexpr int NT = sizeof(R) == 4 ? 1024 : 512;
    size_t smem = nN(h) * (sizeof(double) + sizeof(R) + 1) + 16;
    const size_t stride = (smem + 255) / 256 * 256;
    const int ntask = h->cfg.n_chains * (h->cfg.n_years - 1);
    // beyond one CTA's shared memory (about 13,600 patches in FP64) the per-task state lives in global scratch (slow, parity only)
    const bool spill = smem > 227 * 1024;
    if (spill && !h->d_scan_work) CK(cudaMalloc(&h->d_scan_work, stride * (size_t)ntask));
    if (spill) smem = 16;
    auto kern = k_sweep_y<R, GEOM, NT>;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int nthr = (int)std::min<size_t>(NT, ((nN(h) + 31) / 32) * 32);
    kern<<<ntask, nthr, smem, h->stream>>>(
        sampler_dev(h), h->d_ctr, view<R>(h), h->d_par, (const R *)h->d_aw[0], h->have_era ? h->d_era : nullptr, h->d_z,
        h->d_y, h->d_S[0], h->cfg.n_years, (const int *)h->d_scan, h->d_work, spill ? h->d_scan_work : nullptr, stride);
    CK(cudaGetLastError());
    return MP_OK;
}
// ---- FP32 fast path (mp_sweep_fast.cuh; kernels live in mp_sweep_fast_{linear,coords,dense}.cu)
extern "C" { static int build_block_tasks(mp_engine *h); }   // block tasks of the scan grid (mp_set_scan_blocks), defined with the C ABI below
static int pick_cluster(int tasks, int sms, int max_cs)
{
    // split each task over CS CTAs so that tasks*CS fills the SMs evenly; ties -> smaller CS
    int best = 1; double best_cost = 1e30;
    for (int cs = 1; cs <= max_cs; cs *= 2) {
        const int ctas = tasks * cs;
        const double cost = (double)((ctas + sms - 1) / sms) / cs * (1.0 + 0.08 * cs);   // measured: DSMEM sync cost grows with CS
        if (cost < best_cost - 1e-9) { best_cost = cost; best = cs; }
    }
    return best;
}
static bool fast_sweep_ok(const mp_engine *h)
{
    return !is64(h) && h->cfg.n_patches <= 113000;    // 2 N bytes of shared memory per CTA in a cluster of 8
}
static int launch_sweep_y_fast(mp_engine *h)
{
    const int n = h->cfg.n_patches, ntrans = h->cfg.n_years - 1, C = h->cfg.n_chains;
    {
        Timed tm(h, MP_K_SMALL);
        const int ntask = (C * ntrans - h->task_first + h->task_stride - 1) / h->task_stride;
        if (ntask <= 0) return MP_OK;
        k_build_candidates<<<ntask, 1024, 0, h->stream>>>(h->cfg.seed, h->cfg.chain_offset, h->d_ctr, view<float>(h),
                                                           (const float *)h->d_aw[0], h->d_z, h->d_y, (CandRec *)h->d_cand,
                                                           h->d_cand_count, h->cfg.n_years, h->geom == MP_GEOM_COORDS,
                                                           h->task_first, h->task_stride, h->d_scan, h->d_minv);
        CK(cudaGetLastError());
        k_order_tasks<<<1, 1024, 0, h->stream>>>(h->d_cand_count, ntask, h->task_first, h->task_stride, h->d_task_order);
        CK(cudaGetLastError());
    }
    Timed tm(h, MP_K_SWEEP_Y);
    // threads per task, from measurements: 256 (one CTA, no DSMEM) up to 3,000 patches (cfg2: 0.27 vs 0.35 ms),
    // 512 up to 15,872 (cfg3: 15.5 vs 18.7 ms for 1024)
    int tpt = h->fast_tpt ? h->fast_tpt : (n <= 3000 ? 256 : 512);
    if ((n + tpt - 1) / tpt > 31) tpt = 1024;
    for (int big = 2048; (n + tpt - 1) / tpt > 31 && big <= 8192; big *= 2) tpt = big;   // N > 31k: 2048..8192 threads, cluster of 8
    // large landscapes: a cluster of 8 holds the task's state; with few tasks per GPU (year sharding) spread each
    // task over 16 SMs instead -- the scan is latency-bound per flip
    const int ntask_own = (C * ntrans - h->task_first + h->task_stride - 1) / h->task_stride;
    // exact spatial culling of the evaluation (mp_sweep_cull.cuh) where positions exist and the landscape is large
    const bool culled = h->geom != MP_GEOM_DENSE && tpt >= 512;
    // the culled scan at 512 threads per task runs in clusters of 4 x 128 threads whatever the task count: up to five such CTAs
    // of different tasks share an SM, and their independent trips cover each other's latency.  Measured at cfg3 (one B200,
    // 1,000 W), ms per launch for CS = 1 / 2 / 4 / 8: 64 chains 60.1 / 60.2 / 56.2 / 62.8, 32 chains 32.1 / 32.3 / 29.4 / 32.9,
    // 16 chains 17.7 / 18.0 / 15.3 / 18.6, 8 chains 9.8 / 9.9 / 8.5 / 11.0 (pick_cluster's wave model chose 1, 2, 2 and 4)
    int cs = tpt > 1024 ? (h->fast_cs == 16 || (h->fast_cs == 0 && tpt >= 4096 && ntask_own * 16 <= h->sm_count) ? 16 : 8)
                        : (h->fast_cs ? h->fast_cs : (tpt == 256 ? 1 : culled && tpt == 512 ? 4 : pick_cluster(C * ntrans, h->sm_count, 8)));
    // a CTA holds 16 bytes per target of its share (+ the 2 KB record ring of the culled scan): widen the cluster until that fits
    if (tpt >= 512 && tpt <= 1024) {
        const size_t ept = (size_t)(n + tpt - 1) / tpt;
        while (cs < 8 && ept * (size_t)(tpt / cs) * 16 + 2048 > 227 * 1024) cs *= 2;
    }
    h->last_scan[0] = tpt; h->last_scan[1] = cs; h->last_scan[2] = culled ? (tpt > 1024 ? 4 : 2) : 1; h->last_scan[3] = culled;
    if (culled && h->blk_active) {
        // block grid: decide per task whether its halo suffices this sweep, scan those tasks colour by colour (the blocks of
        // one colour concurrently), then the remaining tasks as whole years (clusters of the other kind return at once)
        int rc;
        if (h->blk_tasks_dirty && (rc = build_block_tasks(h)) != MP_OK) return rc;
        k_block_valid<<<ntask_own, 256, 0, h->stream>>>(h->d_S[0], h->d_par, h->d_cand_count, n, ntrans, h->task_first, h->task_stride,
                                                        h->blk_halo, std::log2(h->area_max), std::log2(h->area_min), h->d_blockmode);
        CK(cudaGetLastError());
        // threads per block task: the smallest of 512 ... 8192 that keeps 31 slots per thread; cluster as wide as the shared memory asks
        int btpt = h->blk_tpt ? h->blk_tpt : 512;
        while ((h->blk_nl_max + btpt - 1) / btpt > 31 && btpt < 8192) btpt *= 2;
        int bcs = btpt > 1024 ? 8 : (h->blk_cs ? h->blk_cs : 4);
        if (btpt <= 1024) {
            const size_t ept = (size_t)(h->blk_nl_max + btpt - 1) / btpt;
            while (bcs < 8 && ept * (size_t)(btpt / bcs) * 16 + 2048 > 227 * 1024) bcs *= 2;
        }
        h->last_scan[0] = btpt; h->last_scan[1] = bcs; h->last_scan[2] = btpt > 1024 ? 4 : 2; h->last_scan[3] = 2;
        for (size_t col = 0; col < h->colour_n.size(); col++) {
            if (h->colour_n[col] == 0) continue;
            const void *bt = (const char *)h->d_btasks + (size_t)h->colour_off[col] * sizeof(mp::BlockTask);
            if ((rc = mp_launch_sweep_cull_coords(h, bcs, btpt, h->blk_nl_max, h->colour_n[col], bt)) != MP_OK) return rc;
        }
    }
    if (culled)
        return h->geom == MP_GEOM_LINEAR ? mp_launch_sweep_cull_linear(h, cs, tpt, n, ntask_own, nullptr)
                                         : mp_launch_sweep_cull_coords(h, cs, tpt, n, ntask_own, nullptr);
    switch (h->geom) {
    case MP_GEOM_LINEAR: return mp_launch_sweep_fast_linear(h, cs, tpt);
    case MP_GEOM_COORDS: return mp_launch_sweep_fast_coords(h, cs, tpt);
    default: return mp_launch_sweep_fast_dense(h, cs, tpt);
    }
}
template <typename R> static int launch_sweep_y(mp_engine *h)
{
    if (fast_sweep_ok(h)) return launch_sweep_y_fast(h);
    REQUIRE(h->task_first == 0 && h->task_stride == 1, MP_ERR_UNSUPPORTED, "year sharding needs the FP32 fast sweep");
    switch (h->geom) {
    case MP_GEOM_LINEAR: return launch_sweep_y_g<R, MP_GEOM_LINEAR>(h);
    case MP_GEOM_COORDS: return launch_sweep_y_g<R, MP_GEOM_COORDS>(h);
    default: return launch_sweep_y_g<R, MP_GEOM_DENSE>(h);
    }
}
template <typename R> static int launch_update_z(mp_engine *h)
{
    Timed tm(h, MP_K_SWEEP_Z);
    const long long cells = (long long)zcells(h);
    dim3 grid((unsigned)std::min<long long>((cells + 255) / 256, 2048), h->cfg.n_chains);
    k_update_z<R><<<grid, 256, 0, h->stream>>>(sampler_dev(h), h->d_ctr, view<R>(h), h->d_par, h->d_obs,
                                               h->have_era ? h->d_era : nullptr, h->d_z, h->d_y, h->d_S[0], h->cfg.n_years);
    CK(cudaGetLastError());
    return MP_OK;
}

// every chain holds the same (alpha, b), known on the host: the connectivity is one dense contraction (mp_conn_gemm.cu)
static bool gemm_eligible(const mp_engine *h)
{
    if (is64(h) || !h->use_gemm || h->geom == MP_GEOM_DENSE || h->conn_hi >= 0 || !h->par_host_valid) return false;
    if (h->cfg.n_patches < h->gemm_min_n || h->par_host.size() != nC(h)) return false;
    for (size_t c = 1; c < nC(h); c++)
        if (h->par_host[c].alpha != h->par_host[0].alpha || h->par_host[c].b != h->par_host[0].b) return false;
    return true;
}
// recompute S (set 0) from the resident y and parameters; allow_gemm: for an evaluation entry point (the FP32 engines may then
// take the tensor-core path or the FP32 contraction of k_conn, after which the next sweep recomputes the sampler's S)
template <typename R> static int refresh_S(mp_engine *h, bool allow_gemm = true)
{
    int rc;
    if ((rc = launch_area_weights<R>(h, 0)) != MP_OK) return rc;
    if (allow_gemm && gemm_eligible(h)) {
        if ((rc = mp_launch_conn_gemm(h, h->par_host[0].alpha)) != MP_OK) return rc;
        h->S_valid = true; h->S_exact = false; h->last_conn_path = 1;
        return MP_OK;
    }
    h->last_conn_path = 0;
    if ((rc = launch_pack_sources<R>(h, 1)) != MP_OK) return rc;
    if ((rc = launch_conn_bounds(h)) != MP_OK) return rc;
    h->S_exact = true;                                   // launch_conn clears it when it takes the FP32 contraction
    const int rc2 = launch_conn<R>(h, 0, 1, allow_gemm);
    if (rc2 == MP_OK) h->S_valid = true;
    return rc2;
}
// per-chain complete-data log-likelihood of the resident state, using the resident S
template <typename R> static int loglik_resident(mp_engine *h, double *d_draw_row, double *d_parts)
{
    int rc;
    if ((rc = launch_counts(h)) != MP_OK) return rc;
    if ((rc = launch_col<R>(h, 1, h->d_par, h->d_S[0], h->d_par, h->d_S[0])) != MP_OK) return rc;
    Timed tm(h, MP_K_SMALL);
    k_record<<<h->cfg.n_chains, 32, 0, h->stream>>>(sampler_dev(h), h->d_par, h->d_counts, h->d_partial[0], h->nblk_col,
                                                    d_draw_row, d_parts, nullptr, 0);
    CK(cudaGetLastError());
    return MP_OK;
}

// One MCMC iteration of every resident chain, in four phases.  A single engine runs them back to back
// (sweep_once); a chain sharded over several GPUs (distributed.ShardedChain) runs the same phases with a
// collective between them: each rank evaluates its own target patches in phase 0 and its own years in
// phase 2, everything else is replicated and deterministic, so all ranks take identical decisions.
enum { PH_PROPOSE_CONN = 0, PH_DECIDE_Z = 1, PH_SWEEP_Y = 2, PH_FINISH = 3 };

// phase 0: proposal for (alpha, b), connectivity of the proposal (and the periodic refresh of the resident S)
// on the target range [conn_lo, conn_hi).  Returns bit 0 = resident S recomputed, bit 1 = proposal computed.
template <typename R> static int phase_propose_conn(mp_engine *h, int *flags_out)
{
    int rc;
    const int C = h->cfg.n_chains;
    const SamplerDev sd = sampler_dev(h);
    const bool do_ab = h->sc.sample_alpha || h->sc.sample_b;
    const bool sharded = h->conn_hi >= 0;
    if ((rc = launch_area_weights<R>(h, 0)) != MP_OK) return rc;
    if (do_ab) {
        { Timed tm(h, MP_K_SMALL);
          k_propose_ab<<<(C + 63) / 64, 64, 0, h->stream>>>(sd, h->d_ctr, h->d_par, h->d_prop, h->d_lsig, h->d_flags, h->d_logu, C);
          CK(cudaGetLastError()); }
        if ((rc = launch_area_weights<R>(h, 1)) != MP_OK) return rc;
    }
    // The resident S is maintained by exact rank-1 updates; the FP32 engine recomputes it from scratch only
    // every MP_REFRESH_EVERY sweeps (the FP64 parity engine every sweep, like the CPU twin).
    const bool refresh = is64(h) || h->refresh_every <= 1 || (h->sweep % (uint32_t)h->refresh_every) == 0 || !h->S_valid || !h->S_exact;
    if (refresh || do_ab) if ((rc = launch_pack_sources<R>(h, (refresh ? 1 : 0) | (do_ab ? 2 : 0))) != MP_OK) return rc;
    if ((rc = launch_conn_bounds(h)) != MP_OK) return rc;
    if (sharded) {   // other ranks fill the other target columns: start from zeros so that a sum over ranks assembles S
        if (refresh) CK(cudaMemsetAsync(h->d_S[0], 0, nC(h) * ycells(h) * 8, h->stream));
        if (do_ab) CK(cudaMemsetAsync(h->d_S[1], 0, nC(h) * ycells(h) * 8, h->stream));
    }
    if ((rc = launch_conn<R>(h, refresh ? 0 : 1, (refresh ? 1 : 0) + (do_ab ? 1 : 0))) != MP_OK) return rc;
    h->S_valid = true; h->S_exact = true;
    if (flags_out) *flags_out = (refresh ? 1 : 0) | (do_ab ? 2 : 0);
    return MP_OK;
}
// phase 1: Metropolis decisions on (alpha, b) and c, Gibbs update of the latent z cells
template <typename R> static int phase_decide_z(mp_engine *h)
{
    int rc;
    const int C = h->cfg.n_chains;
    const SamplerDev sd = sampler_dev(h);
    const bool do_ab = h->sc.sample_alpha || h->sc.sample_b;
    const long long cells = (long long)ycells(h);
    if (do_ab) {
        Timed tm(h, MP_K_SMALL);
        k_sum_S<<<dim3(h->nblk_col, C, 2), COL_THREADS, 0, h->stream>>>(h->d_S[0], h->d_S[1], cells, h->d_partial[0], h->d_partial[1]);
        CK(cudaGetLastError());
        k_ridge_c<<<C, 32, 0, h->stream>>>(sd, h->d_par, h->d_prop, h->d_partial[0], h->d_partial[1], h->nblk_col, h->d_flags, h->d_ljac);
        CK(cudaGetLastError());
    }
    if ((rc = launch_col<R>(h, do_ab ? 2 : 1, h->d_par, h->d_S[0], h->d_prop, h->d_S[1])) != MP_OK) return rc;
    { Timed tm(h, MP_K_SMALL);
      k_decide_ab<<<C, 32, 0, h->stream>>>(sd, h->d_ctr, h->d_par, h->d_prop, h->d_lsig, h->d_flags, h->d_logu,
                                           h->d_partial[0], h->d_partial[1], h->nblk_col, h->d_llc, do_ab ? 1 : 0, h->d_ljac);
      CK(cudaGetLastError()); }
    if (do_ab) {
        Timed tm(h, MP_K_SMALL);
        dim3 grid((unsigned)std::min<long long>((cells + 255) / 256, 1024), C);
        k_commit_ab<R><<<grid, 256, 0, h->stream>>>(h->d_flags, h->d_S[0], h->d_S[1], (R *)h->d_aw[0], (const R *)h->d_aw[1],
                                                    cells, h->cfg.n_patches);
        CK(cudaGetLastError());
    }
    if (h->sc.sample_c)
        for (int s = 0; s < h->sc.n_c_steps; s++) {
            { Timed tm(h, MP_K_SMALL);
              k_propose_c<<<(C + 63) / 64, 64, 0, h->stream>>>(sd, h->d_ctr, s, h->d_par, h->d_prop, h->d_lsig, h->d_flags, h->d_logu, C);
              CK(cudaGetLastError()); }
            // set 0 := the proposal => partial[0] holds the proposal's sums
            if ((rc = launch_col<R>(h, 1, h->d_prop, h->d_S[0], h->d_prop, h->d_S[0])) != MP_OK) return rc;
            Timed tm(h, MP_K_SMALL);
            k_decide_c<<<C, 32, 0, h->stream>>>(sd, h->d_ctr, h->d_par, h->d_prop, h->d_lsig, h->d_flags, h->d_logu,
                                                h->d_partial[0], h->nblk_col, h->d_llc);
            CK(cudaGetLastError());
        }
    // V: variant parameters (K, Ksrc, dsrc): extinction part from the counts, colonisation part over the cells
    if (h->sc.sample_K || h->sc.sample_Ksrc || h->sc.sample_dsrc) {
        if ((rc = launch_counts(h)) != MP_OK) return rc;
        for (int which = 0; which < 3; which++) {
            const int on = which == 0 ? h->sc.sample_K : which == 1 ? h->sc.sample_Ksrc : h->sc.sample_dsrc;
            if (!on) continue;
            for (int s = 0; s < h->sc.n_v_steps; s++) {
                { Timed tm(h, MP_K_SMALL);
                  k_propose_var<<<(C + 63) / 64, 64, 0, h->stream>>>(sd, h->d_ctr, which, s, h->d_par, h->d_prop, h->d_lsig, h->d_flags, h->d_logu, C);
                  CK(cudaGetLastError()); }
                if ((rc = launch_col<R>(h, 1, h->d_prop, h->d_S[0], h->d_prop, h->d_S[0])) != MP_OK) return rc;
                Timed tm(h, MP_K_SMALL);
                k_decide_var<<<C, 32, 0, h->stream>>>(sd, h->d_ctr, which, h->d_par, h->d_prop, h->d_lsig, h->d_flags, h->d_logu,
                                                      h->d_partial[0], h->nblk_col, h->d_llc, h->d_counts);
                CK(cudaGetLastError());
            }
        }
    }
    if (h->sc.update_z) if ((rc = launch_update_z<R>(h)) != MP_OK) return rc;
    return MP_OK;
}
// phase 2: Gibbs scan of the intermediate states of the (chain, year) tasks owned by this engine
template <typename R> static int phase_sweep_y(mp_engine *h)
{
    if (h->sc.update_y) return launch_sweep_y<R>(h);
    return MP_OK;
}
// ---- posterior summaries (mp_set_summaries): z_prob [T][N], S_sum [T-1][N], z_count [T][N], y_count [T-1][N], sample counter
struct SumLayout { size_t z_prob, S_sum, z_count, y_count, nsamples, bytes; };
static SumLayout sum_layout(const mp_engine *h)
{
    SumLayout L;
    size_t off = 0;
    auto carve = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    L.z_prob = carve(zcells(h) * 8); L.S_sum = carve(ycells(h) * 8); L.z_count = carve(zcells(h) * 4);
    L.y_count = carve(ycells(h) * 4); L.nsamples = carve(8); L.bytes = off;
    return L;
}
static bool summary_due(const mp_engine *h, uint32_t s)
{
    return h->sum_thin > 0 && s >= (uint32_t)h->sum_first && (s - (uint32_t)h->sum_first) % (uint32_t)h->sum_thin == 0;
}
// refuse sweeps that could push the sample counter past the range of the uint32 counts
static int summaries_room(mp_engine *h, int nsweeps)
{
    if (h->sum_thin <= 0 || nsweeps <= 0) return MP_OK;
    // qualifying sweeps first + k thin (k >= 0) in [lo, hi)
    const long long first = h->sum_first, thin = h->sum_thin, hi = (long long)h->sweep + nsweeps;
    const long long lo = std::max<long long>(h->sweep, first);
    const unsigned long long due = hi <= lo ? 0ull : (unsigned long long)((hi - first + thin - 1) / thin - (lo - first + thin - 1) / thin);
    REQUIRE(h->sum_samples + due * nC(h) <= 0xffffffffull, MP_ERR_STATE,
            "mp_sweep: the summaries would pass 2^32 - 1 samples (read them with reset, or set them again)");
    return MP_OK;
}
template <typename R> static int launch_summaries(mp_engine *h)
{
    const SumLayout L = sum_layout(h);
    SumBufs b;
    b.z_prob = (double *)(h->d_sum + L.z_prob); b.S_sum = (double *)(h->d_sum + L.S_sum);
    b.z_count = (uint32_t *)(h->d_sum + L.z_count); b.y_count = (uint32_t *)(h->d_sum + L.y_count);
    b.nsamples = (unsigned long long *)(h->d_sum + L.nsamples);
    const long long threads = (long long)nT(h) * (long long)((nN(h) + 3) / 4);
    k_summaries<R><<<(unsigned)((threads + 255) / 256), 256, 0, h->stream>>>(sampler_dev(h), h->d_ctr, h->sum_first, h->sum_thin,
        view<R>(h), h->d_par, h->d_obs, h->have_era ? h->d_era : nullptr, h->d_z, h->d_y, h->d_S[0], h->cfg.n_years, h->cfg.n_chains, b);
    CK(cudaGetLastError());
    if (summary_due(h, h->sweep)) h->sum_samples += nC(h);
    return MP_OK;
}
// ---- pointwise predictive densities for WAIC (mp_set_waic): lik, loglik, loglik_sq [T][N] doubles, then the uint64 sample
// counter: T N 24 + 8 bytes
static size_t waic_bytes(const mp_engine *h) { return zcells(h) * 24 + 8; }
template <typename R> static int launch_waic(mp_engine *h)
{
    WaicBufs b;
    b.lik = (double *)h->d_waic; b.loglik = b.lik + zcells(h); b.loglik_sq = b.loglik + zcells(h);
    b.nsamples = (unsigned long long *)(b.loglik_sq + zcells(h));
    const long long threads = (long long)nT(h) * (long long)((nN(h) + 3) / 4);
    k_waic<R><<<(unsigned)((threads + 255) / 256), 256, 0, h->stream>>>(sampler_dev(h), h->d_ctr, h->waic_first, h->waic_thin,
        view<R>(h), h->d_par, h->d_obs, h->have_era ? h->d_era : nullptr, h->d_z, h->d_S[0], h->cfg.n_years, h->cfg.n_chains, b);
    CK(cudaGetLastError());
    return MP_OK;
}
// ---- colonisation sources (mp_set_sources): the per-sample lists, staging array, per-(chain, transition) externals and counts
// and integer histogram, then the sums (src_sum, ext_sum, events, dist_hist, sample counter)
struct SrcLayout { size_t evt, src, stage, ct_ext, ct_cnt, hist_i, sums, src_sum, ext_sum, events, dist_hist, nsamples, bytes; };
static SrcLayout src_layout(const mp_engine *h, int nbins)
{
    SrcLayout L;
    size_t off = 0;
    auto carve = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t rows = nC(h) * (nT(h) - 1), cells = rows * nN(h), nb = (size_t)nbins;
    L.evt = carve(cells * (is64(h) ? sizeof(EvtRec<double>) : sizeof(EvtRec<float>)));
    L.src = carve(cells * (is64(h) ? sizeof(SrcRec<double>) : sizeof(SrcRec<float>)));
    L.stage = carve(cells * 8); L.ct_ext = carve(rows * 8); L.ct_cnt = carve(rows * 16); L.hist_i = carve((nT(h) - 1) * nb * 8);
    L.sums = off;
    L.src_sum = carve(ycells(h) * 8); L.ext_sum = carve((nT(h) - 1) * 8); L.events = carve(2 * (nT(h) - 1) * 8);
    L.dist_hist = carve((nT(h) - 1) * nb * 8); L.nsamples = carve(8); L.bytes = off;
    return L;
}
template <typename R, int GEOM> static void launch_src_contract(mp_engine *h, const SrcBufs &b)
{
    const int T = h->cfg.n_years;
    const dim3 grid((h->cfg.n_patches + SRC_TILE - 1) / SRC_TILE, T - 1, h->cfg.n_chains);
    if (b.nbins > 0)
        k_src_contract<R, GEOM, true><<<grid, SRC_TILE, (size_t)b.nbins * 8, h->stream>>>(h->d_ctr, h->src_first, h->src_thin, view<R>(h),
                                                                                          h->d_par, T, b);
    else
        k_src_contract<R, GEOM, false><<<grid, SRC_TILE, 0, h->stream>>>(h->d_ctr, h->src_first, h->src_thin, view<R>(h), h->d_par, T, b);
}
// three launches, each gated on the device by the sweep counter
template <typename R> static int launch_sources(mp_engine *h)
{
    const SrcLayout L = src_layout(h, h->src_nbins);
    unsigned char *base = h->d_src;
    SrcBufs b;
    b.evt = base + L.evt; b.src = base + L.src; b.stage = (double *)(base + L.stage); b.ct_ext = (double *)(base + L.ct_ext);
    b.ct_cnt = (uint32_t *)(base + L.ct_cnt); b.hist_i = (unsigned long long *)(base + L.hist_i);
    b.src_sum = (double *)(base + L.src_sum); b.ext_sum = (double *)(base + L.ext_sum); b.events = (unsigned long long *)(base + L.events);
    b.dist_hist = (double *)(base + L.dist_hist); b.nsamples = (unsigned long long *)(base + L.nsamples);
    b.nbins = h->src_nbins; b.bin_width = h->src_bin_width;
    const int T = h->cfg.n_years, n = h->cfg.n_patches;
    k_src_lists<R><<<dim3(T - 1, h->cfg.n_chains), SRC_LIST_THREADS, 0, h->stream>>>(h->d_ctr, h->src_first, h->src_thin, view<R>(h),
        h->geom == MP_GEOM_COORDS ? 1 : 0, h->d_perm, h->d_par, h->have_era ? h->d_era : nullptr, (const R *)h->d_aw[0], h->d_z, h->d_y,
        h->d_S[0], T, b);
    CK(cudaGetLastError());
    if (h->geom == MP_GEOM_COORDS) launch_src_contract<R, MP_GEOM_COORDS>(h, b);
    else if (h->geom == MP_GEOM_DENSE) launch_src_contract<R, MP_GEOM_DENSE>(h, b);
    else launch_src_contract<R, MP_GEOM_LINEAR>(h, b);
    CK(cudaGetLastError());
    const long long threads = (long long)(T - 1) * std::max(n, h->src_nbins);
    k_src_finish<<<(unsigned)((threads + 255) / 256), 256, 0, h->stream>>>(h->d_ctr, h->src_first, h->src_thin, n, T, h->cfg.n_chains, b);
    CK(cudaGetLastError());
    return MP_OK;
}

// phase 3: e and p from the sufficient counts, record the draw
template <typename R> static int phase_finish(mp_engine *h)
{
    int rc;
    const int C = h->cfg.n_chains;
    const SamplerDev sd = sampler_dev(h);
    if ((rc = launch_counts(h)) != MP_OK) return rc;
    { Timed tm(h, MP_K_SMALL);
      k_update_ep<<<(C + 63) / 64, 64, 0, h->stream>>>(sd, h->d_ctr, h->d_par, h->d_lsig, h->d_counts, C);
      CK(cudaGetLastError()); }
    if ((rc = launch_col<R>(h, 1, h->d_par, h->d_S[0], h->d_par, h->d_S[0])) != MP_OK) return rc;
    {
        Timed tm(h, MP_K_SMALL);
        // the row is chosen on the device from the draw counter, and the counters advance there too: the launches of a sweep carry
        // no per-sweep host value, so a captured sweep can be replayed (mp_sweep)
        k_record<<<C, 32, 0, h->stream>>>(sd, h->d_par, h->d_counts, h->d_partial[0], h->nblk_col, h->d_draws, nullptr, h->d_ctr, h->cfg.max_draws);
        CK(cudaGetLastError());
        // the sweep's final z, y, S and theta, gated on the device by the sweep counter before k_advance moves it; one more
        // launch in this span (without summaries the sweep keeps its launches and counts)
        if (h->sum_thin > 0) {
            h->t_launch[MP_K_SMALL]++;
            if ((rc = launch_summaries<R>(h)) != MP_OK) return rc;
        }
        if (h->waic_thin > 0) {                              // the same for the WAIC sums
            h->t_launch[MP_K_SMALL]++;
            if ((rc = launch_waic<R>(h)) != MP_OK) return rc;
        }
        if (h->src_thin > 0) {                               // and for the colonisation sources (three launches)
            h->t_launch[MP_K_SMALL] += 3;
            if ((rc = launch_sources<R>(h)) != MP_OK) return rc;
        }
        k_advance<<<1, 1, 0, h->stream>>>(h->d_ctr, h->cfg.max_draws);
        CK(cudaGetLastError());
    }
    if (h->ndraws < h->cfg.max_draws) h->ndraws++;          // host mirrors of the device counters
    h->sweep++;
    return MP_OK;
}
template <typename R> static int sweep_once(mp_engine *h)
{
    int rc;
    if ((rc = phase_propose_conn<R>(h, nullptr)) != MP_OK) return rc;
    if ((rc = phase_decide_z<R>(h)) != MP_OK) return rc;
    if ((rc = phase_sweep_y<R>(h)) != MP_OK) return rc;
    return phase_finish<R>(h);
}

// ------------------------------------------------------------------ C ABI
extern "C" {

const char *mp_version(void) { return "midaspom_b200 0.1 (sm_100a, abi 1)"; }

int mp_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

const char *mp_last_error(const mp_engine *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int mp_destroy(mp_engine *h)
{
    if (!h) return MP_OK;
    cudaSetDevice(h->cfg.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->comm) mp_comm_destroy(h);
    drop_graphs(h);
    drain_spans(h);
    for (auto e : h->pool) cudaEventDestroy(e);
    void *ptrs[] = { h->d_area, h->d_src_unit, h->d_px, h->d_py, h->d_dist, h->d_obs, h->d_era, h->d_par, h->d_prop,
                     h->d_lsig, h->d_z, h->d_y, h->d_srec, h->d_S[0], h->d_S[1], h->d_aw[0], h->d_aw[1], h->d_partial[0],
                     h->d_partial[1], h->d_llc, h->d_logu, h->d_parts, h->d_scalar, h->d_flags, h->d_counts, h->d_draws, h->d_cand, h->d_cand_count, h->d_task_order, h->d_ljac, h->d_perm, h->d_scan, h->d_minv, h->d_tile_box, h->d_mlow, h->d_work, h->d_gemm, h->d_tlist, h->d_btasks, h->d_blockmode, h->d_scan_work, h->d_comm_send, h->d_comm_recv, h->d_ctr, h->d_sum, h->d_waic, h->d_src };
    for (void *p : ptrs) if (p) cudaFree(p);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return MP_OK;
}

int mp_create(const mp_config *cfg, mp_engine **out)
{
    if (!cfg || !out) { g_create_error = "mp_create: null argument"; return MP_ERR_ARG; }
    *out = nullptr;
    if (cfg->n_patches < 1 || cfg->n_years < 2 || cfg->n_chains < 1 || cfg->max_draws < 0 ||
        (cfg->precision != MP_FP32 && cfg->precision != MP_FP64)) {
        g_create_error = "mp_create: need n_patches>=1, n_years>=2, n_chains>=1, precision MP_FP32|MP_FP64";
        return MP_ERR_ARG;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("mp_create: no CUDA device (") + cudaGetErrorString(e) + "); there is no CPU fallback";
        return MP_ERR_CUDA;
    }
    if (cfg->device < 0 || cfg->device >= ndev) { g_create_error = "mp_create: bad device ordinal"; return MP_ERR_ARG; }
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, cfg->device)) != cudaSuccess) { g_create_error = cudaGetErrorString(e); return MP_ERR_CUDA; }
    if (prop.major != 10) {
        g_create_error = "mp_create: device is not sm_100 (this library carries sm_100a code only)";
        return MP_ERR_CUDA;
    }
    mp_engine *h = new mp_engine();
    h->cfg = *cfg;
    if (const char *env = getenv("MP_CONN_CULL")) h->conn_cull = atoi(env) != 0;
    if (const char *env = getenv("MP_CONN_GEMM")) h->use_gemm = atoi(env) != 0;
    if (const char *env = getenv("MP_CONN_GEMM_MIN_N")) { const int v = atoi(env); if (v >= 1) h->gemm_min_n = v; }
    if (const char *env = getenv("MP_CONN_ACC32")) h->conn_acc32 = atoi(env) != 0;
    if (const char *env = getenv("MP_CONN_SHAPE")) { const int v = atoi(env); if (v >= 0 && v <= 4) h->conn_shape = v; }
    if (const char *env = getenv("MP_REFRESH_EVERY")) { const int v = atoi(env); if (v >= 1) h->refresh_every = v; }
    if (const char *env = getenv("MP_FAST_CS")) { const int v = atoi(env); if (v == 1 || v == 2 || v == 4 || v == 8 || v == 16) h->fast_cs = v; }
    if (const char *env = getenv("MP_FAST_TPT")) { const int v = atoi(env); if (v == 128 || v == 256 || v == 512 || v == 1024 || v == 2048 || v == 4096 || v == 8192) h->fast_tpt = v; }
    if (const char *env = getenv("MP_GRAPH")) h->use_graph = atoi(env) != 0;
    if (const char *env = getenv("MP_BLK_TPT")) { const int v = atoi(env); if (v == 512 || v == 1024 || v == 2048 || v == 4096 || v == 8192) h->blk_tpt = v; }
    if (const char *env = getenv("MP_BLK_CS")) { const int v = atoi(env); if (v == 1 || v == 2 || v == 4 || v == 8) h->blk_cs = v; }
    h->sm_count = prop.multiProcessorCount;
    auto fail = [&](const char *what, cudaError_t ce) {
        g_create_error = std::string("mp_create: ") + what + ": " + cudaGetErrorString(ce);
        mp_destroy(h);
        return MP_ERR_CUDA;
    };
    if ((e = cudaSetDevice(cfg->device)) != cudaSuccess) return fail("cudaSetDevice", e);
    if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) return fail("stream", e);
    const size_t N = nN(h), T = nT(h), C = nC(h), R = rsz(h);
    h->nwords = (int)((T - 1 + 31) / 32);
    const long long cells = (long long)ycells(h);
    h->nblk_col = (int)std::max<long long>(1, std::min<long long>(MAX_COL_BLOCKS, (cells + COL_THREADS * 8 - 1) / (COL_THREADS * 8)));
    struct Req { void **p; size_t bytes; };
    Req reqs[] = {
        { (void **)&h->d_area, N * 8 }, { (void **)&h->d_src_unit, N * 8 }, { &h->d_px, N * R }, { &h->d_py, N * R },
        { (void **)&h->d_obs, T * N }, { (void **)&h->d_era, T }, { (void **)&h->d_par, C * sizeof(mp_params) },
        { (void **)&h->d_prop, C * sizeof(mp_params) }, { (void **)&h->d_lsig, C * MP_NLSIG * 8 },
        { (void **)&h->d_z, C * T * N }, { (void **)&h->d_y, C * (T - 1) * N },
        { &h->d_srec, 2 * C * h->nwords * (size_t)conn_npad((int)N) * (cfg->precision == MP_FP64 ? sizeof(SrcRec<double>) : sizeof(SrcRec<float>)) }, { (void **)&h->d_S[0], C * (T - 1) * N * 8 },
        { (void **)&h->d_S[1], C * (T - 1) * N * 8 }, { &h->d_aw[0], C * N * R }, { &h->d_aw[1], C * N * R },
        { (void **)&h->d_partial[0], C * MAX_COL_BLOCKS * 8 }, { (void **)&h->d_partial[1], C * MAX_COL_BLOCKS * 8 },
        { (void **)&h->d_llc, C * 8 }, { (void **)&h->d_logu, C * 8 }, { (void **)&h->d_ljac, C * 8 }, { (void **)&h->d_parts, C * MP_NPART * 8 },
        { (void **)&h->d_scalar, 64 }, { (void **)&h->d_flags, C * 4 * sizeof(int) },
        { (void **)&h->d_counts, C * NCOUNT * sizeof(unsigned long long) },
        { (void **)&h->d_draws, std::max<size_t>(1, (size_t)cfg->max_draws) * C * MP_NDRAW * 8 },
        { &h->d_cand, cfg->precision == MP_FP32 ? C * (T - 1) * N * sizeof(CandRec) : 32 },
        { (void **)&h->d_cand_count, C * (T - 1) * 2 * sizeof(int) }, { (void **)&h->d_task_order, C * (T - 1) * sizeof(int) },
        { (void **)&h->d_ctr, 2 * sizeof(uint32_t) }, { (void **)&h->d_perm, N * sizeof(int) }, { (void **)&h->d_scan, N * sizeof(int) }, { (void **)&h->d_minv, N * sizeof(int) }, { (void **)&h->d_work, MP_CNT_N * sizeof(unsigned long long) },
        { (void **)&h->d_tile_box, ((N + 31) / 32) * sizeof(float4) }, { (void **)&h->d_mlow, C * ((N + 31) / 32) * sizeof(float) },
    };
    for (auto &r : reqs) {
        if ((e = cudaMalloc(r.p, r.bytes)) != cudaSuccess) return fail("cudaMalloc", e);
        if ((e = cudaMemset(*r.p, 0, r.bytes)) != cudaSuccess) return fail("cudaMemset", e);
    }
    {   // external-source distance units default to u_k = k + 1 (loss.c:365) until mp_set_source_units replaces them
        std::vector<double> u(N);
        for (size_t k = 0; k < N; k++) u[k] = (double)(k + 1);
        if ((e = cudaMemcpy(h->d_src_unit, u.data(), N * 8, cudaMemcpyHostToDevice)) != cudaSuccess) return fail("memcpy", e);
    }
    // defaults: parameters of the reference's defaults (main_MIDASPOM.c:66-73), neutral variant terms
    std::vector<mp_params> par(C, mp_params{ 0.5, 0.5, 1.0 / 400.0, 0.0, 1.0, 1.0, 0.0, 0.0 });
    if ((e = cudaMemcpy(h->d_par, par.data(), C * sizeof(mp_params), cudaMemcpyHostToDevice)) != cudaSuccess) return fail("memcpy", e);
    if ((e = cudaMemcpy(h->d_prop, par.data(), C * sizeof(mp_params), cudaMemcpyHostToDevice)) != cudaSuccess) return fail("memcpy", e);
    *out = h;
    return MP_OK;
}

// ---- landscape
// Uploads below use the blocking default stream; the engine stream is non-blocking, so wait for its
// pending work first (a setter called after an asynchronous mp_sweep must not race with it).
static int quiesce(mp_engine *h) { CK(cudaStreamSynchronize(h->stream)); drop_graphs(h); return MP_OK; }
static int upload_real(mp_engine *h, void *dst, const double *src, size_t n)
{
    if (is64(h)) { CK(cudaMemcpy(dst, src, n * 8, cudaMemcpyHostToDevice)); return MP_OK; }
    std::vector<float> tmp(n);
    for (size_t i = 0; i < n; i++) tmp[i] = (float)src[i];
    CK(cudaMemcpy(dst, tmp.data(), n * 4, cudaMemcpyHostToDevice));
    return MP_OK;
}
static int set_area(mp_engine *h, const double *area)
{
    h->have_area = area != nullptr;
    h->area_max = h->area_min = 1.0;
    if (area) {
        for (size_t i = 0; i < nN(h); i++) REQUIRE(area[i] > 0.0, MP_ERR_ARG, "patch areas must be positive");
        h->area_max = *std::max_element(area, area + nN(h)); h->area_min = *std::min_element(area, area + nN(h));
        CK(cudaMemcpy(h->d_area, area, nN(h) * 8, cudaMemcpyHostToDevice));
    }
    return MP_OK;
}
// cell of a coordinate in a grid of ncell cells over [lo, hi] -- the same arithmetic as the oracle's scan_cell
static inline int scan_cell(double v, double lo, double hi, int ncell)
{
    const double w = (hi - lo) / ncell;
    if (!(w > 0.0)) return 0;
    int c = (int)((v - lo) / w);
    if (c < 0) c = 0;
    if (c > ncell - 1) c = ncell - 1;
    return c;
}
// Two orders of the patches.  LAYOUT order perm[slot] = patch: the Morton (Z-curve) order of planar coordinates, index order
// otherwise -- spatially adjacent patches get adjacent slots, which is what makes the warp-level culling of k_sweep_y_cull
// and k_conn effective.  VISITING order of the y scan scan[pos] = patch: the same without a scan grid; with one
// (mp_set_scan_blocks) colour by colour, block by block, Morton order inside a block (oracle: spom_scan_order).
static int set_patch_order(mp_engine *h, const double *x, const double *y, double spacing = 0.0, double cx = 0.0, double cy = 0.0)
{   // (cx, cy): origin of the coordinates as stored on the device (FP32 engines centre them)
    const size_t N = nN(h);
    std::vector<int> perm(N), scan(N), minv(N);
    for (size_t i = 0; i < N; i++) perm[i] = scan[i] = (int)i;
    h->morton.assign(N, 0u); h->blk_of.assign(N, 0);
    if (x && y) {
        if (x != h->hx.data()) { h->hx.assign(x, x + N); h->hy.assign(y, y + N); }
        h->cx = cx; h->cy = cy;
        double x0 = x[0], x1 = x[0], y0 = y[0], y1 = y[0];
        for (size_t i = 1; i < N; i++) { x0 = std::min(x0, x[i]); x1 = std::max(x1, x[i]); y0 = std::min(y0, y[i]); y1 = std::max(y1, y[i]); }
        h->bb[0] = x0; h->bb[1] = x1; h->bb[2] = y0; h->bb[3] = y1;
        const double span = std::max(std::max(x1 - x0, y1 - y0), 1e-300);
        auto spread = [](uint32_t v) { v &= 0xffffu; v = (v | (v << 8)) & 0x00ff00ffu; v = (v | (v << 4)) & 0x0f0f0f0fu;
                                       v = (v | (v << 2)) & 0x33333333u; v = (v | (v << 1)) & 0x55555555u; return v; };
        const int nbx = std::max(h->blk_nx, 1), nby = std::max(h->blk_ny, 1), bk = std::max(h->blk_k, 1);
        std::vector<uint64_t> key(N);
        for (size_t i = 0; i < N; i++) {
            const uint32_t xi = (uint32_t)std::min(65535.0, (x[i] - x0) / span * 65535.0), yi = (uint32_t)std::min(65535.0, (y[i] - y0) / span * 65535.0);
            h->morton[i] = spread(xi) | (spread(yi) << 1);
            const int bx = scan_cell(x[i], x0, x1, nbx), by = scan_cell(y[i], y0, y1, nby);
            h->blk_of[i] = by * nbx + bx;
            const uint32_t group = (uint32_t)(((bx % bk) + bk * (by % bk)) * (nbx * nby) + by * nbx + bx);   // (colour, block)
            key[i] = ((uint64_t)group << 32) | h->morton[i];
        }
        std::stable_sort(perm.begin(), perm.end(), [&](int a, int b) { return h->morton[a] < h->morton[b]; });
        std::stable_sort(scan.begin(), scan.end(), [&](int a, int b) { return key[a] < key[b]; });
    } else { h->hx.clear(); h->hy.clear(); }
    for (size_t s = 0; s < N; s++) minv[perm[s]] = (int)s;
    h->scan_host = scan;
    CK(cudaMemcpy(h->d_perm, perm.data(), N * sizeof(int), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->d_scan, scan.data(), N * sizeof(int), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->d_minv, minv.data(), N * sizeof(int), cudaMemcpyHostToDevice));
    // bounding boxes of the groups of 32 consecutive layout slots (culled k_conn), in the FP32 coordinates the kernels use
    const size_t ntile = (N + 31) / 32;
    std::vector<float4> box(ntile);
    h->have_boxes = (x && y) || spacing > 0.0;
    for (size_t tI = 0; tI < ntile && h->have_boxes; tI++) {
        float bx0 = 3.0e38f, bx1 = -3.0e38f, by0 = 3.0e38f, by1 = -3.0e38f;
        for (size_t sI = tI * 32; sI < std::min(N, (tI + 1) * 32); sI++) {
            const int q = perm[sI];
            const float fx = x ? (float)(x[q] - cx) : (float)q * (float)spacing, fy = y ? (float)(y[q] - cy) : 0.f;
            bx0 = std::min(bx0, fx); bx1 = std::max(bx1, fx); by0 = std::min(by0, fy); by1 = std::max(by1, fy);
        }
        box[tI] = make_float4(bx0, bx1, by0, by1);
    }
    CK(cudaMemcpy(h->d_tile_box, box.data(), ntile * sizeof(float4), cudaMemcpyHostToDevice));
    return MP_OK;
}
// Block lists of the scan grid: per block its run of scan-order slots and its target list -- own patches in scan order,
// then every other patch within the halo of the block's cell, in Morton order (32 consecutive list entries stay compact).
static int build_scan_blocks(mp_engine *h)
{
    const size_t N = nN(h);
    const int nbx = h->blk_nx, nby = h->blk_ny, nb = nbx * nby;
    h->blk_slot_lo.assign(nb, 0); h->blk_slot_hi.assign(nb, 0); h->blk_tl_off.assign(nb, 0); h->blk_tl_n.assign(nb, 0);
    std::vector<int> seen(nb, 0);
    for (size_t s = 0; s < N; s++) {                      // own positions: contiguous runs of the (colour, block, Morton) visiting order
        const int b = h->blk_of[h->scan_host[s]];
        if (!seen[b]) { seen[b] = 1; h->blk_slot_lo[b] = (int)s; }
        h->blk_slot_hi[b] = (int)s + 1;
    }
    const double x0 = h->bb[0], x1 = h->bb[1], y0 = h->bb[2], y1 = h->bb[3];
    const double wx = (x1 - x0) / nbx, wy = (y1 - y0) / nby, halo2 = h->blk_halo * h->blk_halo;
    std::vector<int> by_morton(N);
    for (size_t i = 0; i < N; i++) by_morton[i] = (int)i;
    std::stable_sort(by_morton.begin(), by_morton.end(), [&](int a, int b) { return h->morton[a] < h->morton[b]; });
    std::vector<int> tlist;
    h->blk_nl_max = 0;
    for (int b = 0; b < nb; b++) {
        h->blk_tl_off[b] = (int)tlist.size();
        if (!seen[b]) continue;
        for (int s = h->blk_slot_lo[b]; s < h->blk_slot_hi[b]; s++) tlist.push_back(h->scan_host[s]);
        const int bx = b % nbx, by = b / nbx;
        const double rx0 = x0 + bx * wx, rx1 = x0 + (bx + 1) * wx, ry0 = y0 + by * wy, ry1 = y0 + (by + 1) * wy;
        for (size_t i = 0; i < N; i++) {
            const int q = by_morton[i];
            if (h->blk_of[q] == b) continue;
            const double dx = std::max(std::max(rx0 - h->hx[q], h->hx[q] - rx1), 0.0), dy = std::max(std::max(ry0 - h->hy[q], h->hy[q] - ry1), 0.0);
            if (dx * dx + dy * dy <= halo2) tlist.push_back(q);
        }
        h->blk_tl_n[b] = (int)tlist.size() - h->blk_tl_off[b];
        h->blk_nl_max = std::max(h->blk_nl_max, h->blk_tl_n[b]);
        while (tlist.size() % 4) tlist.push_back(0);      // 16-byte aligned lists
    }
    if (h->d_tlist) { CK(cudaFree(h->d_tlist)); h->d_tlist = nullptr; }
    CK(cudaMalloc(&h->d_tlist, std::max<size_t>(tlist.size(), 4) * sizeof(int)));
    CK(cudaMemcpy(h->d_tlist, tlist.data(), tlist.size() * sizeof(int), cudaMemcpyHostToDevice));
    h->blk_tasks_dirty = true;
    return MP_OK;
}
// Block tasks of the (chain, year) tasks this engine scans, grouped by colour (one launch per colour)
static int build_block_tasks(mp_engine *h)
{
    const int nbx = h->blk_nx, nby = h->blk_ny, bk = h->blk_k, nb = nbx * nby, ncol = bk * bk;
    const int ntask_all = h->cfg.n_chains * (h->cfg.n_years - 1);
    std::vector<mp::BlockTask> bt;
    h->colour_off.assign(ncol, 0); h->colour_n.assign(ncol, 0);
    for (int col = 0; col < ncol; col++) {
        h->colour_off[col] = (int)bt.size();
        for (int b = 0; b < nb; b++) {
            const int bx = b % nbx, by = b / nbx;
            if ((bx % bk) + bk * (by % bk) != col || h->blk_slot_hi[b] <= h->blk_slot_lo[b]) continue;
            for (int task = h->task_first; task < ntask_all; task += h->task_stride)
                bt.push_back(mp::BlockTask{ task, h->blk_tl_off[b], h->blk_tl_n[b], h->blk_slot_lo[b], h->blk_slot_hi[b] });
        }
        h->colour_n[col] = (int)bt.size() - h->colour_off[col];
    }
    if (h->d_btasks) { CK(cudaFree(h->d_btasks)); h->d_btasks = nullptr; }
    CK(cudaMalloc(&h->d_btasks, std::max<size_t>(bt.size(), 1) * sizeof(mp::BlockTask)));
    CK(cudaMemcpy(h->d_btasks, bt.data(), bt.size() * sizeof(mp::BlockTask), cudaMemcpyHostToDevice));
    if (!h->d_blockmode) { CK(cudaMalloc(&h->d_blockmode, (size_t)ntask_all * sizeof(int))); CK(cudaMemset(h->d_blockmode, 0, (size_t)ntask_all * sizeof(int))); }
    h->blk_tasks_dirty = false;
    return MP_OK;
}
int mp_get_scan_order(mp_engine *h, int32_t *order)
{
    if (!h || !order) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    REQUIRE(h->have_landscape, MP_ERR_STATE, "set the landscape first");
    if (quiesce(h) != MP_OK) return MP_ERR_CUDA;
    CK(cudaMemcpy(order, h->d_scan, nN(h) * sizeof(int), cudaMemcpyDeviceToHost));
    return MP_OK;
}
int mp_set_scan_blocks(mp_engine *h, int nx, int ny, int k, double halo)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    REQUIRE(h->have_landscape && h->geom == MP_GEOM_COORDS, MP_ERR_STATE, "mp_set_scan_blocks: set a landscape with coordinates first");
    if (quiesce(h) != MP_OK) return MP_ERR_CUDA;
    const bool on = nx >= 1 && ny >= 1 && nx * ny > 1;
    if (on) {
        REQUIRE(k >= 2 && halo >= 0.0 && nx <= 1024 && ny <= 1024, MP_ERR_ARG, "mp_set_scan_blocks: need k >= 2, halo >= 0, at most 1024 cells per axis");
        // same-colour cells are k cells apart along an axis with more than k cells: the gap (k - 1) cells must exceed 2 halo
        const double wx = (h->bb[1] - h->bb[0]) / nx, wy = (h->bb[3] - h->bb[2]) / ny;
        REQUIRE((nx <= k || (k - 1) * wx > 2.0 * halo) && (ny <= k || (k - 1) * wy > 2.0 * halo), MP_ERR_ARG,
                "mp_set_scan_blocks: cells of one colour must lie farther apart than twice the halo ((k - 1) x cell width > 2 halo)");
    }
    h->blk_nx = on ? nx : 1; h->blk_ny = on ? ny : 1; h->blk_k = on ? k : 1; h->blk_halo = on ? halo : 0.0; h->blk_active = on;
    std::vector<double> x = h->hx, y = h->hy;             // set_patch_order re-reads the caller's coordinates
    int rc = set_patch_order(h, x.data(), y.data(), 0.0, h->cx, h->cy);
    if (rc != MP_OK) return rc;
    return on ? build_scan_blocks(h) : MP_OK;
}
int mp_set_landscape_linear(mp_engine *h, double spacing, const double *area)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    if (quiesce(h) != MP_OK) return MP_ERR_CUDA;
    REQUIRE(spacing > 0.0, MP_ERR_ARG, "spacing must be positive");
    h->geom = MP_GEOM_LINEAR; h->spacing = spacing;
    h->blk_nx = h->blk_ny = h->blk_k = 1; h->blk_halo = 0.0; h->blk_active = false;   // a new landscape starts without a scan grid
    int rc = set_patch_order(h, nullptr, nullptr, spacing);      // a line is already in spatial order
    if (rc != MP_OK) return rc;
    rc = set_area(h, area);
    if (rc == MP_OK) { h->have_landscape = true; h->S_valid = false; }
    return rc;
}
int mp_set_landscape_coords(mp_engine *h, const double *x, const double *y, const double *area)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    if (quiesce(h) != MP_OK) return MP_ERR_CUDA;
    REQUIRE(x && y, MP_ERR_ARG, "null coordinates");
    h->geom = MP_GEOM_COORDS;
    h->blk_nx = h->blk_ny = h->blk_k = 1; h->blk_halo = 0.0; h->blk_active = false;   // a new landscape starts without a scan grid
    int rc;
    // FP32 engines store positions relative to the centre of the bounding box: only differences enter the model, and
    // halving the largest magnitude halves the quantisation of a coordinate (2^-24 of it).  FP64 keeps the caller's values.
    double cx = 0.0, cy = 0.0;
    std::vector<double> xs, ys;
    const double *ux = x, *uy = y;
    if (!is64(h)) {
        const auto mmx = std::minmax_element(x, x + nN(h)), mmy = std::minmax_element(y, y + nN(h));
        cx = 0.5 * (*mmx.first + *mmx.second); cy = 0.5 * (*mmy.first + *mmy.second);
        xs.resize(nN(h)); ys.resize(nN(h));
        for (size_t i = 0; i < nN(h); i++) { xs[i] = x[i] - cx; ys[i] = y[i] - cy; }
        ux = xs.data(); uy = ys.data();
    }
    if ((rc = upload_real(h, h->d_px, ux, nN(h))) != MP_OK) return rc;
    if ((rc = upload_real(h, h->d_py, uy, nN(h))) != MP_OK) return rc;
    if ((rc = set_patch_order(h, x, y, 0.0, cx, cy)) != MP_OK) return rc;      // the order comes from the caller's values, like the oracle's
    rc = set_area(h, area);
    if (rc == MP_OK) { h->have_landscape = true; h->S_valid = false; }
    return rc;
}
int mp_set_landscape_dense(mp_engine *h, const double *dist, const double *area)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    if (quiesce(h) != MP_OK) return MP_ERR_CUDA;
    REQUIRE(dist, MP_ERR_ARG, "null distance matrix");
    const size_t nn = nN(h) * nN(h);
    if (!h->d_dist) CK(cudaMalloc(&h->d_dist, nn * rsz(h)));
    h->geom = MP_GEOM_DENSE;
    h->blk_nx = h->blk_ny = h->blk_k = 1; h->blk_halo = 0.0; h->blk_active = false;   // a new landscape starts without a scan grid
    int rc;
    if ((rc = upload_real(h, h->d_dist, dist, nn)) != MP_OK) return rc;
    if ((rc = set_patch_order(h, nullptr, nullptr)) != MP_OK) return rc;
    rc = set_area(h, area);
    if (rc == MP_OK) { h->have_landscape = true; h->S_valid = false; }
    return rc;
}
int mp_set_source_units(mp_engine *h, const double *src_unit)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    if (quiesce(h) != MP_OK) return MP_ERR_CUDA;
    std::vector<double> u(nN(h));
    for (size_t k = 0; k < nN(h); k++) u[k] = src_unit ? src_unit[k] : (double)(k + 1);   // loss.c:365
    CK(cudaMemcpy(h->d_src_unit, u.data(), nN(h) * 8, cudaMemcpyHostToDevice));
    return MP_OK;
}

// ---- data
int mp_set_observations(mp_engine *h, const int8_t *obs)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    REQUIRE(obs, MP_ERR_ARG, "null observations");
    for (size_t i = 0; i < zcells(h); i++) REQUIRE(obs[i] >= -1 && obs[i] <= 1, MP_ERR_ARG, "observations must be -1, 0 or 1");
    CK(cudaMemcpyAsync(h->d_obs, obs, zcells(h), cudaMemcpyHostToDevice, h->stream));
    if (h->d_waic) CK(cudaMemsetAsync(h->d_waic, 0, waic_bytes(h), h->stream));   // sums over other observations mean nothing now
    CK(cudaStreamSynchronize(h->stream));
    h->have_obs = true;
    return MP_OK;
}
int mp_set_era(mp_engine *h, const uint8_t *era)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    if (quiesce(h) != MP_OK) return MP_ERR_CUDA;
    h->have_era = era != nullptr;
    if (era) CK(cudaMemcpy(h->d_era, era, nT(h) - 1, cudaMemcpyHostToDevice));
    return MP_OK;
}

// ---- chain state
int mp_set_params(mp_engine *h, const mp_params *par)
{
    if (!h || !par) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    for (size_t c = 0; c < nC(h); c++) REQUIRE(par[c].K > 0.0 && par[c].alpha > 0.0, MP_ERR_ARG, "need K > 0 and alpha > 0");
    h->any_src = false; h->S_valid = false;
    for (size_t c = 0; c < nC(h); c++) if (par[c].Ksrc != 0.0) h->any_src = true;
    h->par_host.assign(par, par + nC(h)); h->par_host_valid = true; h->have_params = true;
    CK(cudaMemcpyAsync(h->d_par, par, nC(h) * sizeof(mp_params), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MP_OK;
}
int mp_get_params(mp_engine *h, mp_params *par)
{
    if (!h || !par) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemcpyAsync(par, h->d_par, nC(h) * sizeof(mp_params), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MP_OK;
}
int mp_set_state(mp_engine *h, const uint8_t *z, const uint8_t *y)
{
    if (!h || !z || !y) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemcpyAsync(h->d_z, z, nC(h) * zcells(h), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_y, y, nC(h) * ycells(h), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->have_state = true; h->S_valid = false;
    return MP_OK;
}
int mp_get_state(mp_engine *h, uint8_t *z, uint8_t *y)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    if (z) CK(cudaMemcpyAsync(z, h->d_z, nC(h) * zcells(h), cudaMemcpyDeviceToHost, h->stream));
    if (y) CK(cudaMemcpyAsync(y, h->d_y, nC(h) * ycells(h), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MP_OK;
}
int mp_set_scales(mp_engine *h, const double *lsig)
{
    if (!h || !lsig) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    if (quiesce(h) != MP_OK) return MP_ERR_CUDA;
    CK(cudaMemcpy(h->d_lsig, lsig, nC(h) * MP_NLSIG * 8, cudaMemcpyHostToDevice));
    return MP_OK;
}
int mp_get_scales(mp_engine *h, double *lsig)
{
    if (!h || !lsig) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(lsig, h->d_lsig, nC(h) * MP_NLSIG * 8, cudaMemcpyDeviceToHost));
    return MP_OK;
}

// ---- likelihood
static int check_ready(mp_engine *h)
{
    REQUIRE(h->have_landscape, MP_ERR_STATE, "landscape not set");
    REQUIRE(h->have_state, MP_ERR_STATE, "chain state not set (mp_set_state or mp_init_chains)");
    return MP_OK;
}
int mp_get_connectivity(mp_engine *h, double *S_out)
{
    if (!h || !S_out) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemcpyAsync(S_out, h->d_S[0], nC(h) * ycells(h) * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MP_OK;
}
int mp_connectivity(mp_engine *h, double *S_out)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    int rc = check_ready(h);
    if (rc != MP_OK) return rc;
    rc = is64(h) ? refresh_S<double>(h) : refresh_S<float>(h);
    if (rc != MP_OK) return rc;
    if (S_out) return mp_get_connectivity(h, S_out);
    return MP_OK;
}
int mp_loglik(mp_engine *h, double *ll, double *parts)
{
    if (!h || !ll) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    int rc = check_ready(h);
    if (rc != MP_OK) return rc;
    REQUIRE(h->have_obs, MP_ERR_STATE, "observations not set");
    rc = is64(h) ? refresh_S<double>(h) : refresh_S<float>(h);
    if (rc != MP_OK) return rc;
    rc = is64(h) ? loglik_resident<double>(h, nullptr, h->d_parts) : loglik_resident<float>(h, nullptr, h->d_parts);
    if (rc != MP_OK) return rc;
    std::vector<double> p(nC(h) * MP_NPART);
    CK(cudaMemcpyAsync(p.data(), h->d_parts, p.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (size_t c = 0; c < nC(h); c++) ll[c] = p[c * 4 + 0] + p[c * 4 + 1] + p[c * 4 + 2] + p[c * 4 + 3];
    if (parts) memcpy(parts, p.data(), p.size() * 8);
    return MP_OK;
}
int mp_loglik_host(mp_engine *h, const mp_params *par, const uint8_t *z, const uint8_t *y, double *ll, double *parts)
{
    int rc;
    if ((rc = mp_set_params(h, par)) != MP_OK) return rc;
    if ((rc = mp_set_state(h, z, y)) != MP_OK) return rc;
    return mp_loglik(h, ll, parts);
}
extern "C++" template <typename R> int flip_delta_t(mp_engine *h, int c, int t, int k)
{
    Timed tm(h, MP_K_SMALL);
    const uint8_t *era = h->have_era ? h->d_era : nullptr;
#define FD(G) k_flip_delta<R, G><<<1, 256, 0, h->stream>>>(view<R>(h), h->d_par, (const R *)h->d_aw[0], era, h->d_z, h->d_y, \
                                                            h->d_S[0], h->cfg.n_years, c, t, k, h->d_scalar)
    switch (h->geom) {
    case MP_GEOM_LINEAR: FD(MP_GEOM_LINEAR); break;
    case MP_GEOM_COORDS: FD(MP_GEOM_COORDS); break;
    default: FD(MP_GEOM_DENSE); break;
    }
#undef FD
    CK(cudaGetLastError());
    return MP_OK;
}
int mp_flip_delta(mp_engine *h, int chain, int t, int k, double *dll)
{
    if (!h || !dll) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    int rc = check_ready(h);
    if (rc != MP_OK) return rc;
    REQUIRE(chain >= 0 && chain < h->cfg.n_chains && t >= 0 && t < h->cfg.n_years - 1 && k >= 0 && k < h->cfg.n_patches,
            MP_ERR_ARG, "mp_flip_delta: index out of range");
    rc = is64(h) ? launch_area_weights<double>(h, 0) : launch_area_weights<float>(h, 0);
    if (rc != MP_OK) return rc;
    rc = is64(h) ? flip_delta_t<double>(h, chain, t, k) : flip_delta_t<float>(h, chain, t, k);
    if (rc != MP_OK) return rc;
    CK(cudaMemcpyAsync(dll, h->d_scalar, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MP_OK;
}

// ---- sampler
int mp_set_sampler(mp_engine *h, const mp_sampler_config *sc)
{
    if (!h || !sc) return MP_ERR_ARG;
    REQUIRE(sc->n_e_steps >= 0 && sc->n_c_steps >= 0 && sc->n_v_steps >= 0, MP_ERR_ARG, "negative sub-step count");
    REQUIRE(!sc->sample_K || (sc->K_min > 0 && sc->K_max >= sc->K_min), MP_ERR_ARG, "sample_K needs 0 < K_min <= K_max");
    REQUIRE(!sc->sample_Ksrc || (sc->Ksrc_min > 0 && sc->Ksrc_max >= sc->Ksrc_min), MP_ERR_ARG, "sample_Ksrc needs 0 < Ksrc_min <= Ksrc_max");
    h->sc = *sc; h->have_sc = true;
    drop_graphs(h);
    return MP_OK;
}
int mp_init_chains(mp_engine *h, const mp_sampler_config *sc, int disperse)
{
    if (!h || !sc) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    REQUIRE(h->have_landscape && h->have_obs, MP_ERR_STATE, "set the landscape and the observations first");
    int rc = mp_set_sampler(h, sc);
    if (rc != MP_OK) return rc;
    const size_t N = nN(h), T = nT(h), C = nC(h);
    std::vector<int8_t> obs(T * N);
    CK(cudaMemcpy(obs.data(), h->d_obs, T * N, cudaMemcpyDeviceToHost));
    std::vector<mp_params> par(C);
    CK(cudaMemcpy(par.data(), h->d_par, C * sizeof(mp_params), cudaMemcpyDeviceToHost));
    std::vector<double> lsig(C * MP_NLSIG);
    std::vector<uint8_t> z(C * T * N), y(C * (T - 1) * N);
    for (size_t c = 0; c < C; c++) {
        const uint32_t gc = (uint32_t)(h->cfg.chain_offset + (int)c);
        mp_params &p = par[c];
        if (disperse) {
            uint4 r = rng(h->cfg.seed, gc, 0, RK_INIT_PARAM, 0, 0);
            if (sc->sample_e) p.e = sc->e_min + u01(r.x) * (sc->e_max - sc->e_min);
            if (sc->sample_c) p.c = sc->c_min + u01(r.y) * (sc->c_max - sc->c_min);
            if (sc->sample_alpha) p.alpha = sc->alpha_min * pow(sc->alpha_max / sc->alpha_min, u01(r.z));
            if (sc->sample_b) p.b = sc->b_min + u01(r.w) * (sc->b_max - sc->b_min);
            r = rng(h->cfg.seed, gc, 0, RK_INIT_PARAM, 1, 0);
            if (sc->sample_p) p.p = sc->p_min + u01(r.x) * (sc->p_max - sc->p_min);
            if (sc->sample_K) p.K = sc->K_min * pow(sc->K_max / sc->K_min, u01(r.y));
            if (sc->sample_Ksrc) p.Ksrc = sc->Ksrc_min * pow(sc->Ksrc_max / sc->Ksrc_min, u01(r.z));
            if (sc->sample_dsrc) p.dsrc = sc->dsrc_min + u01(r.w) * (sc->dsrc_max - sc->dsrc_min);
        }
        double *ls = &lsig[c * MP_NLSIG];
        ls[0] = log(0.05); ls[1] = log(0.1 * p.c); ls[2] = log(0.05); ls[3] = log(0.05); ls[4] = log(0.05);
        ls[5] = log(0.1); ls[6] = log(0.1); ls[7] = log(0.1 * (sc->dsrc_max > sc->dsrc_min ? sc->dsrc_max - sc->dsrc_min : 1.0));
        uint8_t *zc = &z[c * T * N], *yc = &y[c * (T - 1) * N];
        for (size_t t = 0; t < T; t++)
            for (size_t k = 0; k < N; k++) {
                const int o = obs[t * N + k];
                uint8_t v;
                if (o == 1) v = 1;
                else if (o == 0) v = 0;
                else if (disperse) v = u01(rng(h->cfg.seed, gc, 0, RK_INIT_Z, (uint32_t)k, (uint32_t)t).x) < 0.5;
                else v = 1;
                zc[t * N + k] = v;
            }
        for (size_t t = 0; t + 1 < T; t++)
            for (size_t k = 0; k < N; k++) yc[t * N + k] = zc[t * N + k] && zc[(t + 1) * N + k];
    }
    if ((rc = mp_set_params(h, par.data())) != MP_OK) return rc;
    if ((rc = mp_set_state(h, z.data(), y.data())) != MP_OK) return rc;
    h->sweep = 0; h->ndraws = 0;
    if ((rc = push_counters(h)) != MP_OK) return rc;
    // the sampler's resident S always comes from k_conn: its FP64 accumulation is what lets rank-1 removals cancel exactly
    if ((rc = check_ready(h)) != MP_OK) return rc;
    if ((rc = is64(h) ? refresh_S<double>(h, false) : refresh_S<float>(h, false)) != MP_OK) return rc;
    if (disperse) {
        // a dispersed start must be a possible state: an empty cell next year (y=0, z'=0) needs C < 1, i.e.
        // c < 1 / max(K_t S + Ksrc_t g); pull c below that bound (same rule as the CPU twin's spom_init_chain)
        std::vector<double> S(C * (T - 1) * N), unit(N);
        std::vector<uint8_t> era(T, 0);
        // the engine stream is non-blocking: copy on it (a default-stream cudaMemcpy would not wait for k_conn)
        CK(cudaMemcpyAsync(S.data(), h->d_S[0], S.size() * 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(unit.data(), h->d_src_unit, N * 8, cudaMemcpyDeviceToHost, h->stream));
        if (h->have_era) CK(cudaMemcpyAsync(era.data(), h->d_era, T - 1, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        for (size_t c = 0; c < C; c++) {
            mp_params &p = par[c];
            double smax = 0.0;
            for (size_t t = 0; t + 1 < T; t++) {
                const bool pre = era[t] != 0, src = pre && p.Ksrc != 0.0;
                for (size_t k = 0; k < N; k++) {
                    const size_t i = t * N + k;
                    if (y[c * (T - 1) * N + i] || z[c * T * N + i + N]) continue;
                    const double g = src ? exp(-p.alpha * unit[k] * p.dsrc) : 0.0;
                    const double v = pre ? p.K * S[c * (T - 1) * N + i] + p.Ksrc * g : S[c * (T - 1) * N + i];
                    if (v > smax) smax = v;
                }
            }
            if (smax > 0.0 && p.c * smax >= 1.0) { p.c = 0.5 / smax; if (p.c < sc->c_min) p.c = sc->c_min; }
            lsig[c * MP_NLSIG + 1] = log(0.1 * p.c);
        }
        if ((rc = mp_set_params(h, par.data())) != MP_OK) return rc;
        h->S_valid = true;                               // c does not enter S
    }
    return mp_set_scales(h, lsig.data());
}
int mp_sweep(mp_engine *h, int nsweeps)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    int rc = check_ready(h);
    if (rc != MP_OK) return rc;
    REQUIRE(h->have_sc && h->have_obs, MP_ERR_STATE, "sampler not configured (mp_init_chains / mp_set_sampler)");
    if ((rc = summaries_room(h, nsweeps)) != MP_OK) return rc;
    h->par_host_valid = false;                           // the sampler moves the parameters on the device
    for (int s = 0; s < nsweeps; s++) {
        // A sweep is ~20 launches that carry no per-sweep host value (the kernels read the sweep and draw counters from device
        // memory), so it is captured once per kind -- without / with the refresh of the resident S -- and replayed as a CUDA
        // graph: on small landscapes the sweep is launch-bound.  The first sweep of a kind runs eagerly (lazy allocations).
        const bool whole = h->conn_hi < 0 && h->task_first == 0 && h->task_stride == 1;
        if (h->use_graph && !h->timing && h->S_valid && h->S_exact && whole) {
            const int v = (is64(h) || h->refresh_every <= 1 || (h->sweep % (uint32_t)h->refresh_every) == 0) ? 1 : 0;
            if (!h->gexec[v] && h->gwarm[v]) {
                const uint32_t sweep0 = h->sweep; const int ndraws0 = h->ndraws; const unsigned long long samples0 = h->sum_samples;
                long long before[MP_K_NCAT];
                for (int i = 0; i < MP_K_NCAT; i++) before[i] = h->t_launch[i];
                cudaGraph_t g = nullptr;
                bool ok = cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
                if (ok) {
                    rc = is64(h) ? sweep_once<double>(h) : sweep_once<float>(h);
                    ok = cudaStreamEndCapture(h->stream, &g) == cudaSuccess && rc == MP_OK && g != nullptr;
                    if (ok) ok = cudaGraphInstantiate(&h->gexec[v], g, 0) == cudaSuccess;
                    if (g) cudaGraphDestroy(g);
                }
                h->sweep = sweep0; h->ndraws = ndraws0; h->sum_samples = samples0;   // nothing ran yet: the capture only advanced the host mirrors ...
                for (int i = 0; i < MP_K_NCAT; i++) { h->glaunch[v][i] = h->t_launch[i] - before[i]; h->t_launch[i] = before[i]; }   // ... and the launch counts, which every replay adds
                if (!ok) { cudaGetLastError(); h->gexec[v] = nullptr; h->use_graph = 0; }
            }
            if (h->gexec[v]) {
                CK(cudaGraphLaunch(h->gexec[v], h->stream));
                for (int i = 0; i < MP_K_NCAT; i++) h->t_launch[i] += h->glaunch[v][i];
                if (h->ndraws < h->cfg.max_draws) h->ndraws++;
                if (summary_due(h, h->sweep)) h->sum_samples += nC(h);
                h->sweep++;
                continue;
            }
            h->gwarm[v] = true;
        }
        rc = is64(h) ? sweep_once<double>(h) : sweep_once<float>(h);
        if (rc != MP_OK) return rc;
        if (h->timing && h->spans.size() > 16384) { CK(cudaStreamSynchronize(h->stream)); drain_spans(h); }
    }
    return MP_OK;
}
int mp_set_shard(mp_engine *h, int conn_lo, int conn_hi, int task_first, int task_stride)
{
    if (!h) return MP_ERR_ARG;
    const int ntask = h->cfg.n_chains * (h->cfg.n_years - 1);
    REQUIRE(task_stride >= 1 && task_first >= 0 && task_first < std::max(ntask, 1) + task_stride, MP_ERR_ARG, "mp_set_shard: bad task subset");
    REQUIRE(conn_hi < 0 || (conn_lo >= 0 && conn_lo <= conn_hi && conn_hi <= h->cfg.n_patches), MP_ERR_ARG, "mp_set_shard: bad patch range");
    // the culled k_conn takes its bounding boxes per 32-slot group and a CTA owns 256 targets: ranges must start on a CTA boundary
    REQUIRE(conn_hi < 0 || (conn_lo % 256 == 0 && (conn_hi % 256 == 0 || conn_hi == h->cfg.n_patches)), MP_ERR_ARG,
            "mp_set_shard: conn_lo and conn_hi must be multiples of 256 (conn_hi may also be n_patches)");
    h->conn_lo = conn_hi < 0 ? 0 : conn_lo; h->conn_hi = conn_hi; h->task_first = task_first; h->task_stride = task_stride;
    h->blk_tasks_dirty = true;
    drop_graphs(h);
    return MP_OK;
}
int mp_sweep_phase(mp_engine *h, int phase, int *flags_out)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    int rc = check_ready(h);
    if (rc != MP_OK) return rc;
    REQUIRE(h->have_sc && h->have_obs, MP_ERR_STATE, "sampler not configured (mp_init_chains / mp_set_sampler)");
    REQUIRE(!is64(h) || (h->conn_hi < 0 && h->task_stride == 1), MP_ERR_UNSUPPORTED, "sharded phases need the FP32 engine");
    h->par_host_valid = false;
    switch (phase) {
    case PH_PROPOSE_CONN: return is64(h) ? phase_propose_conn<double>(h, flags_out) : phase_propose_conn<float>(h, flags_out);
    case PH_DECIDE_Z: return is64(h) ? phase_decide_z<double>(h) : phase_decide_z<float>(h);
    case PH_SWEEP_Y: return is64(h) ? phase_sweep_y<double>(h) : phase_sweep_y<float>(h);
    case PH_FINISH:
        if ((rc = summaries_room(h, 1)) != MP_OK) return rc;
        return is64(h) ? phase_finish<double>(h) : phase_finish<float>(h);
    default: h->err = "mp_sweep_phase: unknown phase"; return MP_ERR_ARG;
    }
}
// ---- one set of chains over the ranks of a communicator (mp_comm.cu): the phases of a sweep with NCCL between them
// owned connectivity columns (layout slots [lo, lo + per) of every row of S) <-> a dense [row][per] buffer
static __global__ void k_pack_cols(const double *__restrict__ S, const int *__restrict__ perm, int n, int lo, int per, double *__restrict__ out)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x, row = blockIdx.y;
    if (s < per) out[(size_t)row * per + s] = lo + s < n ? S[(size_t)row * n + perm[lo + s]] : 0.0;
}
static __global__ void k_unpack_cols(double *__restrict__ S, const int *__restrict__ perm, int n, int per, int rows, const double *__restrict__ in)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x, row = blockIdx.y, r = blockIdx.z;
    if (s < per && r * per + s < n) S[(size_t)row * n + perm[r * per + s]] = in[((size_t)r * rows + row) * per + s];
}
enum { SH_CONN = 0, SH_GATHER = 1, SH_SCAN = 2, SH_ROWS = 3, SH_FINISH = 4 };
static int sharded_stage(mp_engine *h, int stage)
{
    CK(cudaSetDevice(h->cfg.device));
    const int n = h->cfg.n_patches, rows = h->cfg.n_chains * (h->cfg.n_years - 1), per = h->comm_per, W = h->comm_size;
    const dim3 pgrid((per + 255) / 256, rows), ugrid((per + 255) / 256, rows, W);
    int rc;
    switch (stage) {
    case SH_CONN:
        if ((rc = phase_propose_conn<float>(h, &h->shard_flags)) != MP_OK) return rc;
        for (int set = 0; set < 2; set++)
            if ((h->shard_flags >> set) & 1) {
                k_pack_cols<<<pgrid, 256, 0, h->stream>>>(h->d_S[set], h->d_perm, n, h->conn_lo, per, h->d_comm_send + (size_t)set * rows * per);
                CK(cudaGetLastError());
            }
        return MP_OK;
    case SH_GATHER:
        for (int set = 0; set < 2; set++)
            if ((h->shard_flags >> set) & 1)
                if ((rc = mp_comm_allgather(h, h->d_comm_send + (size_t)set * rows * per, h->d_comm_recv + (size_t)set * W * rows * per,
                                            (size_t)rows * per * 8)) != MP_OK) return rc;
        return MP_OK;
    case SH_SCAN:
        for (int set = 0; set < 2; set++)
            if ((h->shard_flags >> set) & 1) {
                k_unpack_cols<<<ugrid, 256, 0, h->stream>>>(h->d_S[set], h->d_perm, n, per, rows, h->d_comm_recv + (size_t)set * W * rows * per);
                CK(cudaGetLastError());
            }
        if ((rc = phase_decide_z<float>(h)) != MP_OK) return rc;
        return phase_sweep_y<float>(h);
    case SH_ROWS:   // the owner of (chain, year) task r is rank r mod W: its rows of y and S go to everybody
        for (int row = 0; row < rows; row++) {
            if ((rc = mp_comm_broadcast(h, h->d_S[0] + (size_t)row * n, (size_t)n * 8, row % W)) != MP_OK) return rc;
            if ((rc = mp_comm_broadcast(h, h->d_y + (size_t)row * n, (size_t)n, row % W)) != MP_OK) return rc;
        }
        return MP_OK;
    default:
        return phase_finish<float>(h);
    }
}
static int sharded_prepare(mp_engine *h)
{
    CK(cudaSetDevice(h->cfg.device));
    int rc = check_ready(h);
    if (rc != MP_OK) return rc;
    REQUIRE(h->comm, MP_ERR_STATE, "mp_sweep_sharded: no communicator (mp_comm_init / mp_comm_init_all)");
    REQUIRE(h->have_sc && h->have_obs, MP_ERR_STATE, "sampler not configured (mp_init_chains / mp_set_sampler)");
    REQUIRE(!is64(h), MP_ERR_UNSUPPORTED, "sharded sweeps need the FP32 engine");
    const int n = h->cfg.n_patches, per = h->comm_per, W = h->comm_size, r = h->comm_rank;
    const size_t rows = nC(h) * (nT(h) - 1);
    if ((rc = mp_set_shard(h, std::min(n, r * per), std::min(n, (r + 1) * per), r, W)) != MP_OK) return rc;
    if (!h->d_comm_send) {
        CK(cudaMalloc(&h->d_comm_send, 2 * rows * per * 8));
        CK(cudaMalloc(&h->d_comm_recv, 2 * rows * per * 8 * (size_t)W));
    }
    h->par_host_valid = false;
    return MP_OK;
}
int mp_sweep_sharded_all(mp_engine **hs, int n, int nsweeps)
{
    if (!hs || n < 1 || !hs[0]) return MP_ERR_ARG;
    int rc;
    for (int i = 0; i < n; i++) { if (!hs[i]) return MP_ERR_ARG; if ((rc = sharded_prepare(hs[i])) != MP_OK) return rc; }
    for (int i = 0; i < n; i++) if ((rc = summaries_room(hs[i], nsweeps)) != MP_OK) return rc;
    for (int s = 0; s < nsweeps; s++)
        for (int stage = SH_CONN; stage <= SH_FINISH; stage++) {
            const bool coll = stage == SH_GATHER || stage == SH_ROWS;   // the collectives of all local engines form one NCCL group
            if (coll && (rc = mp_comm_group_start(hs[0])) != MP_OK) return rc;
            for (int i = 0; i < n; i++) if ((rc = sharded_stage(hs[i], stage)) != MP_OK) return rc;
            if (coll && (rc = mp_comm_group_end(hs[0])) != MP_OK) return rc;
        }
    return MP_OK;
}
int mp_sweep_sharded(mp_engine *h, int nsweeps) { return mp_sweep_sharded_all(&h, 1, nsweeps); }
int mp_synchronize(mp_engine *h)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    return MP_OK;
}
int mp_set_summaries(mp_engine *h, int first_sweep, int thin)
{
    if (!h) return MP_ERR_ARG;
    REQUIRE(first_sweep >= 0 && thin >= 0, MP_ERR_ARG, "mp_set_summaries: first_sweep and thin must be >= 0");
    CK(cudaSetDevice(h->cfg.device));
    int rc = quiesce(h);                                 // the captured sweeps launch k_summaries or not: capture again
    if (rc != MP_OK) return rc;
    h->sum_first = first_sweep; h->sum_thin = thin; h->sum_samples = 0;
    if (thin == 0) {
        if (h->d_sum) { CK(cudaFree(h->d_sum)); h->d_sum = nullptr; }
        return MP_OK;
    }
    const SumLayout L = sum_layout(h);
    if (!h->d_sum) {
        cudaError_t e = cudaMalloc(&h->d_sum, L.bytes);
        if (e != cudaSuccess) { h->d_sum = nullptr; h->sum_thin = 0; h->err = std::string("mp_set_summaries: ") + cudaGetErrorString(e); return MP_ERR_CUDA; }
    }
    CK(cudaMemsetAsync(h->d_sum, 0, L.bytes, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MP_OK;
}
int mp_get_summaries(mp_engine *h, int64_t *nsamples, uint32_t *z_count, double *z_prob, uint32_t *y_count, double *S_sum, int reset)
{
    if (!h) return MP_ERR_ARG;
    REQUIRE(h->d_sum, MP_ERR_STATE, "mp_get_summaries: summaries not set (mp_set_summaries)");
    CK(cudaSetDevice(h->cfg.device));
    const SumLayout L = sum_layout(h);
    unsigned long long ns = 0;
    CK(cudaMemcpyAsync(&ns, h->d_sum + L.nsamples, 8, cudaMemcpyDeviceToHost, h->stream));
    if (z_count) CK(cudaMemcpyAsync(z_count, h->d_sum + L.z_count, zcells(h) * 4, cudaMemcpyDeviceToHost, h->stream));
    if (z_prob) CK(cudaMemcpyAsync(z_prob, h->d_sum + L.z_prob, zcells(h) * 8, cudaMemcpyDeviceToHost, h->stream));
    if (y_count) CK(cudaMemcpyAsync(y_count, h->d_sum + L.y_count, ycells(h) * 4, cudaMemcpyDeviceToHost, h->stream));
    if (S_sum) CK(cudaMemcpyAsync(S_sum, h->d_sum + L.S_sum, ycells(h) * 8, cudaMemcpyDeviceToHost, h->stream));
    if (reset) CK(cudaMemsetAsync(h->d_sum, 0, L.bytes, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (nsamples) *nsamples = (int64_t)ns;
    if (reset) h->sum_samples = 0;
    return MP_OK;
}
int mp_set_waic(mp_engine *h, int first_sweep, int thin)
{
    if (!h) return MP_ERR_ARG;
    REQUIRE(first_sweep >= 0 && thin >= 0, MP_ERR_ARG, "mp_set_waic: first_sweep and thin must be >= 0");
    REQUIRE(thin == 0 || h->have_obs, MP_ERR_STATE, "mp_set_waic: no observations (mp_set_observations)");
    CK(cudaSetDevice(h->cfg.device));
    int rc = quiesce(h);                                 // the captured sweeps launch k_waic or not: capture again
    if (rc != MP_OK) return rc;
    h->waic_first = first_sweep; h->waic_thin = thin;
    if (thin == 0) {
        if (h->d_waic) { CK(cudaFree(h->d_waic)); h->d_waic = nullptr; }
        return MP_OK;
    }
    if (!h->d_waic) {
        cudaError_t e = cudaMalloc(&h->d_waic, waic_bytes(h));
        if (e != cudaSuccess) { h->d_waic = nullptr; h->waic_thin = 0; h->err = std::string("mp_set_waic: ") + cudaGetErrorString(e); return MP_ERR_CUDA; }
    }
    CK(cudaMemsetAsync(h->d_waic, 0, waic_bytes(h), h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MP_OK;
}
int mp_get_waic(mp_engine *h, int64_t *nsamples, double *lik_sum, double *loglik_sum, double *loglik_sq, int reset)
{
    if (!h) return MP_ERR_ARG;
    REQUIRE(h->d_waic, MP_ERR_STATE, "mp_get_waic: WAIC sums not set (mp_set_waic)");
    CK(cudaSetDevice(h->cfg.device));
    const size_t plane = zcells(h) * 8;
    unsigned long long ns = 0;
    CK(cudaMemcpyAsync(&ns, h->d_waic + 3 * plane, 8, cudaMemcpyDeviceToHost, h->stream));
    if (lik_sum) CK(cudaMemcpyAsync(lik_sum, h->d_waic, plane, cudaMemcpyDeviceToHost, h->stream));
    if (loglik_sum) CK(cudaMemcpyAsync(loglik_sum, h->d_waic + plane, plane, cudaMemcpyDeviceToHost, h->stream));
    if (loglik_sq) CK(cudaMemcpyAsync(loglik_sq, h->d_waic + 2 * plane, plane, cudaMemcpyDeviceToHost, h->stream));
    if (reset) CK(cudaMemsetAsync(h->d_waic, 0, waic_bytes(h), h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (nsamples) *nsamples = (int64_t)ns;
    return MP_OK;
}
int mp_set_sources(mp_engine *h, int first_sweep, int thin, int nbins, double bin_width)
{
    if (!h) return MP_ERR_ARG;
    REQUIRE(first_sweep >= 0 && thin >= 0, MP_ERR_ARG, "mp_set_sources: first_sweep and thin must be >= 0");
    REQUIRE(nbins >= 0 && nbins <= SRC_MAX_BINS, MP_ERR_ARG, "mp_set_sources: nbins must be in [0, 4096]");
    REQUIRE(nbins == 0 || (std::isfinite(bin_width) && bin_width > 0.0), MP_ERR_ARG, "mp_set_sources: bin_width must be finite and > 0");
    CK(cudaSetDevice(h->cfg.device));
    int rc = quiesce(h);                                 // the captured sweeps launch the source kernels or not: capture again
    if (rc != MP_OK) return rc;
    const size_t old = h->d_src ? src_layout(h, h->src_nbins).bytes : 0;
    h->src_first = first_sweep; h->src_thin = thin; h->src_nbins = nbins; h->src_bin_width = nbins > 0 ? bin_width : 0.0;
    const size_t bytes = src_layout(h, nbins).bytes;
    if (h->d_src && (thin == 0 || bytes != old)) { CK(cudaFree(h->d_src)); h->d_src = nullptr; }
    if (thin == 0) return MP_OK;
    if (!h->d_src) {
        cudaError_t e = cudaMalloc(&h->d_src, bytes);
        if (e != cudaSuccess) { h->d_src = nullptr; h->src_thin = 0; h->err = std::string("mp_set_sources: ") + cudaGetErrorString(e); return MP_ERR_CUDA; }
    }
    CK(cudaMemsetAsync(h->d_src, 0, bytes, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MP_OK;
}
int mp_get_sources(mp_engine *h, int64_t *nsamples, uint64_t *events, double *src_sum, double *ext_sum, double *dist_hist, int reset)
{
    if (!h) return MP_ERR_ARG;
    REQUIRE(h->d_src, MP_ERR_STATE, "mp_get_sources: source sums not set (mp_set_sources)");
    CK(cudaSetDevice(h->cfg.device));
    const SrcLayout L = src_layout(h, h->src_nbins);
    const size_t ntrans = nT(h) - 1;
    unsigned long long ns = 0;
    CK(cudaMemcpyAsync(&ns, h->d_src + L.nsamples, 8, cudaMemcpyDeviceToHost, h->stream));
    if (events) CK(cudaMemcpyAsync(events, h->d_src + L.events, 2 * ntrans * 8, cudaMemcpyDeviceToHost, h->stream));
    if (src_sum) CK(cudaMemcpyAsync(src_sum, h->d_src + L.src_sum, ycells(h) * 8, cudaMemcpyDeviceToHost, h->stream));
    if (ext_sum) CK(cudaMemcpyAsync(ext_sum, h->d_src + L.ext_sum, ntrans * 8, cudaMemcpyDeviceToHost, h->stream));
    if (dist_hist && h->src_nbins > 0)
        CK(cudaMemcpyAsync(dist_hist, h->d_src + L.dist_hist, ntrans * h->src_nbins * 8, cudaMemcpyDeviceToHost, h->stream));
    if (reset) CK(cudaMemsetAsync(h->d_src + L.sums, 0, L.bytes - L.sums, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (nsamples) *nsamples = (int64_t)ns;
    return MP_OK;
}
int mp_num_draws(mp_engine *h) { return h ? h->ndraws : MP_ERR_ARG; }
int mp_sweep_index(mp_engine *h) { return h ? (int)h->sweep : MP_ERR_ARG; }
int mp_reset_draws(mp_engine *h) { if (!h) return MP_ERR_ARG; h->ndraws = 0; return push_counters(h); }
int mp_get_draws(mp_engine *h, int first, int count, double *out)
{
    if (!h || !out) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    REQUIRE(first >= 0 && count >= 0 && first + count <= h->ndraws, MP_ERR_ARG, "mp_get_draws: range outside recorded draws");
    const size_t row = nC(h) * MP_NDRAW * 8;
    CK(cudaMemcpyAsync(out, (const char *)h->d_draws + (size_t)first * row, (size_t)count * row, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MP_OK;
}

// ---- forward simulator
extern "C++" template <typename R> int simulate_t(mp_engine *h, const mp_params *d_pars, int per_sim, const uint8_t *d_z0, int nyears,
                                                  int nsims, uint64_t seed, int era_all, uint8_t *d_zout, int32_t *d_occ, uint8_t *d_zc,
                                                  uint8_t *d_yc, int *d_list, int *d_nlist, R *d_aw)
{
    Timed tm(h, MP_K_SIM);
    const int n = h->cfg.n_patches, npar = per_sim ? nsims : 1;
    k_area_weights<R><<<dim3((n + 255) / 256, npar), 256, 0, h->stream>>>(d_pars, h->have_area ? h->d_area : nullptr, d_aw, n);
    CK(cudaGetLastError());
    if (d_occ) CK(cudaMemsetAsync(d_occ, 0, (size_t)nsims * (nyears + 1) * 4, h->stream));
    k_sim_init<<<nsims, 256, 0, h->stream>>>(d_z0, per_sim, n, nyears, d_zc, d_zout, d_occ);
    CK(cudaGetLastError());
    const dim3 cgrid((n + 127) / 128, nsims);
    for (int t = 0; t < nyears; t++) {
        k_sim_ext<R><<<nsims, 1024, 0, h->stream>>>(d_pars, per_sim, n, seed, 0u, t, era_all, d_zc, d_yc, d_list, d_nlist);
        CK(cudaGetLastError());
#define SIM(G) k_sim_col<R, G><<<cgrid, 128, 0, h->stream>>>(view<R>(h), d_pars, per_sim, d_aw, d_yc, d_list, d_nlist, seed, 0u, t, nyears, era_all, d_zc, d_zout, d_occ)
        switch (h->geom) {
        case MP_GEOM_LINEAR: SIM(MP_GEOM_LINEAR); break;
        case MP_GEOM_COORDS: SIM(MP_GEOM_COORDS); break;
        default: SIM(MP_GEOM_DENSE); break;
        }
#undef SIM
        CK(cudaGetLastError());
    }
    return MP_OK;
}
static int simulate_impl(mp_engine *h, const mp_params *par, int per_sim, const uint8_t *z0, int nyears, int nsims, uint64_t seed,
                         int era_all, uint8_t *z_out, int32_t *occupied_out)
{
    if (!h || !par || !z0) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    REQUIRE(h->have_landscape, MP_ERR_STATE, "landscape not set");
    REQUIRE(nyears >= 1 && nsims >= 1, MP_ERR_ARG, "mp_simulate: need nyears>=1, nsims>=1");
    const int npar = per_sim ? nsims : 1;
    for (int i = 0; i < npar; i++) REQUIRE(par[i].K > 0.0 && par[i].alpha > 0.0, MP_ERR_ARG, "mp_simulate: need K>0 and alpha>0");
    const size_t N = nN(h), nz0 = per_sim ? (size_t)nsims * N : N;
    // one arena per call: start states, parameters, current / intermediate state, survivor lists, A^b, outputs
    size_t off = 0;
    auto carve = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t o_z0 = carve(nz0), o_par = carve((size_t)npar * sizeof(mp_params)), o_zc = carve((size_t)nsims * N), o_yc = carve((size_t)nsims * N),
                 o_list = carve((size_t)nsims * N * 4), o_nl = carve((size_t)nsims * 4), o_aw = carve((size_t)npar * N * 8),
                 o_zout = carve(z_out ? (size_t)nsims * (nyears + 1) * N : 0), o_occ = carve(occupied_out ? (size_t)nsims * (nyears + 1) * 4 : 0);
    unsigned char *arena = nullptr;
    int rc = MP_OK;
    cudaError_t e;
#define SIMCK(call) if ((e = (call)) != cudaSuccess) { h->err = std::string(#call) + ": " + cudaGetErrorString(e); rc = MP_ERR_CUDA; goto done; }
    SIMCK(cudaMalloc(&arena, std::max<size_t>(off, 256)));
    {
        uint8_t *d_z0 = arena + o_z0, *d_zc = arena + o_zc, *d_yc = arena + o_yc, *d_zout = z_out ? arena + o_zout : nullptr;
        mp_params *d_pars = (mp_params *)(arena + o_par);
        int *d_list = (int *)(arena + o_list), *d_nlist = (int *)(arena + o_nl);
        int32_t *d_occ = occupied_out ? (int32_t *)(arena + o_occ) : nullptr;
        SIMCK(cudaMemcpyAsync(d_z0, z0, nz0, cudaMemcpyHostToDevice, h->stream));
        SIMCK(cudaMemcpyAsync(d_pars, par, (size_t)npar * sizeof(mp_params), cudaMemcpyHostToDevice, h->stream));
        rc = is64(h) ? simulate_t<double>(h, d_pars, per_sim, d_z0, nyears, nsims, seed, era_all, d_zout, d_occ, d_zc, d_yc, d_list, d_nlist, (double *)(arena + o_aw))
                     : simulate_t<float>(h, d_pars, per_sim, d_z0, nyears, nsims, seed, era_all, d_zout, d_occ, d_zc, d_yc, d_list, d_nlist, (float *)(arena + o_aw));
        if (rc != MP_OK) goto done;
        if (z_out) SIMCK(cudaMemcpyAsync(z_out, d_zout, (size_t)nsims * (nyears + 1) * N, cudaMemcpyDeviceToHost, h->stream));
        if (occupied_out) SIMCK(cudaMemcpyAsync(occupied_out, d_occ, (size_t)nsims * (nyears + 1) * 4, cudaMemcpyDeviceToHost, h->stream));
        SIMCK(cudaStreamSynchronize(h->stream));
    }
#undef SIMCK
done:
    cudaFree(arena);
    return rc;
}
int mp_simulate(mp_engine *h, const mp_params *par, const uint8_t *z0, int nyears, int nsims, uint64_t seed, int era_all,
                uint8_t *z_out, int32_t *occupied_out)
{
    return simulate_impl(h, par, 0, z0, nyears, nsims, seed, era_all, z_out, occupied_out);
}
int mp_simulate_ensemble(mp_engine *h, const mp_params *par_per_sim, const uint8_t *z0_per_sim, int nyears, int nsims,
                         uint64_t seed, int era_all, uint8_t *z_out, int32_t *occupied_out)
{
    return simulate_impl(h, par_per_sim, 1, z0_per_sim, nyears, nsims, seed, era_all, z_out, occupied_out);
}

// ---- replicates of the chains' own state: the year loop of mp_forecast and mp_ppc
// Buffers of one call (one arena); states and S are [chain][replicate][patch], records [chain][word][padded slot]
struct FcBufs {
    const mp_params *par; void *aw; uint8_t *zc, *yc; double *S; void *rec; float *mlow; int32_t *occ; uint32_t *inc;
};
// nyears transitions of nrep trajectories per chain from z[c][t0]; transition t applies K, Ksrc iff era[t].  after_year(t) runs
// once the states of year t are in zc: t = 0 after the start states, t + 1 after the colonisation draws of transition t.
extern "C++" template <typename R, typename F>
int replicate_t(mp_engine *h, const FcBufs &b, int t0, int nyears, int nrep, uint64_t seed, const uint8_t *era, F after_year)
{
    Timed tm(h, MP_K_SIM);
    const int n = h->cfg.n_patches, C = h->cfg.n_chains, T = h->cfg.n_years, npad = conn_npad(n), nwords = (nrep + 31) / 32;
    const unsigned tiles = (unsigned)((n + 255) / 256);
    const uint32_t sim0 = (uint32_t)h->cfg.chain_offset * (uint32_t)nrep;
    mp::Landscape<R> ls = view<R>(h), lsrc = ls;
    if (h->geom != MP_GEOM_COORDS) { lsrc.px = nullptr; lsrc.py = nullptr; }
    k_area_weights<R><<<dim3(tiles, C), 256, 0, h->stream>>>(b.par, h->have_area ? h->d_area : nullptr, (R *)b.aw, n);
    CK(cudaGetLastError());
    k_fc_init<<<dim3(tiles, C), 256, 0, h->stream>>>(h->d_z, T, t0, n, nrep, nyears, b.zc, b.occ, b.inc);
    CK(cudaGetLastError());
    int rc;
    if ((rc = after_year(0)) != MP_OK) return rc;
    // k_conn over the call's own buffers: every target, the replicates in place of the years, the call's culling floor
    ConnArgs<R> a;
    a.ls = ls;
    a.par[0] = a.par[1] = b.par;
    a.S[0] = a.S[1] = b.S;
    a.rec = (const SrcRec<R> *)b.rec;
    a.ntrans = nrep; a.nwords = nwords; a.nchains = C; a.set_base = 0;
    a.k_lo = 0; a.k_hi = n;
    a.perm = h->d_perm; a.box32 = (const float4 *)h->d_tile_box;
    a.mlow = b.mlow; a.area_max = (float)h->area_max; a.area_min = (float)h->area_min;
    a.stats = h->d_work;
    for (int t = 0; t < nyears; t++) {
        k_fc_ext<R><<<dim3(tiles, nrep, C), 256, 0, h->stream>>>(b.par, n, nrep, seed, sim0, t, era[t], b.zc, b.yc);
        CK(cudaGetLastError());
        k_pack_sources<R><<<dim3((npad + 255) / 256, C, nwords), 256, 0, h->stream>>>(lsrc, h->d_perm, (const R *)b.aw, nullptr, b.yc, nrep,
                                                                                      nwords, 1, (SrcRec<R> *)b.rec);
        CK(cudaGetLastError());
        switch (h->geom) {
        case MP_GEOM_LINEAR: rc = launch_conn_args<R, MP_GEOM_LINEAR>(h, a, 1, false); break;
        case MP_GEOM_COORDS: rc = launch_conn_args<R, MP_GEOM_COORDS>(h, a, 1, false); break;
        default: rc = launch_conn_args<R, MP_GEOM_DENSE>(h, a, 1, false); break;
        }
        if (rc != MP_OK) return rc;
        k_fc_col<R><<<dim3(tiles, C), 256, 0, h->stream>>>(ls, b.par, nrep, seed, sim0, t, nyears, era[t], b.S, b.yc, b.zc, b.occ, b.inc);
        CK(cudaGetLastError());
        if ((rc = after_year(t + 1)) != MP_OK) return rc;
    }
    return MP_OK;
}
// The part of a call's arena that replicate_t needs: parameters, A^b, current / surviving states, S, source records, culling
// floor.  rep_carve reserves it at the front of the arena, rep_upload points b at it and uploads the parameters and the floor.
struct RepLayout { size_t par, aw, zc, yc, S, rec, mlow; };
extern "C++" template <typename F> RepLayout rep_carve(const mp_engine *h, int nrep, F carve)
{
    const size_t N = nN(h), C = nC(h), cells = C * (size_t)nrep * N, ngroups = (N + 31) / 32;
    const size_t nwords = ((size_t)nrep + 31) / 32, npad = (size_t)conn_npad((int)N);
    const size_t rec_bytes = is64(h) ? sizeof(SrcRec<double>) : sizeof(SrcRec<float>);
    RepLayout L;
    L.par = carve(C * sizeof(mp_params)); L.aw = carve(C * N * rsz(h)); L.zc = carve(cells); L.yc = carve(cells);
    L.S = carve(cells * 8); L.rec = carve(C * nwords * npad * rec_bytes); L.mlow = carve(C * ngroups * sizeof(float));
    return L;
}
// Culling floor of k_conn (FP32 engines with positions): a source group is skipped for a target group when every weight
// between them is below 2^-30 mlow_c, so the skipped weights change c K_t S of a target by less than N 2^-30 mlow_c c Keff_c =
// 2^-32 (the resolution of the uniform that decides a colonisation) with mlow_c = 2^-2 / (c Keff_c N), Keff_c >= every K_t of
// chain c that the call applies.
static int rep_upload(mp_engine *h, unsigned char *arena, const RepLayout &L, const std::vector<mp_params> &par,
                      const std::vector<double> &Keff, FcBufs &b)
{
    const size_t N = nN(h), C = nC(h), ngroups = (N + 31) / 32;
    std::vector<float> mlow(C * ngroups);
    for (size_t c = 0; c < C; c++)
        std::fill(mlow.begin() + c * ngroups, mlow.begin() + (c + 1) * ngroups, (float)std::min(0.25 / (par[c].c * Keff[c] * (double)N), 3.0e38));
    b.par = (const mp_params *)(arena + L.par); b.aw = arena + L.aw; b.zc = arena + L.zc; b.yc = arena + L.yc;
    b.S = (double *)(arena + L.S); b.rec = arena + L.rec; b.mlow = (float *)(arena + L.mlow);
    b.occ = nullptr; b.inc = nullptr;
    CK(cudaMemcpyAsync(arena + L.par, par.data(), C * sizeof(mp_params), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(b.mlow, mlow.data(), mlow.size() * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    return MP_OK;
}
// the chains' parameters after any queued sweeps
static int chain_params(mp_engine *h, std::vector<mp_params> &par, const char *who)
{
    par.resize(nC(h));
    CK(cudaMemcpyAsync(par.data(), h->d_par, nC(h) * sizeof(mp_params), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (const mp_params &p : par) REQUIRE(p.alpha > 0.0, MP_ERR_STATE, std::string(who) + ": every chain needs alpha > 0");
    return MP_OK;
}

// ---- posterior-predictive forecast from the chains' own state
int mp_forecast(mp_engine *h, int nyears, int nrep, uint64_t seed, const double *scenario, int32_t *occupied_out, uint32_t *incidence_out)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    REQUIRE(nyears >= 1 && nrep >= 1, MP_ERR_ARG, "mp_forecast: need nyears >= 1 and nrep >= 1");
    REQUIRE(nrep <= 65535, MP_ERR_ARG, "mp_forecast: at most 65535 replicates per chain");
    REQUIRE((uint64_t)(h->cfg.chain_offset + h->cfg.n_chains) * (uint64_t)nrep <= 0xffffffffull, MP_ERR_ARG,
            "mp_forecast: simulation numbers (chain_offset + n_chains) * nrep must fit in 32 bits");
    REQUIRE(!scenario || scenario[0] > 0.0, MP_ERR_ARG, "mp_forecast: the scenario needs K > 0");
    int rc = check_ready(h);
    if (rc != MP_OK) return rc;
    const size_t N = nN(h), C = nC(h);
    // a scenario replaces K, Ksrc, dsrc and applies them every year
    std::vector<mp_params> par;
    if ((rc = chain_params(h, par, "mp_forecast")) != MP_OK) return rc;
    if (scenario)
        for (mp_params &p : par) { p.K = scenario[0]; p.Ksrc = scenario[1]; p.dsrc = scenario[2]; }
    const std::vector<double> Keff(C, scenario ? scenario[0] : 1.0);
    const std::vector<uint8_t> era((size_t)nyears, scenario ? 1 : 0);
    // one arena per call: replicate_t's buffers, outputs
    size_t off = 0;
    auto carve = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const RepLayout L = rep_carve(h, nrep, carve);
    const size_t occ_bytes = C * (size_t)nrep * (nyears + 1) * 4, inc_bytes = (size_t)(nyears + 1) * N * 4;
    const size_t o_occ = carve(occupied_out ? occ_bytes : 0), o_inc = carve(incidence_out ? inc_bytes : 0);
    unsigned char *arena = nullptr;
    cudaError_t e;
#define FCCK(call) if ((e = (call)) != cudaSuccess) { h->err = std::string(#call) + ": " + cudaGetErrorString(e); rc = MP_ERR_CUDA; goto done; }
    FCCK(cudaMalloc(&arena, std::max<size_t>(off, 256)));
    {
        FcBufs b;
        if ((rc = rep_upload(h, arena, L, par, Keff, b)) != MP_OK) goto done;
        b.occ = occupied_out ? (int32_t *)(arena + o_occ) : nullptr; b.inc = incidence_out ? (uint32_t *)(arena + o_inc) : nullptr;
        if (b.occ) FCCK(cudaMemsetAsync(b.occ, 0, occ_bytes, h->stream));
        if (b.inc) FCCK(cudaMemsetAsync(b.inc, 0, inc_bytes, h->stream));
        auto none = [](int) { return MP_OK; };
        const int t0 = h->cfg.n_years - 1;
        rc = is64(h) ? replicate_t<double>(h, b, t0, nyears, nrep, seed, era.data(), none)
                     : replicate_t<float>(h, b, t0, nyears, nrep, seed, era.data(), none);
        if (rc != MP_OK) goto done;
        if (occupied_out) FCCK(cudaMemcpyAsync(occupied_out, b.occ, occ_bytes, cudaMemcpyDeviceToHost, h->stream));
        if (incidence_out) FCCK(cudaMemcpyAsync(incidence_out, b.inc, inc_bytes, cudaMemcpyDeviceToHost, h->stream));
        FCCK(cudaStreamSynchronize(h->stream));
    }
#undef FCCK
done:
    cudaStreamSynchronize(h->stream);
    cudaFree(arena);
    return rc;
}

// ---- posterior-predictive replicates of the observation table (DESIGN.md §2)
int mp_ppc(mp_engine *h, int nrep, uint64_t seed, int32_t *stats_out, int32_t *obs_stats_out, uint32_t *patch_ge, uint32_t *patch_gt)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    REQUIRE(nrep >= 1 && nrep <= 65535, MP_ERR_ARG, "mp_ppc: need 1 <= nrep <= 65535");
    REQUIRE((uint64_t)(h->cfg.chain_offset + h->cfg.n_chains) * (uint64_t)nrep <= 0xffffffffull, MP_ERR_ARG,
            "mp_ppc: simulation numbers (chain_offset + n_chains) * nrep must fit in 32 bits");
    int rc = check_ready(h);
    if (rc != MP_OK) return rc;
    REQUIRE(h->have_obs, MP_ERR_STATE, "mp_ppc: observations not set");
    const int T = h->cfg.n_years;
    const size_t N = nN(h), C = nC(h);
    std::vector<mp_params> par;
    if ((rc = chain_params(h, par, "mp_ppc")) != MP_OK) return rc;
    // the fit's era flags, transition by transition (none set: none apply)
    std::vector<uint8_t> era((size_t)T, 0);
    std::vector<int8_t> obs(T * N);
    if (h->have_era) CK(cudaMemcpyAsync(era.data(), h->d_era, T - 1, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(obs.data(), h->d_obs, obs.size(), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    bool any_era = false;
    for (int t = 0; t + 1 < T; t++) any_era = any_era || era[t] != 0;
    std::vector<double> Keff(C, 1.0);
    if (any_era)
        for (size_t c = 0; c < C; c++) Keff[c] = std::max(1.0, par[c].K);
    if (obs_stats_out) {
        std::fill(obs_stats_out, obs_stats_out + (size_t)T * MP_NPPC, 0);
        for (int t = 0; t < T; t++)
            for (size_t k = 0; k < N; k++) {
                const int o = obs[t * N + k], op = t > 0 ? obs[(t - 1) * N + k] : -1;
                obs_stats_out[t * MP_NPPC + 0] += o == 1;
                if (o >= 0 && op >= 0) { obs_stats_out[t * MP_NPPC + 1] += op == 0 && o == 1; obs_stats_out[t * MP_NPPC + 2] += op == 1 && o == 0; }
            }
    }
    // one arena per call: replicate_t's buffers, per-replicate records, statistics, per-patch counts
    size_t off = 0;
    auto carve = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const RepLayout L = rep_carve(h, nrep, carve);
    const size_t stats_bytes = C * (size_t)nrep * T * MP_NPPC * 4;
    const size_t o_rec = carve(C * (size_t)nrep * N * 4), o_stats = carve(stats_bytes), o_ge = carve(N * 4), o_gt = carve(N * 4);
    unsigned char *arena = nullptr;
    cudaError_t e;
#define PPCK(call) if ((e = (call)) != cudaSuccess) { h->err = std::string(#call) + ": " + cudaGetErrorString(e); rc = MP_ERR_CUDA; goto done; }
    PPCK(cudaMalloc(&arena, std::max<size_t>(off, 256)));
    {
        FcBufs b;
        if ((rc = rep_upload(h, arena, L, par, Keff, b)) != MP_OK) goto done;
        uint32_t *rec = (uint32_t *)(arena + o_rec), *ge = (uint32_t *)(arena + o_ge), *gt = (uint32_t *)(arena + o_gt);
        int32_t *stats = (int32_t *)(arena + o_stats);
        PPCK(cudaMemsetAsync(stats, 0, stats_bytes, h->stream));
        PPCK(cudaMemsetAsync(ge, 0, N * 4, h->stream));
        PPCK(cudaMemsetAsync(gt, 0, N * 4, h->stream));
        const dim3 grid((unsigned)((N + 255) / 256), (unsigned)C);
        const uint32_t sim0 = (uint32_t)h->cfg.chain_offset * (uint32_t)nrep;
        auto observe = [&](int t) {
            k_ppc_obs<<<grid, 256, 0, h->stream>>>(b.par, h->d_obs, T, (int)N, nrep, seed, sim0, t, h->cfg.detect, b.zc, rec, stats, ge, gt);
            CK(cudaGetLastError());
            return MP_OK;
        };
        rc = is64(h) ? replicate_t<double>(h, b, 0, T - 1, nrep, seed, era.data(), observe)
                     : replicate_t<float>(h, b, 0, T - 1, nrep, seed, era.data(), observe);
        if (rc != MP_OK) goto done;
        if (stats_out) PPCK(cudaMemcpyAsync(stats_out, stats, stats_bytes, cudaMemcpyDeviceToHost, h->stream));
        if (patch_ge) PPCK(cudaMemcpyAsync(patch_ge, ge, N * 4, cudaMemcpyDeviceToHost, h->stream));
        if (patch_gt) PPCK(cudaMemcpyAsync(patch_gt, gt, N * 4, cudaMemcpyDeviceToHost, h->stream));
        PPCK(cudaStreamSynchronize(h->stream));
    }
#undef PPCK
done:
    cudaStreamSynchronize(h->stream);
    cudaFree(arena);
    return rc;
}

}  // extern "C"

// ---- metapopulation capacity (DESIGN.md §2): LOBPCG with block size 1 (Knyazev 2001) on M~ = D^1/2 K D^1/2, per parameter set

// Rayleigh-Ritz step of one set on the basis (x, r, p), p only when has_p.  g: the CAP_NGRAM inner products of k_cap_gram.  The
// basis is scaled to unit norms; while the Cholesky factor of its Gram matrix has a squared pivot below CAP_GRAM_TOL, p and then r
// leave the basis (Hetmaniuk & Lehoucq 2006: restart without the search direction).  Returns the coefficients of the Ritz vector of
// the largest Ritz value mu (unit norm, x coefficient >= 0) and the size of the basis that was used.
constexpr double CAP_GRAM_TOL = 1e-10;
static int cap_ritz(const double *g, bool has_p, double c[3], double &mu)
{
    const double A[3][3] = { { g[0], g[1], g[2] }, { g[1], g[3], g[4] }, { g[2], g[4], g[5] } };
    const double B[3][3] = { { g[6], g[7], g[8] }, { g[7], g[9], g[10] }, { g[8], g[10], g[11] } };
    int m = has_p ? 3 : 2;
    double d[3] = { 0, 0, 0 }, L[3][3];
    for (int i = 0; i < m; i++) {
        if (!(B[i][i] > 0.0) || !std::isfinite(B[i][i])) { m = i; break; }
        d[i] = 1.0 / std::sqrt(B[i][i]);
    }
    for (;; m--) {                                        // m >= 1: x itself always has a positive norm
        bool ok = true;
        for (int i = 0; i < m && ok; i++)
            for (int j = 0; j <= i; j++) {
                double s = B[i][j] * d[i] * d[j];
                for (int q = 0; q < j; q++) s -= L[i][q] * L[j][q];
                if (i == j) { if (!(s > CAP_GRAM_TOL)) { ok = false; break; } L[i][i] = std::sqrt(s); }
                else L[i][j] = s / L[j][j];
            }
        if (ok || m == 1) break;
    }
    if (m == 1) { c[0] = d[0]; c[1] = c[2] = 0.0; mu = A[0][0] * d[0] * d[0]; return 1; }
    // C = L^-1 An L^-T (An: A scaled like B), then its eigenpairs by cyclic Jacobi rotations
    double Y[3][3], Cm[3][3], V[3][3];
    for (int col = 0; col < m; col++)
        for (int i = 0; i < m; i++) {
            double s = A[i][col] * d[i] * d[col];
            for (int q = 0; q < i; q++) s -= L[i][q] * Y[q][col];
            Y[i][col] = s / L[i][i];
        }
    for (int col = 0; col < m; col++)
        for (int i = 0; i < m; i++) {
            double s = Y[col][i];
            for (int q = 0; q < i; q++) s -= L[i][q] * Cm[q][col];
            Cm[i][col] = s / L[i][i];
        }
    for (int i = 0; i < m; i++)
        for (int j = 0; j < m; j++) { V[i][j] = i == j; if (j > i) Cm[i][j] = Cm[j][i] = 0.5 * (Cm[i][j] + Cm[j][i]); }
    for (int sweep = 0; sweep < 64; sweep++) {
        double off = 0.0, diag = 0.0;
        for (int i = 0; i < m; i++) { diag += Cm[i][i] * Cm[i][i]; for (int j = i + 1; j < m; j++) off += Cm[i][j] * Cm[i][j]; }
        if (off <= 1e-36 * diag) break;
        for (int p = 0; p < m; p++)
            for (int q = p + 1; q < m; q++) {
                if (Cm[p][q] == 0.0) continue;
                const double th = (Cm[q][q] - Cm[p][p]) / (2.0 * Cm[p][q]);
                const double t = (th >= 0 ? 1.0 : -1.0) / (std::fabs(th) + std::sqrt(th * th + 1.0));
                const double cs = 1.0 / std::sqrt(t * t + 1.0), sn = t * cs;
                for (int k = 0; k < m; k++) {                 // Cm <- J^T Cm J, V <- V J
                    const double a = Cm[k][p], b = Cm[k][q];
                    Cm[k][p] = cs * a - sn * b; Cm[k][q] = sn * a + cs * b;
                }
                for (int k = 0; k < m; k++) {
                    const double a = Cm[p][k], b = Cm[q][k];
                    Cm[p][k] = cs * a - sn * b; Cm[q][k] = sn * a + cs * b;
                }
                for (int k = 0; k < m; k++) {
                    const double a = V[k][p], b = V[k][q];
                    V[k][p] = cs * a - sn * b; V[k][q] = sn * a + cs * b;
                }
            }
    }
    int top = 0;
    for (int i = 1; i < m; i++) if (Cm[i][i] > Cm[top][top]) top = i;
    mu = Cm[top][top];
    double y[3] = { 0, 0, 0 };
    for (int i = m - 1; i >= 0; i--) {                    // L^T y = V[:, top]
        double s = V[i][top];
        for (int q = i + 1; q < m; q++) s -= L[q][i] * y[q];
        y[i] = s / L[i][i];
    }
    const double sg = y[0] < 0.0 ? -1.0 : 1.0;
    for (int i = 0; i < 3; i++) c[i] = i < m ? sg * y[i] * d[i] : 0.0;
    return m;
}

struct CapOut { double *out3; int32_t *iters; double *value, *value_sum; };
// sets [s0, s0 + nb) of one batch in the call's arena; every output row of the batch is written
template <typename R>
static int capacity_batch(mp_engine *h, unsigned char *arena, const size_t *o, int nbmax, const mp_params *par, int s0, int nb,
                          double rtol, int max_iter, bool cull, const std::vector<int> &perm, const CapOut &out)
{
    const int n = h->cfg.n_patches, npad = cap_npad(n), nchunk = (n + CAP_CHUNK - 1) / CAP_CHUNK;
    CapSet *d_cs = (CapSet *)(arena + o[4]);
    double *vec = (double *)(arena + o[3]), *part = (double *)(arena + o[7]);
    unsigned *bound = (unsigned *)(arena + o[6]);
    CapArgs<R> a;
    a.ls = view<R>(h); a.cs = d_cs; a.lx = (const R *)(arena + o[0]); a.ly = (const R *)(arena + o[1]); a.hs = (const R *)(arena + o[2]);
    a.vec = vec; a.box32 = (const float4 *)h->d_tile_box; a.bound = bound; a.stats = h->d_work; a.npad = npad;
    // the arena of the previous batch: vectors and bounds start from zero (p, Ap, padding), then the batch's constants
    CK(cudaMemsetAsync(vec, 0, (size_t)nbmax * CAP_NVEC * npad * 8, h->stream));
    CK(cudaMemsetAsync(bound, 0, (size_t)nbmax * 4, h->stream));
    std::vector<double> b(nb);
    std::vector<CapSet> cs(nb);
    for (int i = 0; i < nb; i++) {
        const mp_params &p = par[s0 + i];
        b[i] = p.b;
        cs[i] = CapSet{ p.alpha, 1.0, 0.0, 0.0, 0.0, -INFINITY, (float)(std::max(p.b * std::log2(h->area_max), p.b * std::log2(h->area_min)) + 1e-3), i, 0 };
    }
    CK(cudaMemcpyAsync(arena + o[5], b.data(), nb * 8, cudaMemcpyHostToDevice, h->stream));
    k_cap_prep<R><<<dim3((npad + 255) / 256, nb), 256, 0, h->stream>>>(a.ls, h->d_perm, h->have_area ? h->d_area : nullptr,
                                                                        (const uint8_t *)(arena + o[8]), (const double *)(arena + o[5]),
                                                                        npad, (R *)(arena + o[0]), (R *)(arena + o[1]), (R *)(arena + o[2]), vec);
    CK(cudaGetLastError());
    std::vector<CapSet> up;                               // the active sets of a launch, in batch order
    std::vector<double> hp;
    auto launch_mv = [&](bool culled, int vin, int vout) -> int {
        const dim3 grid(npad / CAP_NT, (unsigned)up.size());
        constexpr bool CAN = sizeof(R) == 4;              // the FP64 engine never culls
        const bool cl = CAN && culled;
#define MV(G) do { if (cl) k_cap_mv<R, G, CAN><<<grid, CAP_NT, 0, h->stream>>>(a, vin, vout); \
                    else k_cap_mv<R, G, false><<<grid, CAP_NT, 0, h->stream>>>(a, vin, vout); } while (0)
        switch (h->geom) {
        case MP_GEOM_LINEAR: MV(MP_GEOM_LINEAR); break;
        case MP_GEOM_COORDS: MV(MP_GEOM_COORDS); break;
        default: k_cap_mv<R, MP_GEOM_DENSE, false><<<grid, CAP_NT, 0, h->stream>>>(a, vin, vout); break;
        }
#undef MV
        CK(cudaGetLastError());
        return MP_OK;
    };
    auto upload = [&]() -> int {
        CK(cudaMemcpyAsync(d_cs, up.data(), up.size() * sizeof(CapSet), cudaMemcpyHostToDevice, h->stream));
        return MP_OK;
    };
    // k_cap_update (gram = false) or k_cap_gram over the sets in `up`; hp[i * K + j]: sum j of up[i], chunks added in order
    auto reduce = [&](bool gram) -> int {
        const int K = gram ? CAP_NGRAM : 3;
        const dim3 grid(nchunk, (unsigned)up.size());
        if (gram) k_cap_gram<<<grid, CAP_RT, 0, h->stream>>>(d_cs, vec, n, npad, part);
        else k_cap_update<<<grid, CAP_RT, 0, h->stream>>>(d_cs, vec, n, npad, part);
        CK(cudaGetLastError());
        std::vector<double> raw(up.size() * nchunk * K);
        CK(cudaMemcpyAsync(raw.data(), part, raw.size() * 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        hp.assign(up.size() * K, 0.0);
        for (size_t i = 0; i < up.size(); i++)
            for (int ch = 0; ch < nchunk; ch++)
                for (int j = 0; j < K; j++) hp[i * K + j] += raw[(i * nchunk + ch) * K + j];
        return MP_OK;
    };
    int rc;
    // start: x = 1 on the kept patches, Ax by an unculled product; theta0 = its Rayleigh quotient sets the culling floor
    // tau = 2^-30 theta0 / N (DESIGN.md §5), then Ax again under the floor and r = Ax - theta0 x
    std::vector<double> theta(nb), res(nb);
    std::vector<int> iters(nb, 0);
    std::vector<char> has_p(nb, 0);
    up = cs;
    if ((rc = upload()) != MP_OK || (rc = launch_mv(false, CAP_X, CAP_AX)) != MP_OK || (rc = reduce(false)) != MP_OK) return rc;
    for (int i = 0; i < nb; i++) {
        theta[i] = hp[i * 3 + 1] / hp[i * 3];
        cs[i].mu = theta[i];
        if (cull && theta[i] > 0.0) cs[i].thr = (float)(CONN_CULL_LOG2 + std::log2(theta[i] / n)) - cs[i].lamax;
    }
    up = cs;
    if ((rc = upload()) != MP_OK) return rc;
    if (cull && (rc = launch_mv(true, CAP_X, CAP_AX)) != MP_OK) return rc;
    if ((rc = reduce(false)) != MP_OK) return rc;
    std::vector<int> act;
    for (int i = 0; i < nb; i++) {
        res[i] = std::sqrt(hp[i * 3 + 2] / hp[i * 3]) / theta[i];
        if (!(res[i] <= rtol)) act.push_back(i);
    }
    for (int it = 1; it <= max_iter && !act.empty(); it++) {
        up.clear();
        for (int i : act) up.push_back(cs[i]);
        if ((rc = upload()) != MP_OK || (rc = launch_mv(cull, CAP_R, CAP_AR)) != MP_OK || (rc = reduce(true)) != MP_OK) return rc;
        for (size_t j = 0; j < act.size(); j++) {
            CapSet &c = cs[act[j]];
            double co[3], mu;
            const int m = cap_ritz(&hp[j * CAP_NGRAM], has_p[act[j]] != 0, co, mu);
            c.cx = co[0]; c.cr = co[1]; c.cp = co[2]; c.mu = mu;
            has_p[act[j]] = m >= 2;
            up[j] = c;
        }
        if ((rc = upload()) != MP_OK || (rc = reduce(false)) != MP_OK) return rc;
        std::vector<int> next;
        for (size_t j = 0; j < act.size(); j++) {
            const int i = act[j];
            const double xx = hp[j * 3], th = hp[j * 3 + 1] / xx;
            iters[i] = it;
            res[i] = std::sqrt(hp[j * 3 + 2] / xx) / th;
            if (!(res[i] <= rtol)) next.push_back(i);
        }
        act.swap(next);
    }
    // report: a fresh product of every returned x, its Rayleigh quotient and residual
    for (int i = 0; i < nb; i++) { cs[i].cx = 1.0; cs[i].cr = cs[i].cp = 0.0; cs[i].mu = 0.0; }
    up = cs;
    if ((rc = upload()) != MP_OK || (rc = launch_mv(cull, CAP_X, CAP_AX)) != MP_OK || (rc = reduce(false)) != MP_OK) return rc;
    std::vector<double> xx(nb);
    for (int i = 0; i < nb; i++) { xx[i] = hp[i * 3]; theta[i] = hp[i * 3 + 1] / xx[i]; cs[i].mu = theta[i]; }
    up = cs;
    if ((rc = upload()) != MP_OK || (rc = reduce(false)) != MP_OK) return rc;
    std::vector<unsigned> bits(nb);
    CK(cudaMemcpyAsync(bits.data(), bound, nb * 4, cudaMemcpyDeviceToHost, h->stream));
    std::vector<double> x;
    if (out.value || out.value_sum) {
        x.resize((size_t)nb * npad);
        for (int i = 0; i < nb; i++)
            CK(cudaMemcpyAsync(&x[(size_t)i * npad], vec + ((size_t)i * CAP_NVEC + CAP_X) * npad, (size_t)npad * 8, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < nb; i++) {
        float bf;
        std::memcpy(&bf, &bits[i], 4);
        double *o3 = out.out3 + (size_t)(s0 + i) * 3;
        o3[0] = theta[i];
        o3[1] = std::sqrt(hp[i * 3 + 2] / xx[i]) / theta[i];
        o3[2] = (double)bf / theta[i];
        if (out.iters) out.iters[s0 + i] = iters[i];
        for (int s = 0; s < n && !x.empty(); s++) {
            const double v = x[(size_t)i * npad + s] * x[(size_t)i * npad + s] / xx[i];
            if (out.value) out.value[(size_t)(s0 + i) * n + perm[s]] = v;
            if (out.value_sum) out.value_sum[perm[s]] += v;
        }
    }
    return MP_OK;
}

extern "C" {
int mp_capacity(mp_engine *h, int nsets, const mp_params *par, const uint8_t *keep, double rtol, int max_iter, double *out3,
                int32_t *iters_out, double *value_out, double *value_sum)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    REQUIRE(out3, MP_ERR_ARG, "mp_capacity: out3 is required");
    REQUIRE(nsets >= 1 && rtol > 0.0 && max_iter >= 1, MP_ERR_ARG, "mp_capacity: need nsets >= 1, rtol > 0 and max_iter >= 1");
    REQUIRE(h->have_landscape, MP_ERR_STATE, "mp_capacity: landscape not set");
    REQUIRE(par || h->have_params, MP_ERR_STATE, "mp_capacity: par = NULL reads the chains' parameters, and none are set");
    REQUIRE(par || nsets == h->cfg.n_chains, MP_ERR_ARG, "mp_capacity: par = NULL needs nsets = n_chains");
    const int n = h->cfg.n_patches;
    std::vector<mp_params> pv;
    if (!par) {
        pv.resize(nC(h));
        CK(cudaMemcpyAsync(pv.data(), h->d_par, nC(h) * sizeof(mp_params), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        par = pv.data();
    }
    for (int s = 0; s < nsets; s++) REQUIRE(par[s].alpha > 0.0, MP_ERR_ARG, "mp_capacity: every set needs alpha > 0");
    int nkeep = n;
    if (keep) { nkeep = 0; for (int k = 0; k < n; k++) nkeep += keep[k] != 0; }
    REQUIRE(nkeep >= 2, MP_ERR_ARG, "mp_capacity: need at least 2 kept patches");
    Timed tm(h, MP_K_SIM);
    const size_t npad = (size_t)cap_npad(n), R = rsz(h), nchunk = (n + CAP_CHUNK - 1) / CAP_CHUNK;
    // one arena per call, reused by the batches of at most ~1 GB: positions, area constants, vectors, b, launch records, bounds,
    // reduction partials, keep, symmetry flag
    const size_t per_set = npad * (R + CAP_NVEC * 8) + 8 + sizeof(CapSet) + 4 + nchunk * CAP_NGRAM * 8 + 4 * 256;
    const int nbmax = (int)std::max<size_t>(1, std::min<size_t>({ (size_t)nsets, ((size_t)1 << 30) / per_set, 65535 }));
    size_t off = 0, o[10];
    auto carve = [&](size_t bytes) { const size_t r = off; off += (bytes + 255) / 256 * 256; return r; };
    o[0] = carve(npad * R); o[1] = carve(npad * R); o[2] = carve(nbmax * npad * R); o[3] = carve(nbmax * CAP_NVEC * npad * 8);
    o[4] = carve(nbmax * sizeof(CapSet)); o[5] = carve(nbmax * 8); o[6] = carve(nbmax * 4); o[7] = carve(nbmax * nchunk * CAP_NGRAM * 8);
    o[8] = carve(n); o[9] = carve(4);
    unsigned char *arena = nullptr;
    int rc = MP_OK;
    cudaError_t e;
#define CAPCK(call) if ((e = (call)) != cudaSuccess) { h->err = std::string(#call) + ": " + cudaGetErrorString(e); rc = MP_ERR_CUDA; goto done; }
    CAPCK(cudaMalloc(&arena, off));
    {
        std::vector<uint8_t> kp(n, 1);
        if (keep) for (int k = 0; k < n; k++) kp[k] = keep[k] != 0;
        CAPCK(cudaMemcpyAsync(arena + o[8], kp.data(), n, cudaMemcpyHostToDevice, h->stream));
        if (h->geom == MP_GEOM_DENSE) {                   // M~ is symmetric only for a symmetric distance matrix
            int *flag = (int *)(arena + o[9]), hf = 0;
            CAPCK(cudaMemsetAsync(flag, 0, 4, h->stream));
            const dim3 grid((n + 255) / 256, std::min(n, 65535));
            if (is64(h)) k_cap_symcheck<double><<<grid, 256, 0, h->stream>>>((const double *)h->d_dist, n, flag);
            else k_cap_symcheck<float><<<grid, 256, 0, h->stream>>>((const float *)h->d_dist, n, flag);
            CAPCK(cudaGetLastError());
            CAPCK(cudaMemcpyAsync(&hf, flag, 4, cudaMemcpyDeviceToHost, h->stream));
            CAPCK(cudaStreamSynchronize(h->stream));
            if (hf) { h->err = "mp_capacity: the distance matrix is not symmetric"; rc = MP_ERR_UNSUPPORTED; goto done; }
        }
        std::vector<int> perm(n);
        CAPCK(cudaMemcpyAsync(perm.data(), h->d_perm, n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CAPCK(cudaStreamSynchronize(h->stream));
        if (value_sum) std::fill(value_sum, value_sum + n, 0.0);
        const bool cull = !is64(h) && h->geom != MP_GEOM_DENSE && h->conn_cull && h->have_boxes;
        const CapOut out{ out3, iters_out, value_out, value_sum };
        for (int s0 = 0; s0 < nsets && rc == MP_OK; s0 += nbmax) {
            const int nb = std::min(nbmax, nsets - s0);
            rc = is64(h) ? capacity_batch<double>(h, arena, o, nbmax, par, s0, nb, rtol, max_iter, cull, perm, out)
                         : capacity_batch<float>(h, arena, o, nbmax, par, s0, nb, rtol, max_iter, cull, perm, out);
        }
    }
#undef CAPCK
done:
    cudaStreamSynchronize(h->stream);
    cudaFree(arena);
    return rc;
}

// ---- plumbing
int mp_device_ptr(mp_engine *h, int which, void **ptr, size_t *bytes)
{
    if (!h || !ptr) return MP_ERR_ARG;
    size_t b = 0; void *p = nullptr;
    switch (which) {
    case MP_BUF_DRAWS: p = h->d_draws; b = std::max<size_t>(1, (size_t)h->cfg.max_draws) * nC(h) * MP_NDRAW * 8; break;
    case MP_BUF_Z: p = h->d_z; b = nC(h) * zcells(h); break;
    case MP_BUF_Y: p = h->d_y; b = nC(h) * ycells(h); break;
    case MP_BUF_S: p = h->d_S[0]; b = nC(h) * ycells(h) * 8; break;
    case MP_BUF_S_PROP: p = h->d_S[1]; b = nC(h) * ycells(h) * 8; break;
    case MP_BUF_PARAMS: p = h->d_par; b = nC(h) * sizeof(mp_params); break;
    default: h->err = "mp_device_ptr: unknown buffer"; return MP_ERR_ARG;
    }
    *ptr = p;
    if (bytes) *bytes = b;
    return MP_OK;
}
int mp_get_stream(mp_engine *h, void **stream)
{
    if (!h || !stream) return MP_ERR_ARG;
    *stream = (void *)h->stream;
    return MP_OK;
}
int mp_set_timing(mp_engine *h, int enabled)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    drain_spans(h);
    drop_graphs(h);
    h->timing = enabled != 0;
    return MP_OK;
}
int mp_get_timing(mp_engine *h, double *ms, int64_t *launches, int reset)
{
    if (!h) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    drain_spans(h);
    for (int i = 0; i < MP_K_NCAT; i++) {
        if (ms) ms[i] = h->t_ms[i];
        if (launches) launches[i] = h->t_launch[i];
        if (reset) { h->t_ms[i] = 0.0; h->t_launch[i] = 0; }
    }
    return MP_OK;
}
int mp_get_conn_path(mp_engine *h) { return h ? h->last_conn_path : MP_ERR_ARG; }
int mp_get_scan_geometry(mp_engine *h, int *out4)
{
    if (!h || !out4) return MP_ERR_ARG;
    for (int i = 0; i < 4; i++) out4[i] = h->last_scan[i];
    return MP_OK;
}
int mp_get_work_counters(mp_engine *h, uint64_t *out, int reset)
{
    if (!h || !out) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    unsigned long long dev[MP_CNT_N];
    CK(cudaMemcpyAsync(dev, h->d_work, sizeof(dev), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < MP_CNT_N; i++) out[i] = (uint64_t)dev[i];
    if (reset) CK(cudaMemsetAsync(h->d_work, 0, sizeof(dev), h->stream));
    return MP_OK;
}
int mp_probe_peaks(mp_engine *h, double *out4)
{
    if (!h || !out4) return MP_ERR_ARG;
    CK(cudaSetDevice(h->cfg.device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, h->cfg.device));
    const int nsm = prop.multiProcessorCount, blocks = nsm * 4, thr = 512, iters = 4096;
    float *d_f = nullptr; double *d_d = nullptr;
    CK(cudaMalloc(&d_f, 64)); CK(cudaMalloc(&d_d, 64));
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    auto timeit = [&](auto launch) -> double {
        launch(); cudaStreamSynchronize(h->stream);
        double best = 1e30;
        for (int r = 0; r < 5; r++) {
            cudaEventRecord(a, h->stream); launch(); cudaEventRecord(b, h->stream); cudaEventSynchronize(b);
            float ms = 0.f; cudaEventElapsedTime(&ms, a, b);
            best = std::min(best, (double)ms);
        }
        return best * 1e-3;
    };
    const double work = (double)blocks * thr * iters;
    double s = timeit([&] { k_probe_mufu<<<blocks, thr, 0, h->stream>>>(d_f, iters); });
    out4[0] = work * 4 / s * 1e-9;
    s = timeit([&] { k_probe_ffma<<<blocks, thr, 0, h->stream>>>(d_f, iters); });
    out4[1] = work * 8 / s * 1e-9;
    s = timeit([&] { k_probe_dadd<<<blocks, thr, 0, h->stream>>>(d_d, iters); });
    out4[2] = work * 8 / s * 1e-9;
    const size_t bytes = (size_t)1 << 30;
    float4 *src = nullptr, *dst = nullptr;
    CK(cudaMalloc(&src, bytes)); CK(cudaMalloc(&dst, bytes));
    CK(cudaMemsetAsync(src, 1, bytes, h->stream));
    s = timeit([&] { k_probe_copy<<<nsm * 16, 512, 0, h->stream>>>(src, dst, bytes / 16); });
    out4[3] = 2.0 * (double)bytes / s * 1e-9;
    cudaFree(src); cudaFree(dst); cudaFree(d_f); cudaFree(d_d);
    cudaEventDestroy(a); cudaEventDestroy(b);
    CK(cudaGetLastError());
    return MP_OK;
}

}  // extern "C"
