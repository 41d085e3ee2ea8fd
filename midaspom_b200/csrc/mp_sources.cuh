// mp_sources.cuh -- attribution of every colonisation to its source patches during sweeps (mp_set_sources; DESIGN §2).
//
// For a sample (chain c after a qualifying sweep) and transition t, an event is a target k with y_tk = 0 and z_{t+1,k} = 1.
// With the pressure P_tk = K_t S_tk + Ksrc_t g_k (the resident S, FP64), source l (y_tl = 1) takes the share
// rho_tkl = K_t w(k<-l) / P_tk of the event and the external source the share Ksrc_t g_k / P_tk; an event with P_tk = 0 is
// counted as unattributed.
//
//  k_src_lists     one CTA per (transition, chain): the attributed events {position or index, u = K_t / P} and the sources
//                  {position or index, area constant} compacted in layout order (perm), the event counts and the external share
//  k_src_contract  grid (source tiles, transition, chain): each thread owns one compacted source and adds sum_k w(k<-l) u_k in
//                  FP64 over the event list in its fixed order, with pair_weight -- the weight k_conn adds into S, so the shares
//                  of an event sum to 1 against the resident S.  Optionally a fixed-point histogram of rho over the distance bins.
//  k_src_finish    adds the per-sample arrays into the sums, chains in order
//
// Every kernel returns at once unless the sweep qualifies (sweep_due on the device counter), so captured sweeps replay
// unchanged.  No floating-point atomics: the sums are bit-identical whatever the launch geometry.
#pragma once
#include "mp_kernels.cuh"   // sweep_due, SrcRec (mp_conn.cuh)

namespace mp {

constexpr int SRC_LIST_THREADS = 256;
constexpr int SRC_TILE = 128;                        // sources per CTA of k_src_contract = events per shared-memory tile
constexpr double SRC_HIST_ONE = 1099511627776.0;     // 2^40: fixed-point unit of the per-sample histogram
constexpr int SRC_MAX_BINS = 4096;

// event record: position (landscapes with positions) or patch index, and u = K_t / P_tk in FP64.  16 B (FP32), 32 B (FP64).
// Source records are SrcRec<R> {x, y, area constant, patch index}.
template <typename R> struct EvtRec;
template <> struct __align__(16) EvtRec<float> { union { float x; int k; }; float y; double u; };
template <> struct __align__(16) EvtRec<double> { union { double x; int k; }; double y, u, pad; };

struct SrcBufs {
    void *evt, *src;                 // [chain][transition][N] records; the first n_attr / n_src of a row are valid
    double *stage;                   // [chain][transition][N] sum_k rho_tkl of the sample at the patch's index (0: no source)
    double *ct_ext;                  // [chain][transition] sum_k rho_tk,ext of the sample
    uint32_t *ct_cnt;                // [chain][transition][4]: events, unattributed, attributed (event list), sources
    unsigned long long *hist_i;      // [transition][nbins] histogram of the sample in units of 2^-40 (zero between samples)
    double *src_sum, *ext_sum, *dist_hist;   // the sums: [transition][N], [transition], [transition][nbins]
    unsigned long long *events;      // [2][transition]: events, unattributed
    unsigned long long *nsamples;
    int nbins;
    double bin_width;
};

template <typename R>
__global__ void __launch_bounds__(SRC_LIST_THREADS)
k_src_lists(const uint32_t *__restrict__ sweep_p /* device-resident sweep counter (k_advance) */, int first, int thin, Landscape<R> ls,
            int coords, const int *__restrict__ perm, const mp_params *__restrict__ par, const uint8_t *__restrict__ era,
            const R *__restrict__ aw, const uint8_t *__restrict__ z, const uint8_t *__restrict__ y, const double *__restrict__ S,
            int T, SrcBufs b)
{
    if (!sweep_due(*sweep_p, first, thin)) return;
    __shared__ double scratch[32];
    __shared__ int wcnt[2][SRC_LIST_THREADS / 32];
    const int n = ls.n, t = blockIdx.x, c = blockIdx.y, ntrans = T - 1, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const size_t ct = (size_t)c * ntrans + t, row = ct * n;
    const uint8_t *yr = y + row, *zr = z + ((size_t)c * T + t + 1) * n;
    const double *Sr = S + row;
    const R *awc = aw + (size_t)c * n;
    const Trans<R> tr = make_trans<R>(par[c], era ? era[t] : 0);
    const double Kt = (double)tr.Kt, Ks = (double)tr.Ks;
    EvtRec<R> *evt = (EvtRec<R> *)b.evt + row;
    SrcRec<R> *src = (SrcRec<R> *)b.src + row;
    double *stage = b.stage + row;
    int nsrc = 0, nattr = 0;                                  // list lengths so far (block-uniform)
    double nev = 0.0, nun = 0.0, ext = 0.0;                   // this thread's events, unattributed events, external share
    const uint32_t below = (1u << lane) - 1u;
    for (int s0 = 0; s0 < n; s0 += SRC_LIST_THREADS) {
        const int s = s0 + tid;
        bool is_src = false, is_evt = false;
        int q = 0;
        double u = 0.0;
        if (s < n) {
            q = perm[s];
            is_src = yr[q] != 0;
            if (!is_src) {
                stage[q] = 0.0;
                if (zr[q]) {
                    nev += 1.0;
                    const double g = (double)source_term<R>(ls, tr, q);
                    const double P = Kt * Sr[q] + Ks * g;
                    if (P > 0.0) { is_evt = true; u = Kt / P; ext += Ks * g / P; }
                    else nun += 1.0;
                }
            }
        }
        const uint32_t ms = __ballot_sync(0xffffffffu, is_src), me = __ballot_sync(0xffffffffu, is_evt);
        if (lane == 0) { wcnt[0][wid] = __popc(ms); wcnt[1][wid] = __popc(me); }
        __syncthreads();
        int os = nsrc, oe = nattr;
#pragma unroll
        for (int w = 0; w < SRC_LIST_THREADS / 32; w++) {
            if (w < wid) { os += wcnt[0][w]; oe += wcnt[1][w]; }
            nsrc += wcnt[0][w]; nattr += wcnt[1][w];
        }
        if (is_src) {
            SrcRec<R> r;
            r.x = coords ? ls.px[q] : (R)0; r.y = coords ? ls.py[q] : (R)0; r.aw = awc[q]; r.bits = (uint32_t)q;
            src[os + __popc(ms & below)] = r;
        }
        if (is_evt) {
            EvtRec<R> r;
            if (coords) r.x = ls.px[q]; else r.k = q;
            r.y = coords ? ls.py[q] : (R)0; r.u = u;
            evt[oe + __popc(me & below)] = r;
        }
        __syncthreads();                                     // wcnt is rewritten by the next round
    }
    nev = block_sum(nev, scratch);
    __syncthreads();
    nun = block_sum(nun, scratch);
    __syncthreads();
    ext = block_sum(ext, scratch);
    if (tid == 0) {
        b.ct_ext[ct] = ext;
        uint32_t *cnt = b.ct_cnt + ct * 4;
        cnt[0] = (uint32_t)nev; cnt[1] = (uint32_t)nun; cnt[2] = (uint32_t)nattr; cnt[3] = (uint32_t)nsrc;
    }
}

// HIST: bins [i w, (i + 1) w), the last one open; each pair adds round(rho 2^40) to a shared-memory histogram (pairs that round to
// 0 skip the atomic), flushed with integer atomics -- sums that do not depend on the order of the adds.  A per-sample bin holds
// at most events x chains < 2^23 (10^5 patches, 64 chains) in units of 2^-40.
template <typename R, int GEOM, bool HIST>
__global__ void __launch_bounds__(SRC_TILE)
k_src_contract(const uint32_t *__restrict__ sweep_p, int first, int thin, Landscape<R> ls, const mp_params *__restrict__ par, int T, SrcBufs b)
{
    if (!sweep_due(*sweep_p, first, thin)) return;
    __shared__ EvtRec<R> sev[SRC_TILE];
    extern __shared__ unsigned long long src_hist[];           // HIST: [nbins]
    const int n = ls.n, t = blockIdx.y, c = blockIdx.z, ntrans = T - 1, tid = threadIdx.x;
    const size_t ct = (size_t)c * ntrans + t, row = ct * n;
    const int nattr = (int)b.ct_cnt[ct * 4 + 2], nsrc = (int)b.ct_cnt[ct * 4 + 3];
    const int j0 = blockIdx.x * SRC_TILE;
    if (j0 >= nsrc) return;                                    // CTA-uniform
    if (HIST) {
        for (int i = tid; i < b.nbins; i += SRC_TILE) src_hist[i] = 0ull;
    }
    const bool own = j0 + tid < nsrc;
    R sx = (R)0, sy = (R)0, saw = (R)0;
    int l = 0;
    if (own) {
        const SrcRec<R> s = ((const SrcRec<R> *)b.src)[row + j0 + tid];
        sx = s.x; sy = s.y; saw = s.aw; l = (int)s.bits;
    }
    const R apre = alpha_pre<R>(par[c].alpha);
    const EvtRec<R> *evt = (const EvtRec<R> *)b.evt + row;
    const double last = (double)(b.nbins - 1);
    double acc = 0.0;
    for (int e0 = 0; e0 < nattr; e0 += SRC_TILE) {
        __syncthreads();                                       // the previous tile (and the zeroed histogram) are done with
        if (e0 + tid < nattr) sev[tid] = evt[e0 + tid];
        __syncthreads();
        const int m = min(SRC_TILE, nattr - e0);
        if (!own) continue;
        for (int i = 0; i < m; i++) {
            const int k = GEOM == MP_GEOM_COORDS ? 0 : sev[i].k;          // broadcast loads
            const R ex = GEOM == MP_GEOM_COORDS ? sev[i].x : (R)0, ey = GEOM == MP_GEOM_COORDS ? sev[i].y : (R)0;
            const R w = pair_weight<R, GEOM>(ls, apre, saw, k, l, ex, ey, sx, sy);
            const double rho = (double)w * sev[i].u;
            acc += rho;
            if (HIST && rho * SRC_HIST_ONE > 0.5) {
                const double q = (double)pair_distance<R, GEOM>(ls, k, l, ex, ey, sx, sy) / b.bin_width;
                const int bin = q >= last ? b.nbins - 1 : (int)q;
                atomicAdd(&src_hist[bin], (unsigned long long)llrint(rho * SRC_HIST_ONE));
            }
        }
    }
    if (own) b.stage[row + l] = acc;
    if (HIST) {
        __syncthreads();
        for (int i = tid; i < b.nbins; i += SRC_TILE)
            if (src_hist[i]) atomicAdd(&b.hist_i[(size_t)t * b.nbins + i], src_hist[i]);
    }
}

// one thread per (transition, patch) of src_sum, per (transition, bin) of the histogram and per transition of the counts
__global__ void __launch_bounds__(256)
k_src_finish(const uint32_t *__restrict__ sweep_p, int first, int thin, int n, int T, int nchains, SrcBufs b)
{
    if (!sweep_due(*sweep_p, first, thin)) return;
    const int ntrans = T - 1;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx == 0) *b.nsamples += (unsigned long long)nchains;
    if (idx < (long long)ntrans * n) {
        double v = b.src_sum[idx];
        for (int c = 0; c < nchains; c++) v += b.stage[(size_t)c * ntrans * n + idx];
        b.src_sum[idx] = v;
    }
    if (idx < (long long)ntrans * b.nbins) {
        b.dist_hist[idx] += (double)b.hist_i[idx] * (1.0 / SRC_HIST_ONE);
        b.hist_i[idx] = 0ull;
    }
    if (idx < ntrans) {
        double x = b.ext_sum[idx];
        unsigned long long ne = 0, nu = 0;
        for (int c = 0; c < nchains; c++) {
            const size_t ct = (size_t)c * ntrans + idx;
            x += b.ct_ext[ct]; ne += b.ct_cnt[ct * 4]; nu += b.ct_cnt[ct * 4 + 1];
        }
        b.ext_sum[idx] = x; b.events[idx] += ne; b.events[ntrans + idx] += nu;
    }
}

}  // namespace mp
