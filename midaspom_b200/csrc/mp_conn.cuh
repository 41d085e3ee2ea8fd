// mp_conn.cuh -- the fused on-the-fly dispersal-kernel x occupancy contraction (main_MIDASPOM.c:350-358):
//     S[chain][t][k] = sum_{l != k} A_l^b exp(-alpha d_kl) y[chain][t][l]           for every transition t at once.
//
//  k_pack_sources  one 16-byte (FP32) / 32-byte (FP64) record {x, y, area constant, year bit word} per (parameter set,
//                  chain, 32-year word, scan-order slot): the sources of k_conn as one contiguous stream
//  k_group_min_S   lower bound of S per group of 32 scan-order slots (culling bound)
//  k_conn          one thread owns TGT target patches and NYB year accumulators per target.  Source records arrive
//                  NTHR at a time through a two-stage shared-memory ring filled by the TMA engine (cp.async.bulk,
//                  completion counted on an mbarrier), so the loads of tile i+1 overlap the arithmetic of tile i; the
//                  dispersal weight is evaluated once per (target, source) pair and contracted over the years with
//                  acc[t] = fma(w, y01[t], acc[t]) (exactly acc[t] + w or acc[t]).  FP64 accumulation in both precisions so
//                  that later rank-1 removals of the same FP32 weight by the y scan cancel exactly.
//                  A32 variant (mp_conn32.cu; the evaluation entry points of the FP32 engines -- the sampler's resident S keeps
//                  the FP64 form, see launch_conn_g in mp_engine.cu): the year contraction of each group of 32 sources runs on the
//                  FP32 pipe as packed FFMA2 (fma.rn.f32x2: two years per instruction) into FP32 partial sums, which join
//                  the FP64 accumulators (in shared memory, one column per thread) after every group of 32 sources -- half
//                  the pipe time of the DFMA form and a third of its issue slots.  A partial sum rounds at 2^-24 over at most
//                  32 terms (bound 2e-6 relative; measured on the cfg3 landscape rms 3.5e-8, max 1.1e-7: far inside the FP32
//                  path's 1e-5 and below the 2^-30 culling of the same kernel); it is taken per (target, aligned group of 32
//                  sources), so the result does not depend on the launch shape or on how the targets are sharded.
#pragma once
#include <type_traits>
#include "mp_device.cuh"

namespace mp {

constexpr int CONN_BATCH = 4;      // sources whose weights are evaluated together before their year contractions
constexpr int CONN_PAD = 128;       // the record stream of a (set, chain, word) is padded to whole tiles (zero records)
constexpr int CONN_A32_GROUPS = 1;  // A32: groups of 32 sources whose FP32 partial sums are added up before they join the FP64 accumulators
                                    // (measured on the cfg3 landscape, error of S against the FP64 sum of the same weights: 1 group rms 3.5e-8 /
                                    // max 1.1e-7, 2 groups 5.6e-8 / 1.8e-7, 4 groups 8.6e-8 / 3.4e-7)
// dynamic shared memory of the A32 variant: FP64 accumulators [2 targets x NYB years][NTHR threads]
inline __host__ __device__ size_t conn_a32_smem(int nyb, int nthr) { return (size_t)2 * nyb * nthr * sizeof(double); }

template <typename R> struct SrcRec;
template <> struct __align__(16) SrcRec<float> { float x, y, aw; uint32_t bits; };
template <> struct __align__(16) SrcRec<double> { double x, y, aw; uint32_t bits, pad; };

inline __host__ __device__ int conn_npad(int n) { return (n + CONN_PAD - 1) / CONN_PAD * CONN_PAD; }

// grid (ceil(npad / 256), chains, nwords); writes the records of the parameter sets in set_mask (bit 0: resident, bit 1: proposal)
template <typename R>
__global__ void k_pack_sources(Landscape<R> ls, const int *__restrict__ perm, const R *__restrict__ aw0, const R *__restrict__ aw1,
                               const uint8_t *__restrict__ y, int ntrans, int nwords, int set_mask, SrcRec<R> *__restrict__ rec)
{
    const int n = ls.n, npad = conn_npad(n), c = blockIdx.y, w = blockIdx.z, C = gridDim.y;
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= npad) return;
    SrcRec<R> r;
    memset(&r, 0, sizeof r);
    int q = -1;
    if (s < n) {
        q = perm[s];
        if (ls.px) { r.x = ls.px[q]; r.y = ls.py[q]; }
        const uint8_t *yc = y + (size_t)c * ntrans * n;
        uint32_t bits = 0;
        const int t1 = min(32, ntrans - 32 * w);
        for (int t = 0; t < t1; t++) bits |= (uint32_t)(yc[(size_t)(32 * w + t) * n + q] != 0) << t;
        r.bits = bits;
    }
#pragma unroll
    for (int set = 0; set < 2; set++) {
        if (!((set_mask >> set) & 1)) continue;
        if (q >= 0) r.aw = (set ? aw1 : aw0)[(size_t)c * n + q];
        rec[(((size_t)set * C + c) * nwords + w) * npad + s] = r;
    }
}

template <typename R> struct ConnArgs {
    Landscape<R> ls;
    const mp_params *par[2];
    double *S[2];
    const SrcRec<R> *rec;  // [set][chain][word][npad], scan order
    int ntrans, nwords, nchains;
    int set_base;          // first parameter set of this launch (blockIdx.z counts from it)
    int k_lo, k_hi;        // target slots [k_lo, k_hi) of this launch (patch sharding over GPUs; whole range otherwise)
    const int *perm;       // scan-order slot -> patch (the identity for linear and dense landscapes)
    const float4 *box32;   // culled variant: bounding box {xmin, xmax, ymin, ymax} of every group of 32 consecutive slots
    const float *mlow;     // culled variant: [chain][group] lower bound of the group's S over all years (0 = unknown: no culling)
    float area_max, area_min;   // extremes of the patch areas (1, 1 without areas): A_l^b <= max(area_max^b, area_min^b)
    unsigned long long *stats;  // MP_CNT_CONN_* work counters
};
// Culled variant (FP32 engines, landscapes with positions): slots follow the scan (Morton) order, so groups of 32
// consecutive slots are spatially compact.  A group of 32 sources is skipped for a group of 32 targets when every weight
// between them is below 2^-30 of the smallest S the target group currently has (k_group_min_S: the resident S, any year),
// and a tile of sources is not even loaded when that holds for all of the CTA's target groups.  What is skipped is
// dominated by the sources just beyond the reach (2 pi R rho / alpha of them, a few hundred at the benchmark density),
// i.e. ~1e-7 of S -- relative to each group's own S, so isolated patches with a small S keep their accuracy.  Without a
// valid resident S (first sweep) mlow = 0 and nothing is skipped.  The decision is taken per (group of 32 targets, group
// of 32 sources): it does not depend on the launch shape, so every launch shape gives bit-identical sums.  The FP64 parity
// engine never culls.
constexpr float CONN_CULL_LOG2 = -30.f;

// min over years and over the 32 patches of a scan-order group of the resident S (culling bound of k_conn)
static __global__ void __launch_bounds__(32)
k_group_min_S(const double *__restrict__ S, const int *__restrict__ perm, int n, int ntrans, int valid, float *__restrict__ mlow)
{
    const int g = blockIdx.x, c = blockIdx.y, slot = g * 32 + threadIdx.x, ngroups = gridDim.x;
    float m = 3.0e38f;
    if (valid && slot < n) {
        const double *Sc = S + (size_t)c * ntrans * n + perm[slot];
        for (int t = 0; t < ntrans; t++) m = fminf(m, (float)Sc[(size_t)t * n]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (threadIdx.x == 0) mlow[(size_t)c * ngroups + g] = valid ? fmaxf(m * 0.999f, 0.f) : 0.f;
}

// ---- TMA bulk copy (global -> shared, completion on an mbarrier) and the mbarrier primitives it needs
__device__ __forceinline__ uint32_t conn_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void conn_mbar_init(uint32_t mbar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void conn_mbar_expect_tx(uint32_t mbar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void conn_mbar_wait(uint32_t mbar, uint32_t parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(mbar), "r"(parity), "r"(20000u) : "memory");
}
__device__ __forceinline__ void conn_bulk_load(uint32_t dst_smem, const void *src, uint32_t bytes, uint32_t mbar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst_smem), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}

// packed FP32 pairs (sm_100a FFMA2)
__device__ __forceinline__ unsigned long long conn_pack2(float lo, float hi)
{
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void conn_unpack2(unsigned long long v, float &lo, float &hi)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ void conn_ffma2(unsigned long long &acc, unsigned long long a, unsigned long long b)
{
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}

template <typename R, int GEOM, int NYB, bool CULL, int TGT, int NTHR, bool A32 = false>
__global__ void __launch_bounds__(NTHR) k_conn(ConnArgs<R> a)
{
    static_assert(!A32 || (sizeof(R) == 4 && NYB % 4 == 0), "the FP32 contraction is for FP32 engines, four years per shared-memory load");
    using YT = typename std::conditional<A32, float, double>::type;
    static_assert(CONN_PAD % NTHR == 0 && NTHR % 32 == 0, "tiles must divide the padding of the record stream");
    __shared__ __align__(128) SrcRec<R> srec[2][NTHR];                // two-stage ring of source tiles (TMA destination)
    __shared__ __align__(16) YT sy01[NTHR][NYB];                      // year bits of the current tile as 0.0 / 1.0
    __shared__ __align__(8) unsigned long long full[2];
    extern __shared__ __align__(16) unsigned char conn_dyn[];        // A32: the thread's FP64 accumulators, sacc[(g * NYB + t) * NTHR + tid]
    double *sacc = reinterpret_cast<double *>(conn_dyn) + threadIdx.x;
    const int n = a.ls.n, npad = conn_npad(n), c = blockIdx.y, set = blockIdx.z + a.set_base, tid = threadIdx.x;
    const int lane = tid & 31, wid = tid >> 5;
    const int slot0 = a.k_lo + blockIdx.x * NTHR * TGT;              // first target slot of the CTA
    const int kbase = slot0 + wid * 32 * TGT + lane;                 // the thread's targets: slots kbase, kbase + 32, ...: a warp owns TGT groups
    const mp_params *parp = set ? a.par[1] : a.par[0];
    const R apre = alpha_pre<R>(parp[c].alpha);
    double *Sout = (set ? a.S[1] : a.S[0]) + (size_t)c * a.ntrans * n;
    R tx[TGT], ty[TGT];
    int ks[TGT], kp[TGT], kq[TGT];                                   // slot and patch number of the thread's targets (-1: none); patch used in the arithmetic
#pragma unroll
    for (int g = 0; g < TGT; g++) {
        const int k = kbase + g * 32;
        ks[g] = k < a.k_hi ? k : -1;
        kp[g] = k < a.k_hi ? a.perm[k] : -1;
        kq[g] = a.perm[min(k, a.k_hi - 1)];                          // a thread without a target evaluates the last one (branch-free; never stored)
        tx[g] = 0; ty[g] = 0;
        if (GEOM == MP_GEOM_COORDS) { tx[g] = a.ls.px[kq[g]]; ty[g] = a.ls.py[kq[g]]; }
    }
    if (tid == 0) {
        conn_mbar_init(conn_smem_u32(&full[0]), 1); conn_mbar_init(conn_smem_u32(&full[1]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // boxes {xmin, xmax, ymin, ymax} of the CTA's targets and of the warp's target groups
    float4 tbox = make_float4(0.f, 0.f, 0.f, 0.f), gbox[TGT];
    auto box_union = [](const float4 &p, const float4 &q) { return make_float4(fminf(p.x, q.x), fmaxf(p.y, q.y), fminf(p.z, q.z), fmaxf(p.w, q.w)); };
    // log2 of the largest distance factor exp(-alpha d) between two boxes (apre = -alpha log2 e), with a rounding margin
    auto reach_log2 = [&](const float4 &p, const float4 &q) {
        const float dx = fmaxf(0.f, fmaxf(q.x - p.y, p.x - q.y)), dy = fmaxf(0.f, fmaxf(q.z - p.w, p.z - q.w));
        return (float)apre * (0.9999f * sqrtf(dx * dx + dy * dy));
    };
    // skip when log2(exp(-alpha d)) < thr: thr = CONN_CULL_LOG2 + log2(mlow / max_l A_l^b) of the target group(s); -inf = never
    float thr_cta = 0.f, thr[TGT];
    const int gend = (a.k_hi + 31) / 32;
    if (CULL) {
        const int g0 = slot0 / 32, ngroups = (n + 31) / 32;
        const float b = (float)parp[c].b;
        const float law_max = fmaxf(b * log2f(a.area_max), b * log2f(a.area_min)) + 1e-3f;     // log2 of max_l A_l^b, rounded up
        // mlow bounds the resident S, which belongs to the current parameters (set 0).  For the proposal (set 1) it becomes a
        // bound of S' through w' = w^p A^(b' - p b) with p = alpha' / alpha: S' >= A^(b' - p b)_min S^p for p <= 1, since
        // (sum w)^p <= sum w^p, and S' >= A^(b' - p b)_min n^(1 - p) S^p for p > 1 (power means over the n <= N sources).
        // Without it a proposal with a larger alpha would be culled at 2^-30 of the current S rather than of its own.
        float lscale = 1.f, loff = 0.f;
        if (set == 1 && (parp[c].alpha != a.par[0][c].alpha || parp[c].b != a.par[0][c].b)) {
            const double p = parp[c].alpha / a.par[0][c].alpha;
            const float db = (float)(parp[c].b - p * a.par[0][c].b);
            lscale = (float)p;
            loff = fminf(db * log2f(a.area_max), db * log2f(a.area_min)) - (p > 1.0 ? (float)(p - 1.0) * log2f((float)n) : 0.f) - 1e-3f;
        }
        auto thr_of = [&](int g) { return CONN_CULL_LOG2 + lscale * log2f(a.mlow[(size_t)c * ngroups + g]) + loff - law_max; };   // log2f(0) = -inf
        tbox = a.box32[g0]; thr_cta = thr_of(g0);
        for (int i = 1; i < NTHR * TGT / 32; i++)
            if (g0 + i < gend) { tbox = box_union(tbox, a.box32[g0 + i]); thr_cta = fminf(thr_cta, thr_of(g0 + i)); }
        const int w0 = g0 + wid * TGT;
#pragma unroll
        for (int g = 0; g < TGT; g++) { gbox[g] = a.box32[min(w0 + g, gend - 1)]; thr[g] = thr_of(min(w0 + g, gend - 1)); }   // the warp's g-th group
    }
    const int ntile = (n + NTHR - 1) / NTHR;
    // first tile >= i with a (target, source) pair within reach of the CTA (CTA-uniform).  The tiles are tested 32 at a time, one
    // per lane (every warp does the same test and holds the same mask): one round of box loads per 32 tiles instead of a
    // dependent load per tile -- on wide landscapes most tiles are out of reach (97 % at cfg5) and the scan over them is latency.
    uint32_t tmask = 0u;                                             // in-reach tiles of the chunk of 32 tiles at hand
    int tchunk = -1;
    auto next_tile = [&](int i) {
        if (!CULL) return i;
        while (i < ntile) {
            const int ch = i >> 5;
            if (ch != tchunk) {
                const int ti = ch * 32 + lane;
                bool in = false;
                if (ti < ntile) {
                    float4 sb = a.box32[ti * (NTHR / 32)];
                    for (int u = 1; u < NTHR / 32; u++) if (ti * NTHR + 32 * u < n) sb = box_union(sb, a.box32[ti * (NTHR / 32) + u]);
                    in = !(reach_log2(tbox, sb) < thr_cta);
                }
                tmask = __ballot_sync(0xffffffffu, in);
                tchunk = ch;
            }
            const uint32_t m = tmask >> (i & 31);
            if (m) return i + __ffs((int)m) - 1;
            i = (ch + 1) * 32;
        }
        return i;
    };
    const bool warp_live = slot0 + wid * 32 * TGT < a.k_hi;          // the warp has at least one target
    bool gvalid[TGT];                                                // the warp's g-th target group lies inside the launch's range
#pragma unroll
    for (int g = 0; g < TGT; g++) gvalid[g] = slot0 + (wid * TGT + g) * 32 < a.k_hi;
    uint32_t nexec = 0;                                              // (target group, source group) tiles evaluated by this warp
    uint32_t phase = 0u;                                             // bit s: parity the next wait on stage s expects
    int stage = 0;
    for (int w = 0; w < a.nwords; w++) {
        const SrcRec<R> *rw = a.rec + (((size_t)set * a.nchains + c) * a.nwords + w) * npad;
        auto issue = [&](int tile, int st) {                         // thread 0: one bulk copy of a whole tile of records
            const uint32_t bar = conn_smem_u32(&full[st]);
            conn_mbar_expect_tx(bar, (uint32_t)(NTHR * sizeof(SrcRec<R>)));
            conn_bulk_load(conn_smem_u32(&srec[st][0]), rw + (size_t)tile * NTHR, (uint32_t)(NTHR * sizeof(SrcRec<R>)), bar);
        };
        double acc[A32 ? 1 : TGT][A32 ? 1 : NYB];
#pragma unroll
        for (int g = 0; g < (A32 ? 1 : TGT); g++)
#pragma unroll
            for (int t = 0; t < (A32 ? 1 : NYB); t++) acc[g][t] = 0.0;
        // A32: FP32 partial sums of the sources at hand, two years per register pair; the FP64 accumulators live in shared memory
        unsigned long long part[A32 ? TGT : 1][A32 ? NYB / 2 : 1];
#pragma unroll
        for (int g = 0; g < (A32 ? TGT : 1); g++)
#pragma unroll
            for (int t = 0; t < (A32 ? NYB / 2 : 1); t++) part[g][t] = 0ull;
        if constexpr (A32) {
#pragma unroll
            for (int i = 0; i < TGT * NYB; i++) sacc[i * NTHR] = 0.0;
        }
        int pend = -1;                                               // A32: aligned source group the partial sums belong to (-1: none pending)
        auto flush = [&]() {
            if constexpr (A32) {
#pragma unroll
                for (int g = 0; g < TGT; g++)
#pragma unroll
                    for (int t2 = 0; t2 < NYB / 2; t2++) {
                        float lo, hi;
                        conn_unpack2(part[g][t2], lo, hi);
                        sacc[(g * NYB + 2 * t2) * NTHR] += (double)lo; sacc[(g * NYB + 2 * t2 + 1) * NTHR] += (double)hi;
                        part[g][t2] = 0ull;
                    }
            }
        };
        bool far[TGT];                                               // culled variant: group g is out of reach of the 32 sources at hand
#pragma unroll
        for (int g = 0; g < TGT; g++) far[g] = false;
        int cur = next_tile(0);
        if (tid == 0 && cur < ntile) issue(cur, stage);
        while (cur < ntile) {
            const int nxt = next_tile(cur + 1);
            if (tid == 0 && nxt < ntile) issue(nxt, stage ^ 1);      // the other stage was released by the barrier that ended the previous tile
            conn_mbar_wait(conn_smem_u32(&full[stage]), (phase >> stage) & 1u);
            phase ^= 1u << stage;
            const SrcRec<R> *sr = srec[stage];
            {
                const uint32_t bits = sr[tid].bits;
#pragma unroll
                for (int t = 0; t < NYB; t++) sy01[tid][t] = (bits >> t) & 1u ? YT(1) : YT(0);
            }
            __syncthreads();
            const int l0 = cur * NTHR;
            // CONN_BATCH sources at a time: first all their weights (independent SQRT / EX2 chains that overlap), then the
            // year contraction of each -- the weight latency is paid once per batch, not once per source
            auto batch = [&](int j0, auto SPECIAL) {
                // SPECIAL: some weight of this group of 32 sources is forced to zero (the target itself, a target group out
                // of reach); otherwise the test is not even evaluated (A32; the FP64 form always evaluates it)
                constexpr bool special = decltype(SPECIAL)::value;
                if constexpr (A32) {
                    float wf[CONN_BATCH][TGT];
#pragma unroll
                    for (int u = 0; u < CONN_BATCH; u++) {
                        const SrcRec<R> s = sr[j0 + u];              // broadcast LDS.128
                        const int lj = l0 + j0 + u;
#pragma unroll
                        for (int g = 0; g < TGT; g++) {
                            float wgt = pair_weight<R, GEOM>(a.ls, apre, s.aw, kq[g], lj, tx[g], ty[g], s.x, s.y);
                            if (special && (lj == ks[g] || (CULL && far[g]))) wgt = 0.f;
                            wf[u][g] = wgt;
                        }
                    }
#pragma unroll
                    for (int u = 0; u < CONN_BATCH; u++) {
                        const ulonglong2 *yb = reinterpret_cast<const ulonglong2 *>(&sy01[j0 + u][0]);
                        unsigned long long ww[TGT];
#pragma unroll
                        for (int g = 0; g < TGT; g++) ww[g] = conn_pack2(wf[u][g], wf[u][g]);
#pragma unroll
                        for (int t4 = 0; t4 < NYB / 4; t4++) {
                            const ulonglong2 m = yb[t4];             // four years of this source
#pragma unroll
                            for (int g = 0; g < TGT; g++) {
                                conn_ffma2(part[g][2 * t4], ww[g], m.x);
                                conn_ffma2(part[g][2 * t4 + 1], ww[g], m.y);
                            }
                        }
                    }
                } else {
                    double wd[CONN_BATCH][TGT];
#pragma unroll
                    for (int u = 0; u < CONN_BATCH; u++) {
                        const SrcRec<R> s = sr[j0 + u];              // broadcast LDS.128
                        const int lj = l0 + j0 + u;                  // slot of the source (== patch number without coordinates)
#pragma unroll
                        for (int g = 0; g < TGT; g++) {
                            R wgt = pair_weight<R, GEOM>(a.ls, apre, s.aw, kq[g], lj, tx[g], ty[g], s.x, s.y);
                            if (lj == ks[g] || (CULL && far[g])) wgt = 0;    // l != k  (main_MIDASPOM.c:354)
                            wd[u][g] = (double)wgt;
                        }
                    }
#pragma unroll
                    for (int u = 0; u < CONN_BATCH; u++) {
                        const double2 *yb = reinterpret_cast<const double2 *>(&sy01[j0 + u][0]);
#pragma unroll
                        for (int t2 = 0; t2 < NYB / 2; t2++) {
                            const double2 m = yb[t2];
#pragma unroll
                            for (int g = 0; g < TGT; g++) {
                                acc[g][2 * t2] = fma(wd[u][g], m.x, acc[g][2 * t2]);
                                acc[g][2 * t2 + 1] = fma(wd[u][g], m.y, acc[g][2 * t2 + 1]);
                            }
                        }
                    }
                }
            };
            if (warp_live) {
                float4 sbox[NTHR / 32];                              // boxes of the tile's source groups: independent loads, one latency
                if (CULL) {
#pragma unroll
                    for (int sub = 0; sub < NTHR / 32; sub++) sbox[sub] = a.box32[min(l0 / 32 + sub, (n + 31) / 32 - 1)];
                }
#pragma unroll
                for (int sub = 0; sub < NTHR / 32; sub++) {          // warp-uniform: 32 sources against the warp's TGT target groups
                    if (l0 + 32 * sub >= n) continue;
                    if (CULL) {
                        bool all_far = true;
                        uint32_t nlive = 0;
#pragma unroll
                        for (int g = 0; g < TGT; g++) {
                            far[g] = reach_log2(gbox[g], sbox[sub]) < thr[g];
                            all_far = all_far && far[g]; nlive += !far[g] && gvalid[g];
                        }
                        if (all_far) continue;
                        nexec += nlive;
                    } else {
#pragma unroll
                        for (int g = 0; g < TGT; g++) nexec += gvalid[g];
                    }
                    if constexpr (A32) {
                        // partial sums of another aligned source group are still pending: they join the FP64 accumulators first
                        const int sg = (l0 / 32 + sub) / CONN_A32_GROUPS;
                        if (pend >= 0 && pend != sg) flush();
                        pend = sg;
                        // does the group of 32 sources at hand hold one of the warp's own targets, or is one of its target groups out of reach?
                        bool special = false;
#pragma unroll
                        for (int g = 0; g < TGT; g++) special = special || (CULL && far[g]) || l0 + 32 * sub == slot0 + (wid * TGT + g) * 32;
                        if (special) {
#pragma unroll 1
                            for (int j = 32 * sub; j < 32 * sub + 32; j += CONN_BATCH) batch(j, std::true_type());
                        } else {
#pragma unroll 1
                            for (int j = 32 * sub; j < 32 * sub + 32; j += CONN_BATCH) batch(j, std::false_type());
                        }
                    } else {
#pragma unroll 1
                        for (int j = 32 * sub; j < 32 * sub + 32; j += CONN_BATCH) batch(j, std::true_type());
                    }
                }
            }
            __syncthreads();
            cur = nxt; stage ^= 1;
        }
        if (pend >= 0) flush();
#pragma unroll
        for (int g = 0; g < TGT; g++) {
            const int k = kp[g];
            if (k >= 0) {
#pragma unroll
                for (int t = 0; t < NYB; t++)
                    if (32 * w + t < a.ntrans) Sout[(size_t)(32 * w + t) * n + k] = A32 ? sacc[(g * NYB + t) * NTHR] : acc[A32 ? 0 : g][A32 ? 0 : t];
            }
        }
    }
    if (a.stats && lane == 0 && warp_live) {
        int ngrp = 0;
#pragma unroll
        for (int g = 0; g < TGT; g++) ngrp += gvalid[g];
        atomicAdd(&a.stats[MP_CNT_CONN_EXEC], (unsigned long long)nexec);
        atomicAdd(&a.stats[MP_CNT_CONN_TOTAL], (unsigned long long)ngrp * (unsigned long long)((n + 31) / 32) * (unsigned long long)a.nwords);
    }
}

}  // namespace mp
