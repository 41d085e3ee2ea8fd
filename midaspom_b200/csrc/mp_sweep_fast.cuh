// mp_sweep_fast.cuh -- FP32 throughput path of the Gibbs scan of the intermediate state y_t | z.
//
// Same update as k_sweep_y (mp_kernels.cuh) -- visit the candidate cells (z_t = z_t+1 = 1) of one
// (chain, transition) in patch order, evaluate the N-wide rank-1 change of the colonisation terms
// (compPePc:40 of main_MIDASPOM.c), flip when logit(u) < delta -- laid out for the SM:
//
//  * k_build_candidates compacts the candidates of every (chain, transition) into 32-byte records
//    {patch | y<<31, x, y, log2 A^b, logit(u)} with u = Philox(seed, chain, sweep, RK_Y, k, t): the
//    scan kernel streams them with a one-record prefetch and the random stream still depends on
//    (chain, sweep, cell) only;
//  * one task is split over a thread-block CLUSTER of CS CTAs (CS x NT = 1024 threads, thread g
//    owns targets g, g+1024, ...), so that C x (T-1) tasks that do not divide the 148 SMs (cfg3:
//    8 x 19 = 152) still fill them; per-flip partial sums travel through distributed shared memory
//    with st.async + mbarrier complete_tx (no cluster-wide barrier or fence per flip);
//  * per target one float4 {S_hi, S_lo, x, y} in shared memory: S_t is an unevaluated float pair,
//    so adding and later removing the same FP32 weight cancels to ~2^-48 without FP64 in the loop;
//  * the colonisation factor of a cell is one FFMA.SAT: z'=1 -> sat(cK S), z'=0 -> sat(1 - cK S);
//    the sum of log-ratios is lg2 of a running PRODUCT of the new factors (one MUFU.LG2 per U
//    targets) minus a per-thread cached sum D of the current factors' logs, refreshed on commit.
// MUFU budget per (candidate, target) pair, planar geometry: SQRT + EX2 + LG2/U.
//
// Exceptional cases (a zero current factor, i.e. an impossible current state; removal of the last
// occupied patch) are re-evaluated cell by cell with the (-inf) - (-inf) := 0 convention of the
// generic kernel so that a chain can leave an impossible initial state.
#pragma once
#include "mp_device.cuh"

namespace mp {

struct CandRec { uint32_t kinfo; float kx, ky, lawk, thr; uint32_t pad[3]; };   // 32 bytes; pad[0] = layout (Morton) slot of the patch, pad[1] = its position in the visiting order

// ------------------------------------------------------------------ cluster / DSMEM primitives
__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r;
}
__device__ __forceinline__ void cluster_barrier()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t map_to_rank(uint32_t smem_addr, uint32_t rank)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity)
{
    // the suspend-time hint lets the hardware park the warp until the phase completes instead of re-issuing the poll
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(mbar), "r"(parity), "r"(20000u) : "memory");
}
// remote 4-byte store that completes 4 tx bytes on the destination CTA's mbarrier
__device__ __forceinline__ void st_async_f32(uint32_t remote_addr, float v, uint32_t remote_mbar)
{
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];"
                 ::"r"(remote_addr), "r"(__float_as_uint(v)), "r"(remote_mbar) : "memory");
}
__device__ __forceinline__ void st_async_f32x4(uint32_t remote_addr, float4 v, uint32_t remote_mbar)
{
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];"
                 ::"r"(remote_addr), "r"(__float_as_uint(v.x)), "r"(__float_as_uint(v.y)), "r"(__float_as_uint(v.z)), "r"(__float_as_uint(v.w)),
                   "r"(remote_mbar) : "memory");
}
__device__ __forceinline__ float warp_sum_f(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------ candidate records
// One CTA per (chain, transition): candidates in patch order, compacted by a block scan.
static __global__ void __launch_bounds__(1024)
k_build_candidates(uint64_t seed, int chain_offset, const uint32_t *__restrict__ sweep_p /* device-resident sweep counter */, Landscape<float> ls, const float *__restrict__ aw,
                   const uint8_t *__restrict__ z, const uint8_t *__restrict__ y, CandRec *__restrict__ rec,
                   int *__restrict__ count /* [task][2]: candidates, occupied */, int T, int coords, int task_first, int task_stride,
                   const int *__restrict__ scan /* visiting order: position -> patch */, const int *__restrict__ minv /* patch -> layout (Morton) slot */)
{
    __shared__ int s_cnt[1024], s_occ[32];
    const uint32_t sweep = *sweep_p;
    const int n = ls.n, ntrans = T - 1, tid = threadIdx.x;
    const int task = task_first + blockIdx.x * task_stride, c = task / ntrans, t = task - c * ntrans;
    const uint8_t *zt = z + ((size_t)c * T + t) * n, *zn = zt + n, *yt = y + ((size_t)c * ntrans + t) * n;
    // candidates are emitted in the visiting order of the scan (Morton order, block by block with a scan grid; the identity
    // without coordinates): consecutive candidates are spatial neighbours, which the culled scan exploits; any fixed
    // visiting order is a valid Gibbs scan
    const int per = (n + 1023) / 1024, s0 = min(n, tid * per), s1 = min(n, s0 + per);
    int cnt = 0, occ = 0;
    for (int s = s0; s < s1; s++) { const int q = scan[s]; cnt += (zt[q] != 0 && zn[q] != 0); occ += (yt[q] != 0); }
    s_cnt[tid] = cnt;
    occ = (int)warp_sum_f((float)occ);
    if ((tid & 31) == 0) s_occ[tid >> 5] = occ;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {              // inclusive Hillis-Steele scan
        const int v = tid >= o ? s_cnt[tid - o] : 0;
        __syncthreads();
        s_cnt[tid] += v;
        __syncthreads();
    }
    int off = s_cnt[tid] - cnt;
    CandRec *out = rec + (size_t)task * n;
    for (int s = s0; s < s1; s++) {
        const int q = scan[s];
        if (!(zt[q] != 0 && zn[q] != 0)) continue;
        CandRec r;
        r.kinfo = (uint32_t)q | ((uint32_t)(yt[q] != 0) << 31);
        r.kx = coords ? ls.px[q] : 0.f; r.ky = coords ? ls.py[q] : 0.f;
        r.lawk = aw[(size_t)c * n + q];                 // FP32 engines keep log2 A^b (area_pre<float>)
        r.thr = (float)logit_u(rng(seed, (uint32_t)(chain_offset + c), sweep, RK_Y, (uint32_t)q, (uint32_t)t).x);
        r.pad[0] = (uint32_t)minv[q]; r.pad[1] = (uint32_t)s; r.pad[2] = 0;
        out[off++] = r;
    }
    if (tid == 1023) count[2 * task] = s_cnt[1023];
    if (tid == 0) { int tot = 0; for (int w = 0; w < 32; w++) tot += s_occ[w]; count[2 * task + 1] = tot; }
}

// ------------------------------------------------------------------ the scan
template <int GEOM>
__device__ __forceinline__ float fast_weight(const Landscape<float> &ls, float nal2e, float lawk, int k, float kx, float ky,
                                             int q, float qx, float qy, const float *__restrict__ drow)
{
    float d;                                            // same expressions as pair_distance / weight_of (mp_device.cuh)
    if (GEOM == MP_GEOM_LINEAR) d = (float)(q > k ? q - k : k - q) * ls.spacing;
    else if (GEOM == MP_GEOM_COORDS) { const float dx = qx - kx, dy = qy - ky; d = Num<float>::sqrtv(fmaf(dx, dx, dy * dy)); }
    else d = drow[q < ls.n ? q : k];
    return weight_of(nal2e, lawk, d);                   // A_k^b exp(-alpha d) = 2^(log2 A_k^b - alpha log2(e) d)
}
// colonisation factor of a cell with y=0: class A (z'=1): sat(cK S) ; class B (z'=0): sat(1 - cK S) ; neither: 1
__device__ __forceinline__ float col_factor(float cK, float s, bool a, bool b)
{
    const float u = cK * s;
    float f = 1.f;
    if (a) f = __saturatef(u);
    if (b) f = __saturatef(1.f - u);
    return f;
}

// Launch order of the scan tasks: the (chain, year) scans are sequential and of unequal length (candidates per year
// differ), all start together and the kernel ends with the longest.  Longest first is the classic LPT rule: the CTAs
// dispatched last -- the ones that share an SM with more neighbours, or wait for a second wave -- get the shortest scans.
static __global__ void __launch_bounds__(1024)
k_order_tasks(const int *__restrict__ count, int ntask, int task_first, int task_stride, int *__restrict__ order)
{
    for (int m = threadIdx.x; m < ntask; m += blockDim.x) {
        const int tm = task_first + m * task_stride, cm = count[2 * tm];
        int rank = 0;
        for (int o = 0; o < ntask; o++) {
            const int co = count[2 * (task_first + o * task_stride)];
            rank += (co > cm) || (co == cm && o < m);
        }
        order[rank] = tm;
    }
}

template <int GEOM, int CS, int U, int TPT>
__global__ void __launch_bounds__(TPT / CS, TPT > 1024 ? 1 : CS == 16 ? 17 : CS == 8 ? 9 : CS == 4 ? 5 : CS == 2 ? 2 : 1)
k_sweep_y_fast(Landscape<float> ls, const mp_params *__restrict__ par, const uint8_t *__restrict__ era,
               const uint8_t *__restrict__ z, uint8_t *__restrict__ y, double *__restrict__ S,
               const CandRec *__restrict__ rec, const int *__restrict__ count, int T, int ept, const int *__restrict__ order,
               unsigned long long *__restrict__ stats)
{
    constexpr int NT = TPT / CS, NW = NT / 32;
    constexpr bool HIER = TPT / 32 > 32;                // more than 32 warps per task: reduce inside the CTA first
    constexpr int NSLOT = HIER ? CS : TPT / 32;          // partial sums exchanged per flip (<= 32)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ float red[2][2][32];                    // [round: fast, careful][parity][cluster rank * NW + warp]
    __shared__ float wred[2][2][32];                   // HIER only: per-warp partials inside the CTA
    __shared__ __align__(8) unsigned long long mbar[2][2];
    const int n = ls.n, ntrans = T - 1, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint32_t rank = CS > 1 ? cluster_ctarank() : 0u;
    const int task = order[blockIdx.x / CS];        // this engine's tasks (year sharding over GPUs), longest first (k_order_tasks)
    const int c = task / ntrans, t = task - c * ntrans;
    float4 *sT = reinterpret_cast<float4 *>(smem_raw);               // {S_hi, S_lo, x, y} of own targets, slot tid + j NT

    const Trans<float> tr = make_trans<float>(par[c], era ? era[t] : 0);
    const float cK = tr.c * tr.Kt;
    const float nal2e = alpha_pre<float>(par[c].alpha);
    // external source (loss.c:93-101, future.c:90-97): C = c (K S + Ksrc g_q) = cK (S + (Ksrc/K) g_q).  The
    // per-target offset is folded into the stored S for the duration of the scan and removed on write-back.
    const double src_scale = tr.src ? (double)tr.Ks / (double)tr.Kt : 0.0;
    auto src_offset = [&](int q) -> double {
        if (!tr.src) return 0.0;
        const double u = ls.src_unit ? ls.src_unit[q] : (double)(q + 1);
        return src_scale * exp(-(par[c].alpha * u) * par[c].dsrc);
    };
    uint8_t *yt = y + ((size_t)c * ntrans + t) * n;
    const uint8_t *zn = z + ((size_t)c * T + t + 1) * n;
    double *St = S + ((size_t)c * ntrans + t) * n;

    // own targets: q_j = g + TPT j, g = rank * NT + tid.  Amask: y=0,z'=1 ; Bmask: y=0,z'=0 ; ybits: y
    const int g = (int)rank * NT + tid;
    uint32_t Amask = 0, Bmask = 0, ybits = 0;
    for (int j = 0; j < ept; j++) {
        const int q = g + j * TPT;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q < n) {
            if (GEOM == MP_GEOM_COORDS) { v.z = ls.px[q]; v.w = ls.py[q]; }
            const double s = St[q] + src_offset(q);
            v.x = (float)s; v.y = (float)(s - (double)v.x);
            const uint32_t yq = yt[q] != 0, zq = zn[q] != 0;
            ybits |= yq << j; Amask |= ((yq ^ 1u) & zq) << j; Bmask |= ((yq ^ 1u) & (zq ^ 1u)) << j;
        }
        sT[tid + j * NT] = v;
    }
    // D = sum over own cells with y=0 of lg2 f(S): the denominator of every ratio until the next commit
    auto refresh_D = [&]() {
        float D = 0.f, P = 1.f;
        int j = 0;
        for (; j + U <= ept; j += U) {
#pragma unroll
            for (int u = 0; u < U; u++) P *= col_factor(cK, sT[tid + (j + u) * NT].x, (Amask >> (j + u)) & 1u, (Bmask >> (j + u)) & 1u);
            D += Num<float>::lg2(P); P = 1.f;
        }
        if (j < ept) {
            for (; j < ept; j++) P *= col_factor(cK, sT[tid + j * NT].x, (Amask >> j) & 1u, (Bmask >> j) & 1u);
            D += Num<float>::lg2(P);
        }
        return D;
    };
    float D = refresh_D();

    if (CS > 1) {
        if (tid == 0) {
#pragma unroll
            for (int i = 0; i < 4; i++) mbar_init(smem_u32(&mbar[i >> 1][i & 1]), 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        cluster_barrier();                              // barriers initialised and every CTA running before remote stores
    }
    // DSMEM addresses of this lane's destination CTA (lane < CS): red[0][0][0] and mbar[0][0] of CTA `lane`
    const uint32_t red_remote = CS > 1 ? map_to_rank(smem_u32(&red[0][0][0]), (uint32_t)(lane < CS ? lane : 0)) : 0u;
    const uint32_t bar_remote = CS > 1 ? map_to_rank(smem_u32(&mbar[0][0]), (uint32_t)(lane < CS ? lane : 0)) : 0u;
    const uint32_t bar_local = smem_u32(&mbar[0][0]);
    const int ncand = count[2 * task];
    int nocc = count[2 * task + 1];
    const CandRec *recs = rec + (size_t)task * n;
    uint32_t uses[2] = { 0u, 0u };                      // completed reduction rounds per kind

    // all-reduce of one float per warp over the cluster; every thread returns the same total
    auto all_reduce = [&](int round, float v) -> float {
        const uint32_t u = uses[round]++;
        const int p = u & 1;
        v = warp_sum_f(v);
        if (HIER) {                                     // CTA partial first (one __syncthreads), then CS partials over DSMEM
            if (lane == 0) wred[round][p][wid] = v;
            __syncthreads();
            v = warp_sum_f(lane < NW ? wred[round][p][lane] : 0.f);
        }
        if (CS > 1) {
            const uint32_t boff = (uint32_t)(round * 2 + p) * 8u;                       // &mbar[round][p] - &mbar[0][0]
            const uint32_t slot = HIER ? rank : rank * NW + wid;
            const uint32_t roff = (uint32_t)((round * 2 + p) * 32 + (int)slot) * 4u;    // &red[round][p][slot] - &red[0][0][0]
            if (tid == 0) mbar_expect_tx(bar_local + boff, NSLOT * 4);  // NSLOT slots x 4 bytes land on this CTA
            if (lane < CS && (!HIER || wid == 0)) st_async_f32(red_remote + roff, v, bar_remote + boff);
            mbar_wait(bar_local + boff, (u >> 1) & 1u);
            return warp_sum_f(lane < NSLOT ? red[round][p][lane] : 0.f);
        }
        if (HIER) return v;                             // single CTA: the CTA partial is the total
        if (lane == 0) red[round][p][wid] = v;
        __syncthreads();
        return warp_sum_f(lane < NSLOT ? red[round][p][lane] : 0.f);
    };

    float4 r0 = make_float4(0.f, 0.f, 0.f, 0.f), r1 = r0;     // current record as two 16-byte halves
    if (ncand > 0) { r0 = reinterpret_cast<const float4 *>(recs)[0]; r1 = reinterpret_cast<const float4 *>(recs)[1]; }
    for (int i = 0; i < ncand; i++) {
        float4 n0 = r0, n1 = r1;                        // prefetch the next record while this one is evaluated
        if (i + 1 < ncand) { n0 = reinterpret_cast<const float4 *>(recs)[2 * (i + 1)]; n1 = reinterpret_cast<const float4 *>(recs)[2 * (i + 1) + 1]; }
        const uint32_t kinfo = __float_as_uint(r0.x);
        const int k = (int)(kinfo & 0x7fffffffu);
        const uint32_t cur = kinfo >> 31;               // y[k] is untouched until its own visit
        const float kx = r0.y, ky = r0.z, lawk = r0.w, thr_k = r1.x;
        const bool zero_after = (nocc + (cur ? -1 : 1)) == 0;
        const float sgn = cur ? -1.f : 1.f;
        const float *drow = GEOM == MP_GEOM_DENSE ? ls.dist + (size_t)k * n : nullptr;
        const bool own = k >= g && (k - g) % TPT == 0;
        const int kj = own ? (k - g) / TPT : 31;         // slot of k if this thread owns it (bit 31 is never a valid slot... ept <= 31)
        const uint32_t ownbit = own ? 1u << kj : 0u;
        const uint32_t Ae = Amask & ~ownbit, Be = Bmask;  // a candidate has z'=1: it can only be in class A

        float total = 0.f;
        bool careful = zero_after;
        if (!careful) {
            float acc2 = -D, P = 1.f;
            auto eval_one = [&](int j) {
                const float4 tq = sT[tid + j * NT];
                const float w = fast_weight<GEOM>(ls, nal2e, lawk, k, kx, ky, g + j * TPT, tq.z, tq.w, drow);
                const float sa = fmaf(sgn, w, tq.x) + tq.y;            // a negative rounding residue saturates like 0 below
                P *= col_factor(cK, sa, (Ae >> j) & 1u, (Be >> j) & 1u);
            };
            int j = 0;
            for (; j + U <= ept; j += U) {
#pragma unroll
                for (int u = 0; u < U; u++) eval_one(j + u);
                acc2 += Num<float>::lg2(P); P = 1.f;
            }
            if (j < ept) { for (; j < ept; j++) eval_one(j); acc2 += Num<float>::lg2(P); }
            if (own) {
                // own cell.  cur=0: D already holds lg2 C_k, the flip adds log(1-E) - log E.
                // cur=1: the flip adds log E + log C_k - log(1-E).
                const float lg2e = 1.4426950408889634f;
                if (cur) acc2 += lg2e * (tr.logE - tr.log1mE) + Num<float>::lg2(__saturatef(cK * sT[tid + kj * NT].x));
                else acc2 += lg2e * (tr.log1mE - tr.logE);
            }
            total = all_reduce(0, acc2);
            careful = isnan(total);
        }
        if (careful) {
            // cell-by-cell log differences with (-inf) - (-inf) := 0 and finite - (-inf) := +inf
            float acc2 = 0.f;
            for (int j = 0; j < ept; j++) {
                const bool a = (Ae >> j) & 1u, b = (Be >> j) & 1u;
                if (!(a || b)) continue;
                const float4 tq = sT[tid + j * NT];
                const float w = fast_weight<GEOM>(ls, nal2e, lawk, k, kx, ky, g + j * TPT, tq.z, tq.w, drow);
                const float sa = zero_after ? (float)src_offset(g + j * TPT) : fmaxf(fmaf(sgn, w, tq.x) + tq.y, 0.f);
                acc2 += ldiff<float>(Num<float>::lg2(col_factor(cK, sa, a, b)), Num<float>::lg2(col_factor(cK, tq.x, a, b)));
            }
            if (own) {
                const float lg2e = 1.4426950408889634f;
                const float l0 = lg2e * tr.logE + Num<float>::lg2(__saturatef(cK * sT[tid + kj * NT].x));
                const float l1 = lg2e * tr.log1mE;
                acc2 += cur ? ldiff<float>(l0, l1) : ldiff<float>(l1, l0);
            }
            total = all_reduce(1, acc2);
        }
        const float delta = 0.6931471805599453f * total;
        if (thr_k < delta) {                              // NaN compares false: no flip
            if (own) { ybits ^= ownbit; Amask ^= ownbit; }  // cur=1 -> y=0 joins class A ; cur=0 -> leaves it
            nocc += cur ? -1 : 1;
            // commit: S +- w for every own target (two-float), and the new denominator D in the same pass
            float Dn = 0.f, P = 1.f;
            auto commit_one = [&](int j) {
                const float4 tq = sT[tid + j * NT];
                const float w = fast_weight<GEOM>(ls, nal2e, lawk, k, kx, ky, g + j * TPT, tq.z, tq.w, drow);
                const float a = j == kj ? 0.f : sgn * w;               // S_k does not contain y_k
                const float s = tq.x + a, bb = s - tq.x;
                const float e = (tq.x - (s - bb)) + (a - bb);           // exact rounding error of hi + a
                const float lo2 = tq.y + e;
                float hi = s + lo2, lo = lo2 - (hi - s);
                if (hi < 0.f) { hi = 0.f; lo = 0.f; }
                *reinterpret_cast<float2 *>(&sT[tid + j * NT]) = make_float2(hi, lo);
                P *= col_factor(cK, hi, (Amask >> j) & 1u, (Bmask >> j) & 1u);
            };
            if (!zero_after) {
                int j = 0;
                for (; j + U <= ept; j += U) {
#pragma unroll
                    for (int u = 0; u < U; u++) commit_one(j + u);
                    Dn += Num<float>::lg2(P); P = 1.f;
                }
                if (j < ept) { for (; j < ept; j++) commit_one(j); Dn += Num<float>::lg2(P); }
            } else {
                // the last occupied patch left: every S is exactly its external-source offset
                for (int j = 0; j < ept; j++) {
                    const double so = src_offset(g + j * TPT);
                    const float hi = (float)so, lo = (float)(so - (double)hi);
                    *reinterpret_cast<float2 *>(&sT[tid + j * NT]) = make_float2(hi, lo);
                    P = col_factor(cK, hi, (Amask >> j) & 1u, (Bmask >> j) & 1u);
                    Dn += Num<float>::lg2(P);
                }
            }
            D = Dn;
        }
        r0 = n0; r1 = n1;
    }
    for (int j = 0; j < ept; j++) {
        const int q = g + j * TPT;
        if (q < n) {
            const float4 tq = sT[tid + j * NT];
            St[q] = fmax(((double)tq.x + (double)tq.y) - src_offset(q), 0.0);
            yt[q] = (uint8_t)((ybits >> j) & 1u);
        }
    }
    if (stats && tid == 0 && rank == 0) atomicAdd(&stats[MP_CNT_SCAN_DENSE], (unsigned long long)ncand * (unsigned long long)n);
    if (CS > 1) cluster_barrier();                      // no CTA leaves while a peer could still address its smem
}

}  // namespace mp

// ------------------------------------------------------------------ host-side dispatch (one TU per geometry)
#ifdef MP_FAST_GEOM
#include "mp_host.h"
namespace mp {
template <int CS, int U, int TPT> static int launch_fast(mp_engine *h, int ept)
{
    constexpr int NT = TPT / CS;
    const size_t smem = (size_t)ept * NT * 16;
    REQUIRE(smem <= 227 * 1024 && ept <= 31, MP_ERR_UNSUPPORTED, "n_patches too large for the fast y sweep");
    auto kern = k_sweep_y_fast<MP_FAST_GEOM, CS, U, TPT>;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (CS > 8) CK(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    const int ntask_all = h->cfg.n_chains * (h->cfg.n_years - 1);
    const int ntask = (ntask_all - h->task_first + h->task_stride - 1) / h->task_stride;
    if (ntask <= 0) return MP_OK;
    cfg.gridDim = dim3((unsigned)(ntask * CS));
    cfg.blockDim = dim3(NT);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = h->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = CS > 1 ? 1 : 0;
    CK(cudaLaunchKernelEx(&cfg, kern, view<float>(h), (const mp_params *)h->d_par,
                          (const uint8_t *)(h->have_era ? h->d_era : nullptr), (const uint8_t *)h->d_z, h->d_y, h->d_S[0],
                          (const CandRec *)h->d_cand, (const int *)h->d_cand_count, h->cfg.n_years, ept, (const int *)h->d_task_order,
                          h->d_work));
    return MP_OK;
}
template <int CS, int TPT> static int launch_fast_u(mp_engine *h, int ept)
{
    return ept % 5 == 0 ? launch_fast<CS, 5, TPT>(h, ept) : launch_fast<CS, 4, TPT>(h, ept);
}
// tpt = threads per task: 1024 for small landscapes; 512 for large ones (fewer warps pay the
// per-flip bookkeeping and reduction, each thread carries more independent targets)
static int launch_fast_any(mp_engine *h, int cs, int tpt)
{
    const int ept = (h->cfg.n_patches + tpt - 1) / tpt;
    if (tpt == 256) return cs >= 2 ? launch_fast_u<2, 256>(h, ept) : launch_fast_u<1, 256>(h, ept);   // small landscapes
    if (tpt == 128) return launch_fast_u<1, 128>(h, ept);
#ifndef MP_FAST_HAS_POSITIONS                           // with positions, 512 threads per task and more take the culled scan
    if (tpt > 1024) {                                   // large landscapes: clusters of 8 (or 16), 256..1024 threads per CTA
        if (tpt == 2048) return launch_fast_u<8, 2048>(h, ept);
        if (tpt == 4096) return cs == 16 ? launch_fast_u<16, 4096>(h, ept) : launch_fast_u<8, 4096>(h, ept);
        return cs == 16 ? launch_fast_u<16, 8192>(h, ept) : launch_fast_u<8, 8192>(h, ept);
    }
    if (tpt == 512) switch (cs) {
        case 1: return launch_fast_u<1, 512>(h, ept);
        case 2: return launch_fast_u<2, 512>(h, ept);
        case 4: return launch_fast_u<4, 512>(h, ept);
        case 16: return launch_fast_u<16, 512>(h, ept);
        default: return launch_fast_u<8, 512>(h, ept);
    }
    switch (cs) {
    case 1: return launch_fast_u<1, 1024>(h, ept);
    case 2: return launch_fast_u<2, 1024>(h, ept);
    case 4: return launch_fast_u<4, 1024>(h, ept);
    case 16: return launch_fast_u<16, 1024>(h, ept);
    default: return launch_fast_u<8, 1024>(h, ept);
    }
#endif
    return MP_ERR_UNSUPPORTED;
}
}  // namespace mp
#endif
