// mp_sweep_cull.cuh -- the FP32 fast y scan (mp_sweep_fast.cuh) with EXACT spatial culling of the evaluation.
//
// Targets are laid out in Morton order (perm[slot] = patch): thread g owns slots g, g+TPT, ..., so the 32
// lanes of a warp hold, for every j, 32 spatially adjacent patches -- a "group" with a bounding circle
// (centre, radius) and a lower bound mlow on its S values.  For a candidate k the dispersal weight of every
// target of a group is at most wub = A_k^b exp(-alpha max(0, |centre - k| - radius)).  If wub < 2^-26 mlow then
// fl(S_hi +- w) = S_hi for every target of the group: the factor ratio is exactly 1 and the group's lg2
// contribution exactly 0 -- the whole slot is skipped for the warp, with no approximation (a chain's path
// is that of the unculled kernel up to FP32 ties).  With landscapes much wider than the dispersal range
// (cfg3: 25 km vs 1/alpha = 0.4 km) most groups are skipped.  The commit skips a group when wub < 2^-36 mlow:
// the skipped mass, summed over all commits between two refreshes of S (every 16 sweeps), stays orders of
// magnitude below the FP32 resolution of S (measured drift of S against k_conn: tests/test_gpu_parity.py).
//
// Differences from k_sweep_y_fast:
//  * candidate records carry the candidate's Morton slot and are staged through a two-chunk ring in shared memory;
//  * the denominator product is formed on the fly over the evaluated slots (no cached D);
//  * lane j of every warp keeps the bounds of the warp's group j in registers; a removal recomputes the exact
//    min S of every group it commits to with one REDUX (S_hi >= 0, so the IEEE bit pattern orders like the value);
//  * the evaluated slots are taken from the ballot mask in batches of up to 4 independent dependency chains;
//  * every trip evaluates SP consecutive candidates (the first and SP-1 speculative ones) in one pass over the union
//    of their active groups and reduces the SP sums in ONE exchange: a rejected flip (2 of 3) costs no reduction
//    latency of its own.  The decisions are exactly those of the one-at-a-time scan: a later candidate's sum is
//    used only if every earlier one of the window left the state unchanged;
//  * BR (SP = 2 with at most 16 senders: how every 512-thread task, whole-year or block, runs): a trip also forms a third sum,
//    candidate i+1 GIVEN that i is accepted.  The state after i's commit differs only by +-w_i, which the pass already computes
//    for every slot it visits:
//    fn(fma(sgn_{i+1}, w_{i+1}, fma(sgn_i, w_i, S_hi)) + S_lo) over the post-commit denominator fn(fma(sgn_i, w_i, S_hi) + S_lo),
//    which is candidate i's own numerator -- no weight is evaluated twice.  A trip thus retires both candidates whatever i's
//    outcome (about 0.5 instead of 0.6 trips per candidate).  The branch sum stands for the exact post-commit evaluation up to
//    ~ulp(S) on every S, i.e. up to FP32 ties, except under cancellation (a removal leaving less than S_hi/4 of a target, or the
//    clamp at 0) and the careful cases: those poison it with NaN and defer i+1 to the next trip.
#pragma once
#include "mp_sweep_fast.cuh"

namespace mp {

// candidates evaluated per trip (1 + speculative ones), measured: cfg3 (512 threads per task) 10.0 / 10.4 / 11.1 ms for 2 / 3 / 4,
// cfg5t (4096 threads per task, exchange-latency bound) 43.4 / 39.3 / 38.3 ms (6: 42.9, 8: 51.3)
constexpr int MP_CULL_SPEC = 2;
constexpr int MP_CULL_SPEC_LARGE = 4;

// One unit of work of a block launch: the candidates of one block of the scan grid in one (chain, year) task, with the
// block's own patches and every patch within the halo around it as targets (mp_set_scan_blocks).  Blocks of one colour
// lie farther apart than twice the halo, so their target sets are disjoint and their scans run concurrently.
struct BlockTask { int task, tl_off, nl, slot_lo, slot_hi; };

// CTAs of NT threads that should share an SM (registers: about 96 per thread)
__host__ __device__ constexpr int cull_min_blocks(int nt) { return nt <= 32 ? 17 : nt <= 64 ? 9 : nt <= 128 ? 5 : nt <= 256 ? 2 : 1; }

template <int GEOM, int CS, int TPT>
__global__ void __launch_bounds__(TPT / CS, TPT > 1024 ? 1 : cull_min_blocks(TPT / CS))
k_sweep_y_cull(Landscape<float> ls, const int *__restrict__ perm, const mp_params *__restrict__ par,
               const uint8_t *__restrict__ era, const uint8_t *__restrict__ z, uint8_t *__restrict__ y, double *__restrict__ S,
               const CandRec *__restrict__ rec, const int *__restrict__ count, int T, int ept_max, const int *__restrict__ order,
               unsigned long long *__restrict__ stats /* MP_CNT_SCAN_* work counters of the engine (mp_get_work_counters) */,
               const BlockTask *__restrict__ btasks /* block launch: one entry per cluster (order is unused); nullptr: whole (chain, year) tasks */,
               const int *__restrict__ tlist /* block launch: target lists (patch numbers) */,
               const int *__restrict__ blockmode /* per (chain, year) task: 1 = scanned by the block launches, 0 = by the whole-task launch (nullptr: no block grid) */)
{
    static_assert(GEOM != MP_GEOM_DENSE, "culling needs positions");
    constexpr int NT = TPT / CS, NW = NT / 32, SP = TPT > 1024 ? MP_CULL_SPEC_LARGE : MP_CULL_SPEC;
    constexpr bool HIER = TPT / 32 > 32;
    constexpr int NSLOT = HIER ? CS : TPT / 32;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NV = (SP + 3) / 4;                                 // float4 per sender in the exchange of the SP sums
    // the "i+1 given i accepted" sum: two candidates from at most 16 senders (every 512-thread task)
    constexpr bool BR = SP == 2 && !HIER && NSLOT <= 16;
    constexpr int NS = SP + (BR ? 1 : 0);                            // sums exchanged per trip
    __shared__ __align__(16) float4 red[2][2][32][NV];
    __shared__ __align__(16) float4 wred[HIER ? 2 : 1][2][32][NV];
    __shared__ __align__(8) unsigned long long mbar[2][2];
    const int n = ls.n, ntrans = T - 1, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint32_t rank = CS > 1 ? cluster_ctarank() : 0u;
    // what this cluster scans: a whole (chain, year) task (targets = all patches in scan order) or one block of it
    const BlockTask bt = btasks ? btasks[blockIdx.x / CS] : BlockTask{ order[blockIdx.x / CS] /* longest task first (k_order_tasks) */, 0, n, 0, n };
    const int task = bt.task;
    const int c = task / ntrans, t = task - c * ntrans;
    // a (chain, year) task is scanned either by the block launches or by the whole-task launch, decided per sweep
    // (k_block_valid); the whole cluster takes the same branch, before any cluster-wide synchronisation
    if (blockmode && (blockmode[task] != 0) != (btasks != nullptr)) return;
    const int nl = bt.nl;                                            // targets of this cluster
    const int *tl = btasks ? tlist + bt.tl_off : perm;               // local slot -> patch
    const int ept = (nl + TPT - 1) / TPT;                            // slots per thread (<= ept_max, which sizes the shared memory)
    float4 *sT = reinterpret_cast<float4 *>(smem_raw);               // {S_hi, S_lo, x, y} (COORDS) or {S_hi, S_lo, patch, -} (LINEAR)
    float4 *ring = sT + ept_max * NT;                                // 2 chunks of RC candidate records (two float4 each)
    // this thread's column of sT (slot j at sTt[j * NT]) from a shared address held in a register: left to the compiler, the
    // column's base was rebuilt from the shared window base in every batch of the slot loops
    uint32_t col_off = smem_u32(sT + tid);
    asm volatile("" : "+r"(col_off));
    float4 *const sTt = reinterpret_cast<float4 *>(__cvta_shared_to_generic(col_off));

    const Trans<float> tr = make_trans<float>(par[c], era ? era[t] : 0);
    const float cK = tr.c * tr.Kt;
    const float nal2e = alpha_pre<float>(par[c].alpha);
    const double src_scale = tr.src ? (double)tr.Ks / (double)tr.Kt : 0.0;
    auto src_offset = [&](int q) -> double {
        if (!tr.src) return 0.0;
        const double u = ls.src_unit ? ls.src_unit[q] : (double)(q + 1);
        return src_scale * exp(-(par[c].alpha * u) * par[c].dsrc);
    };
    uint8_t *yt = y + ((size_t)c * ntrans + t) * n;
    const uint8_t *zn = z + ((size_t)c * T + t + 1) * n;
    double *St = S + ((size_t)c * ntrans + t) * n;

    const int g = (int)rank * NT + tid;
    uint32_t Amask = 0, Bmask = 0, ybits = 0, valid = 0;
    // lane j of every warp keeps the bounds of the warp's group j: COORDS {centre x, centre y, radius}, LINEAR {first, last patch}; Gw = min S
    float Gx = 0.f, Gy = 0.f, Gr = 3.0e38f, Gw = 0.f;
    for (int j = 0; j < ept; j++) {
        const int s = g + j * TPT;
        const int q = s < nl ? tl[s] : -1;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q >= 0) {
            if (GEOM == MP_GEOM_COORDS) { v.z = ls.px[q]; v.w = ls.py[q]; }
            else v.z = __int_as_float(q);
            const double sv = St[q] + src_offset(q);
            v.x = (float)sv; v.y = (float)(sv - (double)v.x);
            const uint32_t yq = yt[q] != 0, zq = zn[q] != 0;
            ybits |= yq << j; Amask |= ((yq ^ 1u) & zq) << j; Bmask |= ((yq ^ 1u) & (zq ^ 1u)) << j; valid |= 1u << j;
        }
        sT[tid + j * NT] = v;
        const float big = 3.0e38f;
        float a0, a1, b0, b1, ml = q >= 0 ? v.x : big;
        if (GEOM == MP_GEOM_COORDS) { a0 = q >= 0 ? v.z : big; a1 = q >= 0 ? v.z : -big; b0 = q >= 0 ? v.w : big; b1 = q >= 0 ? v.w : -big; }
        else { a0 = q >= 0 ? (float)q : big; a1 = q >= 0 ? (float)q : -big; b0 = 0.f; b1 = 0.f; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a0 = fminf(a0, __shfl_xor_sync(0xffffffffu, a0, o)); a1 = fmaxf(a1, __shfl_xor_sync(0xffffffffu, a1, o));
            b0 = fminf(b0, __shfl_xor_sync(0xffffffffu, b0, o)); b1 = fmaxf(b1, __shfl_xor_sync(0xffffffffu, b1, o));
            ml = fminf(ml, __shfl_xor_sync(0xffffffffu, ml, o));
        }
        if (lane == j) {
            if (a0 > a1) { Gx = 0.f; Gy = 0.f; Gr = 3.0e38f; Gw = 0.f; }     // empty group: every factor is 1 anyway
            else if (GEOM == MP_GEOM_COORDS) { const float dx = a1 - a0, dy = b1 - b0;
                                               Gx = 0.5f * (a0 + a1); Gy = 0.5f * (b0 + b1); Gr = 0.5000005f * sqrtf(dx * dx + dy * dy) + 1e-3f; Gw = ml; }
            else { Gx = a0; Gy = a1; Gr = 0.f; Gw = ml; }
        }
    }
    if (CS > 1) {
        if (tid == 0) {
#pragma unroll
            for (int i = 0; i < 4; i++) mbar_init(smem_u32(&mbar[i >> 1][i & 1]), 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        cluster_barrier();
    } else __syncthreads();
    const uint32_t red_remote = CS > 1 ? map_to_rank(smem_u32(&red[0][0][0]), (uint32_t)(lane < CS ? lane : 0)) : 0u;
    const uint32_t bar_remote = CS > 1 ? map_to_rank(smem_u32(&mbar[0][0]), (uint32_t)(lane < CS ? lane : 0)) : 0u;
    const uint32_t bar_local = smem_u32(&mbar[0][0]);
    // candidates: the task's list is in visiting order; a block owns the contiguous run whose positions lie in [slot_lo, slot_hi)
    const CandRec *recs = rec + (size_t)task * n;
    int ncand = count[2 * task];
    int nocc = count[2 * task + 1];
    if (btasks) {
        auto first_at_least = [&](int slot) {                        // first candidate whose scan-order slot is >= slot
            int lo = 0, hi = ncand;
            while (lo < hi) { const int mid = (lo + hi) >> 1; if ((int)recs[mid].pad[1] < slot) lo = mid + 1; else hi = mid; }
            return lo;
        };
        const int i0 = first_at_least(bt.slot_lo), i1 = first_at_least(bt.slot_hi);
        recs += i0; ncand = i1 - i0;
        nocc = 1 << 30;   // other blocks change the year's occupancy count concurrently; "the last occupied patch left" cannot arise (k_block_valid)
    }
    // slot of a candidate among the targets: whole tasks lay the targets out in Morton order (record field pad[0]); a block's
    // list starts with its own patches in visiting order (pad[1] - slot_lo)
    const int slot_lo = bt.slot_lo;
    const bool blk = btasks != nullptr;
    uint32_t uses[2] = { 0u, 0u };
    // work counters of this warp (warp-uniform values, added to the engine's totals once at the end): trips, (candidate,
    // 32-target group) evaluations executed, the part of them that belongs to retired candidates, groups committed
    uint32_t st_trips = 0, st_exec = 0, st_ret = 0, st_commit = 0;

    // sums of NS per-thread values over the task's TPT threads (warp shuffles, then st.async of the warp or CTA
    // partials -- NV float4 per sender, one float4 with BR -- to every CTA of the cluster, completion counted on the
    // destination's mbarrier)
    auto all_reduce = [&](int round, float (&v)[NS]) {
        const uint32_t u = uses[round]++;
        const int p = u & 1;
        auto pack = [&](int q) {
            float f[4];
#pragma unroll
            for (int i = 0; i < 4; i++) f[i] = 4 * q + i < SP ? v[(4 * q + i) % SP] : 0.f;
            return make_float4(f[0], f[1], f[2], f[3]);
        };
        auto unpack_sum = [&](int q, const float4 &t) {
            if (4 * q + 0 < SP) v[(4 * q + 0) % SP] = warp_sum_f(t.x);
            if (4 * q + 1 < SP) v[(4 * q + 1) % SP] = warp_sum_f(t.y);
            if (4 * q + 2 < SP) v[(4 * q + 2) % SP] = warp_sum_f(t.z);
            if (4 * q + 3 < SP) v[(4 * q + 3) % SP] = warp_sum_f(t.w);
        };
        // value of a slot of the exchange buffer, zero for lanes without a sender (a plain predicated LDS: selecting between
        // a reference into shared memory and a local constant made the compiler emit a generic load from the stack per trip)
        auto slot_of = [&](const float4 *base, int nslot, int q) -> float4 {
            float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
            if (lane < nslot) t = base[lane * NV + q];
            return t;
        };
        if constexpr (BR) {
            // three sums, one float4 {v0, v1, v2, 0} per sender: rounds 16 and 8 of the butterfly as a reduce-scatter, quarter-warp q
            // going on adding v[q] (q = 3: zeros).  Every addition is one the full butterfly of that component forms (IEEE addition
            // commutes), so each sum is bit for bit the full butterfly's, whatever the cluster split
            const bool h16 = lane & 16, h8 = lane & 8;
            const float a = (h16 ? v[2] : v[0]) + __shfl_xor_sync(0xffffffffu, h16 ? v[0] : v[2], 16);
            const float b = (h16 ? 0.f : v[1]) + __shfl_xor_sync(0xffffffffu, h16 ? v[1] : 0.f, 16);
            float x = (h8 ? b : a) + __shfl_xor_sync(0xffffffffu, h8 ? a : b, 8);
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
            // the senders (lanes < CS <= 8, quarter 0) gather the other quarters' sums
            const float4 part = make_float4(x, __shfl_down_sync(0xffffffffu, x, 8), __shfl_down_sync(0xffffffffu, x, 16), 0.f);
            float4 *slots4 = &red[round][p][0][0];
            if (CS > 1) {
                const uint32_t boff = (uint32_t)(round * 2 + p) * 8u;
                if (tid == 0) mbar_expect_tx(bar_local + boff, NSLOT * 16);
                if (lane < CS) st_async_f32x4(red_remote + (uint32_t)((round * 2 + p) * 32 + (int)rank * NW + wid) * 16u, part, bar_remote + boff);
                mbar_wait(bar_local + boff, (u >> 1) & 1u);
            } else {
                if (lane == 0) slots4[wid] = part;
                __syncthreads();
            }
            // second level: lane l adds component l >> 3 of senders l & 7 and (l & 7) + 8 -- round 8 of the butterfly over the
            // senders (its round 16 only added +0.0, which can change nothing but the sign of a zero sum, and no decision tells
            // -0 from +0) -- then rounds 4, 2, 1 within the quarter
            const float *sf = reinterpret_cast<const float *>(slots4);
            const int s = lane & 7, q = lane >> 3;
            float y = 0.f;
            if (NSLOT == 16 || s < NSLOT) y = sf[4 * s + q];
            if (NSLOT == 16 || s + 8 < NSLOT) y += sf[4 * (s + 8) + q];
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) y += __shfl_xor_sync(0xffffffffu, y, o);
            v[0] = __shfl_sync(0xffffffffu, y, 0);
            v[1] = __shfl_sync(0xffffffffu, y, 8);
            v[2] = __shfl_sync(0xffffffffu, y, 16);
        } else {
#pragma unroll
            for (int c = 0; c < SP; c++) v[c] = warp_sum_f(v[c]);
            if (HIER) {
                if (lane == 0) {
#pragma unroll
                    for (int q = 0; q < NV; q++) wred[round][p][wid][q] = pack(q);
                }
                __syncthreads();
#pragma unroll
                for (int q = 0; q < NV; q++) unpack_sum(q, slot_of(&wred[round][p][0][0], NW, q));
            }
            if (CS > 1) {
                const uint32_t boff = (uint32_t)(round * 2 + p) * 8u;
                const uint32_t slot = HIER ? rank : rank * NW + wid;
                const uint32_t roff = (uint32_t)(((round * 2 + p) * 32 + (int)slot) * NV) * 16u;
                if (tid == 0) mbar_expect_tx(bar_local + boff, NSLOT * 16 * NV);
                if (lane < CS && (!HIER || wid == 0)) {
#pragma unroll
                    for (int q = 0; q < NV; q++) st_async_f32x4(red_remote + roff + 16u * q, pack(q), bar_remote + boff);
                }
                mbar_wait(bar_local + boff, (u >> 1) & 1u);
#pragma unroll
                for (int q = 0; q < NV; q++) unpack_sum(q, slot_of(&red[round][p][0][0], NSLOT, q));
                return;
            }
            if (HIER) return;
            if (lane == 0) {
#pragma unroll
                for (int q = 0; q < NV; q++) red[round][p][wid][q] = pack(q);
            }
            __syncthreads();
#pragma unroll
            for (int q = 0; q < NV; q++) unpack_sum(q, slot_of(&red[round][p][0][0], NSLOT, q));
        }
    };
    // weight of (candidate k, target in slot data tq)
    auto weight = [&](const float4 &tq, int k, float kx, float ky, float lawk) -> float {
        float d;
        if (GEOM == MP_GEOM_LINEAR) { const int q = __float_as_int(tq.z); d = (float)(q > k ? q - k : k - q) * ls.spacing; }
        else { const float dx = tq.z - kx, dy = tq.w - ky; d = Num<float>::sqrtv(fmaf(dx, dx, dy * dy)); }
        return weight_of(nal2e, lawk, d);
    };

    // upper bound of the weights of candidate (k; kx, ky) on this lane's group (margins cover the rounding of the bound itself)
    auto group_bound = [&](int k, float kx, float ky, float lawk) -> float {
        float dlow;
        if (GEOM == MP_GEOM_COORDS) { const float dx = Gx - kx, dy = Gy - ky; dlow = fmaxf(0.f, Num<float>::sqrtv(fmaf(dx, dx, dy * dy)) - Gr); }
        else dlow = ls.spacing * fmaxf(0.f, fmaxf(Gx - (float)k, (float)k - Gy));
        return 1.001f * weight_of(nal2e, lawk, 0.99999f * dlow);     // sqrt.approx, ex2.approx: a few ulp each
    };
    // the flip's own cell, whose connectivity is s
    auto own_term_s = [&](float s, uint32_t cur) -> float {
        const float lg2e = 1.4426950408889634f;
        const float l0 = lg2e * tr.logE + Num<float>::lg2(__saturatef(cK * s));
        const float l1 = lg2e * tr.log1mE;
        return cur ? ldiff<float>(l0, l1) : ldiff<float>(l1, l0);
    };
    auto own_term = [&](int kj, uint32_t cur) -> float {
        const float4 tq = sTt[kj * NT];
        return own_term_s(tq.x + tq.y, cur);
    };

    // ---- candidate records travel through a two-chunk ring in shared memory (chunks c and c+1 resident while i is in chunk c)
    constexpr int RC = 32;
    const float4 *recs4 = reinterpret_cast<const float4 *>(recs);
    auto load_chunk = [&](int cidx) -> float4 {
        const int idx = cidx * RC * 2 + tid;
        return (tid < 2 * RC && idx < 2 * ncand) ? recs4[idx] : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    float4 pre;
    {
        const float4 c0 = load_chunk(0), c1 = load_chunk(1);
        pre = load_chunk(2);
        if (tid < 2 * RC) { ring[tid] = c0; ring[2 * RC + tid] = c1; }
        __syncthreads();
    }
    int chunk = 0;
    struct Cand { int k; uint32_t cur; float kx, ky, lawk; };
    auto bound_of = [&](int i) -> float {
        const float4 a = ring[(i & (2 * RC - 1)) * 2];
        return group_bound((int)(__float_as_uint(a.x) & 0x7fffffffu), a.y, a.z, a.w);
    };
    // cell-by-cell evaluation with the (-inf) - (-inf) := 0 convention (impossible current state, removal of the last occupied patch)
    auto evaluate_careful = [&](const Cand &cd, bool zero_after, bool own, int kj, uint32_t Ae, uint32_t Be) -> float {
        const float sgn = cd.cur ? -1.f : 1.f;
        float acc2 = 0.f;
        for (int j = 0; j < ept; j++) {
            const bool a = (Ae >> j) & 1u, b = (Be >> j) & 1u;
            if (!(a || b)) continue;
            const float4 tq = sTt[j * NT];
            const int s = g + j * TPT;
            const float w = weight(tq, cd.k, cd.kx, cd.ky, cd.lawk);
            const float sa = zero_after ? (float)src_offset(tl[s]) : fmaf(sgn, w, tq.x) + tq.y;
            acc2 += ldiff<float>(Num<float>::lg2(col_factor(cK, sa, a, b)), Num<float>::lg2(col_factor(cK, tq.x + tq.y, a, b)));
        }
        if (own) acc2 += own_term(kj, cd.cur);
        return acc2;
    };
    auto commit = [&](const Cand &cd, float wub, bool zero_after, bool own, int kj, uint32_t ownbit) {
        if (own) { ybits ^= ownbit; Amask ^= ownbit; }
        nocc += cd.cur ? -1 : 1;
        if (!zero_after) {
            const float sgn = cd.cur ? -1.f : 1.f;
            // groups where the weight exceeds 2^-36 min S: what is skipped stays far below the FP32 resolution of S even
            // when summed over every commit between two refreshes of S (at most 2^-36 x commits, in practice << 2^-30)
            const bool reach = lane < ept && !(wub < 1.4551915e-11f * Gw);
            // far part of the reach: every weight is below 2^-24 of the group's smallest S_hi, i.e. below half an ulp of each
            // S_hi -- the two-sum would put all of it into S_lo and leave S_hi (and the group minimum) as they are, so only S_lo is
            // touched.  |S_lo| stays below ~2^-13 S_hi between two normalising commits, far inside a float's exponent range of it.
            const bool far = reach && wub < 5.9604645e-8f * Gw;
            uint32_t m = __ballot_sync(0xffffffffu, reach && !far), mf = __ballot_sync(0xffffffffu, far);
            st_commit += __popc(m) + __popc(mf);
            // B slots per trip: B independent (LDS, sqrt, ex2, two-sum, STS) chains, the loop is latency bound otherwise
            auto batch = [&](auto BB) {
                constexpr int B = decltype(BB)::value;
                int jj[B];
                float4 tq[B];
#pragma unroll
                for (int u = 0; u < B; u++) { jj[u] = __ffs((int)m) - 1; m &= m - 1u; tq[u] = sTt[jj[u] * NT]; }
#pragma unroll
                for (int u = 0; u < B; u++) {
                    const int j = jj[u];
                    const float w = weight(tq[u], cd.k, cd.kx, cd.ky, cd.lawk);
                    const float a = j == kj ? 0.f : sgn * w;
                    const float s = tq[u].x + a, bb = s - tq[u].x;
                    const float e = (tq[u].x - (s - bb)) + (a - bb);
                    const float lo2 = tq[u].y + e;
                    float hi = s + lo2, lo = lo2 - (hi - s);
                    if (hi < 0.f) { hi = 0.f; lo = 0.f; }
                    *reinterpret_cast<float2 *>(&sTt[j * NT]) = make_float2(hi, lo);
                    if (cd.cur) {
                        // a removal lowers S: exact new minimum of the group (S_hi >= 0, so the bit pattern is order
                        // preserving); after an addition the old minimum is still a lower bound
                        const uint32_t mn = __reduce_min_sync(0xffffffffu, ((valid >> j) & 1u) ? (__float_as_uint(hi) & 0x7fffffffu) : 0x7f7fffffu);
                        if (lane == j) Gw = __uint_as_float(mn);
                    }
                }
            };
            while (m) {                                   // warp-uniform
                const int left = __popc(m);
                if (left >= 4) batch(std::integral_constant<int, 4>());
                else if (left == 3) batch(std::integral_constant<int, 3>());
                else if (left == 2) batch(std::integral_constant<int, 2>());
                else batch(std::integral_constant<int, 1>());
            }
            auto batch_far = [&](auto BB) {
                constexpr int B = decltype(BB)::value;
                int jj[B];
                float4 tq[B];
#pragma unroll
                for (int u = 0; u < B; u++) { jj[u] = __ffs((int)mf) - 1; mf &= mf - 1u; tq[u] = sTt[jj[u] * NT]; }
#pragma unroll
                for (int u = 0; u < B; u++) sTt[jj[u] * NT].y = fmaf(sgn, weight(tq[u], cd.k, cd.kx, cd.ky, cd.lawk), tq[u].y);
            };
            while (mf) {                                  // warp-uniform; the candidate's own group is never far (distance 0)
                const int left = __popc(mf);
                if (left >= 4) batch_far(std::integral_constant<int, 4>());
                else if (left == 3) batch_far(std::integral_constant<int, 3>());
                else if (left == 2) batch_far(std::integral_constant<int, 2>());
                else batch_far(std::integral_constant<int, 1>());
            }
        } else {
            for (int j = 0; j < ept; j++) {
                const int s = g + j * TPT;
                const double so = s < nl ? src_offset(tl[s]) : 0.0;
                const float hi = (float)so, lo = (float)(so - (double)hi);
                *reinterpret_cast<float2 *>(&sTt[j * NT]) = make_float2(hi, lo);
            }
            Gw = 0.f;
        }
        __syncwarp();
    };

    // ---- the scan.  Every trip evaluates SP consecutive candidates i .. i+SP-1 against the CURRENT state, in one pass over
    // the union of their active groups (candidates come in Morton order, so the sets nearly coincide; a slot that only some
    // of them feel contributes an exact factor ratio of 1 to the others) and one exchange of SP sums.  They are then
    // decided in order: candidate c's sum is valid as long as all before it were rejected (2 of 3 flips are), the first
    // accepted one is committed and the rest of the window is evaluated again on the next trip.  Decisions and state
    // are exactly those of the one-at-a-time scan.
    float wub[SP];
#pragma unroll
    for (int c = 0; c < SP; c++) wub[c] = c < ncand ? bound_of(c) : 0.f;
    for (int i = 0; i < ncand;) {
        if ((i / RC) != chunk) {                          // entered the next chunk: recycle the half we left
            chunk = i / RC;
            __syncthreads();
            if (tid < 2 * RC) ring[((chunk + 1) & 1) * 2 * RC + tid] = pre;
            __syncthreads();
            pre = load_chunk(chunk + 2);
        }
        const int nc = min(SP, ncand - i);
        float kx[SP], ky[SP], lawk[SP], sgn[SP], thr[SP], pn[SP], acc[NS];
        int kj[SP], kk[SP];
        bool zero[SP];
        bool feel = false;
#pragma unroll
        for (int c = 0; c < SP; c++) {
            const float4 a = ring[((i + c) & (2 * RC - 1)) * 2];
            const float4 rb = ring[((i + c) & (2 * RC - 1)) * 2 + 1];
            const int kslot = blk ? (int)__float_as_uint(rb.z) - slot_lo : (int)__float_as_uint(rb.y);
            const uint32_t cur = __float_as_uint(a.x) >> 31;
            kk[c] = (int)(__float_as_uint(a.x) & 0x7fffffffu);
            kx[c] = a.y; ky[c] = a.z; lawk[c] = a.w; sgn[c] = cur ? -1.f : 1.f; thr[c] = rb.x;
            kj[c] = (c < nc && (kslot % TPT) == g) ? kslot / TPT : 31;   // window entries past the list are zero records: no own cell
            zero[c] = (nocc + (cur ? -1 : 1)) == 0;
            pn[c] = 1.f; acc[c] = 0.f;
            // groups that can feel the candidate at the FP32 resolution of S_hi (2^-26 min S, with a margin for the drift
            // of min S in groups whose commits were skipped)
            feel = feel || (c < nc && !zero[c] && !(wub[c] < 1.4886e-8f * Gw));
        }
        uint32_t m = __ballot_sync(0xffffffffu, lane < ept && feel);
        const uint32_t nfeel = __popc(m);
        float pd = 1.f;
        int cnt = 0;
        // BR: product of the branch factors, and the cancellation cut of candidate 0 (a removal that leaves u0 = fl(S_hi - w0) below
        // S_hi / 4; an addition never cancels).  Above the cut u0 + S_lo is within ~2^-23 of S_hi + S_lo - w0 relative to itself
        // (|S_lo| < 2^-13 S_hi), the accuracy of the post-commit evaluation; below it S_lo and the commit's clamp at 0 matter
        float pn2 = 1.f;
        const float cut0 = sgn[0] < 0.f ? 0.25f : -1.f;
        if constexpr (BR) acc[SP] = 0.f;
        // B slots x SP candidates per trip: B * SP independent (sqrt, ex2, FFMA.SAT) chains
        auto slots = [&](auto BB) {
            constexpr int B = decltype(BB)::value;
            int jj[B];
            float4 tq[B];
#pragma unroll
            for (int u = 0; u < B; u++) { jj[u] = __ffs((int)m) - 1; m &= m - 1u; tq[u] = sTt[jj[u] * NT]; }
#pragma unroll
            for (int u = 0; u < B; u++) {
                const int j = jj[u];
                // class A (z'=1): sat(cK S); class B (z'=0): sat(1 - cK S); neither: 1 -- one FFMA.SAT with selected constants
                const bool a = (Amask >> j) & 1u, b = (Bmask >> j) & 1u;
                const float mul = a ? cK : (b ? -cK : 0.f), add = a ? 0.f : 1.f;
                const float fd = __saturatef(fmaf(mul, tq[u].x + tq[u].y, add));
                pd *= fd;
                float u0 = 0.f, fn0 = 1.f, w1 = 0.f;
#pragma unroll
                for (int c = 0; c < SP; c++) {
                    const float w = weight(tq[u], kk[c], kx[c], ky[c], lawk[c]);
                    const float uc = fmaf(sgn[c], w, tq[u].x);
                    const float fn = __saturatef(fmaf(mul, uc + tq[u].y, add));
                    pn[c] *= j == kj[c] ? fd : fn;        // the candidate's own cell is handled by own_term
                    if (c == 0) { u0 = uc; fn0 = fn; }
                    if (c == 1) w1 = w;
                }
                if constexpr (BR) {
                    // candidate 1 after candidate 0's commit: numerator fn(S + sgn0 w0 + sgn1 w1); the denominator fn(S + sgn0 w0) is fn0,
                    // already in pn[0].  At candidate 0's own cell (S unchanged, class flipped) and at candidate 1's own cell the
                    // factors cancel, the owners add those cells' terms after the loop
                    const float f2 = u0 < cut0 * tq[u].x ? __int_as_float(0x7fffffff)
                                                         : __saturatef(fmaf(mul, fmaf(sgn[1], w1, u0) + tq[u].y, add));
                    pn2 *= j == kj[0] ? fd : (j == kj[1] ? fn0 : f2);
                }
            }
            cnt += B;
        };
        while (m) {                                       // warp-uniform
            if (SP <= 2 && (m & (m - 1u))) slots(std::integral_constant<int, 2>());
            else slots(std::integral_constant<int, 1>());
            if (cnt >= 4 || m == 0u) {                    // products of at most 4 factors stay far from underflow
                const float lpd = Num<float>::lg2(pd);
                float lpn[SP];
#pragma unroll
                for (int c = 0; c < SP; c++) { lpn[c] = Num<float>::lg2(pn[c]); acc[c] += lpn[c] - lpd; pn[c] = 1.f; }
                if constexpr (BR) { acc[SP] += Num<float>::lg2(pn2) - lpn[0]; pn2 = 1.f; }
                pd = 1.f; cnt = 0;
            }
        }
#pragma unroll
        for (int c = 0; c < SP; c++) if (kj[c] != 31) acc[c] += own_term(kj[c], sgn[c] < 0.f);
        if constexpr (BR) {
            if (kj[1] != 31) {                            // candidate 1's own cell, S after candidate 0's commit (same cut)
                const float4 tq = sTt[kj[1] * NT];
                const float u = fmaf(sgn[0], weight(tq, kk[0], kx[0], ky[0], lawk[0]), tq.x);
                acc[SP] += u < cut0 * tq.x ? __int_as_float(0x7fffffff) : own_term_s(u + tq.y, sgn[1] < 0.f);
            }
            if (kj[0] != 31 && sgn[0] < 0.f) {            // candidate 0's own cell: its removal makes it class A with S unchanged
                const float4 tq = sTt[kj[0] * NT];
                const float w = weight(tq, kk[1], kx[1], ky[1], lawk[1]);
                acc[SP] += Num<float>::lg2(__saturatef(cK * (fmaf(sgn[1], w, tq.x) + tq.y))) - Num<float>::lg2(__saturatef(cK * (tq.x + tq.y)));
            }
        }
        // bounds of the SP candidates after this window: independent of this trip's outcome, they complete under the reduction
        float nxt[SP];
#pragma unroll
        for (int c = 0; c < SP; c++) nxt[c] = bound_of(i + SP + c);
        all_reduce(0, acc);

        int adv = nc;
        if constexpr (BR) {
            // candidate 0 as below; candidate 1 from its own sum if 0 is rejected, from the branch sum if 0 is accepted.  The branch
            // is deferred (adv = 1) when it is NaN (cut, or a zero factor), when candidate 0 took the careful path, and when
            // candidate 1 would take it with or without 0's flip (the last occupied patch leaving)
            bool take[SP];
#pragma unroll
            for (int c = 0; c < SP; c++) {
                take[c] = false;
                if (c >= nc) continue;
                float tot = acc[c];
                if (c == 1 && take[0]) {
                    tot = acc[SP];
                    const bool ok = !zero[0] && !isnan(acc[0]) && !zero[1] && nocc + (sgn[0] < 0.f ? -1 : 1) + (sgn[1] < 0.f ? -1 : 1) != 0;
                    if (!ok || isnan(tot)) { adv = 1; continue; }
                } else if (zero[c] || isnan(tot)) {
                    const uint32_t bit = kj[c] != 31 ? 1u << kj[c] : 0u;
                    float v[NS] = {};
                    v[0] = evaluate_careful(Cand{ kk[c], sgn[c] < 0.f, kx[c], ky[c], lawk[c] }, zero[c], kj[c] != 31, kj[c], Amask & ~bit, Bmask);
                    all_reduce(1, v);
                    tot = v[0];
                }
                take[c] = thr[c] < 0.6931471805599453f * tot;
            }
            // commits in order, one inlined copy of the commit (warp-uniform)
#pragma unroll 1
            for (int c = 0; c < SP; c++) {
                if (!(c ? take[1] : take[0])) continue;
                const int kjc = c ? kj[1] : kj[0];
                commit(c ? Cand{ kk[1], sgn[1] < 0.f, kx[1], ky[1], lawk[1] } : Cand{ kk[0], sgn[0] < 0.f, kx[0], ky[0], lawk[0] },
                       c ? wub[1] : wub[0], c ? zero[1] : zero[0], kjc != 31, kjc, kjc != 31 ? 1u << kjc : 0u);
            }
        } else {
            // decisions in order, from the window's registers; the accepted entry ca (if any) ends the window and is committed once
            int ca = -1;
#pragma unroll
            for (int c = 0; c < SP; c++) {
                if (c < adv) {                                // still undecided and inside the list (adv shrinks on the first accept)
                    float tot = acc[c];
                    if (zero[c] || isnan(tot)) {
                        const uint32_t bit = kj[c] != 31 ? 1u << kj[c] : 0u;
                        float v[SP];
#pragma unroll
                        for (int d = 0; d < SP; d++) v[d] = 0.f;
                        v[0] = evaluate_careful(Cand{ kk[c], sgn[c] < 0.f, kx[c], ky[c], lawk[c] }, zero[c], kj[c] != 31, kj[c], Amask & ~bit, Bmask);
                        all_reduce(1, v);
                        tot = v[0];
                    }
                    if (thr[c] < 0.6931471805599453f * tot) { ca = c; adv = c + 1; }
                }
            }
            if (ca >= 0) {                                    // warp-uniform: every lane holds the task's sums
                Cand cd{ kk[0], sgn[0] < 0.f, kx[0], ky[0], lawk[0] };
                float wb = wub[0];
                bool zr = zero[0];
                int kjc = kj[0];
#pragma unroll
                for (int c = 1; c < SP; c++)
                    if (ca == c) { cd = Cand{ kk[c], sgn[c] < 0.f, kx[c], ky[c], lawk[c] }; wb = wub[c]; zr = zero[c]; kjc = kj[c]; }
                commit(cd, wb, zr, kjc != 31, kjc, kjc != 31 ? 1u << kjc : 0u);
            }
        }
        i += adv;
        st_trips++; st_exec += nfeel * (uint32_t)nc; st_ret += nfeel * (uint32_t)adv;
        // slide the window of bounds by adv
#pragma unroll
        for (int aa = 1; aa <= SP; aa++)
            if (adv == aa) {
#pragma unroll
                for (int c = 0; c < SP; c++) wub[c] = aa + c < SP ? wub[(aa + c) % SP] : nxt[(aa + c - SP) % SP];
            }
    }
    for (int j = 0; j < ept; j++) {
        const int s = g + j * TPT;
        if (s < nl) {
            const int q = tl[s];
            const float4 tq = sT[tid + j * NT];
            St[q] = fmax(((double)tq.x + (double)tq.y) - src_offset(q), 0.0);
            yt[q] = (uint8_t)((ybits >> j) & 1u);
        }
    }
    if (stats && lane == 0) {
        atomicAdd(&stats[MP_CNT_SCAN_TRIPS], (unsigned long long)st_trips);
        atomicAdd(&stats[MP_CNT_SCAN_EXEC], (unsigned long long)st_exec);
        atomicAdd(&stats[MP_CNT_SCAN_RETIRED], (unsigned long long)st_ret);
        atomicAdd(&stats[MP_CNT_SCAN_COMMIT], (unsigned long long)st_commit);
        if (btasks && tid == 0 && rank == 0) atomicAdd(&stats[MP_CNT_SCAN_BLOCKS], 1ull);
    }
    if (CS > 1) cluster_barrier();
}

// Which (chain, year) tasks may be scanned block by block this sweep (mp_set_scan_blocks).  A block task leaves out every
// target farther than the halo from its cell; that is the culled scan's own commit rule (weights below 2^-36 of the
// target group's smallest S are not applied) as long as the largest weight at the halo distance, max_k A_k^b exp(-alpha halo),
// stays below 2^-36 of the year's smallest S.  The year must also hold enough occupied patches that "the last occupied
// patch left" (which the whole-task scan treats exactly) cannot arise while blocks change the count concurrently.
// The decision depends on the task's own data only, so it is the same however the tasks are sharded over engines.
static __global__ void __launch_bounds__(256)
k_block_valid(const double *__restrict__ S, const mp_params *__restrict__ par, const int *__restrict__ count, int n, int ntrans,
              int task_first, int task_stride, double halo, double log2_area_max, double log2_area_min, int *__restrict__ blockmode)
{
    __shared__ double s_min[8];
    const int task = task_first + blockIdx.x * task_stride, c = task / ntrans;
    const double *St = S + (size_t)task * n;
    double m = 1e300;
    for (int q = threadIdx.x; q < n; q += 256) m = fmin(m, St[q]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmin(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) s_min[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++) m = fmin(m, s_min[w]);
        const double b = par[c].b, law = b >= 0.0 ? b * log2_area_max : b * log2_area_min;
        const double wmax = exp2(law - par[c].alpha * halo * 1.4426950408889634);
        blockmode[task] = (wmax < 1.4551915228366852e-11 * m && count[2 * task + 1] >= 64) ? 1 : 0;
    }
}

}  // namespace mp

#if defined(MP_FAST_GEOM) && defined(MP_FAST_HAS_POSITIONS)
namespace mp {
// nclusters whole (chain, year) tasks (btasks == nullptr) or block tasks of one colour
template <int CS, int TPT> static int launch_cull(mp_engine *h, int ept, int nclusters, const BlockTask *btasks)
{
    constexpr int NT = TPT / CS;
    const size_t smem = (size_t)ept * NT * 16 + 2 * 32 * 32;   // targets + the two-chunk record ring
    REQUIRE(smem <= 227 * 1024 && ept <= 31, MP_ERR_UNSUPPORTED, "n_patches too large for the fast y sweep");
    auto kern = k_sweep_y_cull<MP_FAST_GEOM, CS, TPT>;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (CS > 8) CK(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    if (nclusters <= 0) return MP_OK;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(nclusters * CS));
    cfg.blockDim = dim3(NT);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = h->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = CS > 1 ? 1 : 0;
    CK(cudaLaunchKernelEx(&cfg, kern, view<float>(h), (const int *)h->d_perm, (const mp_params *)h->d_par,
                          (const uint8_t *)(h->have_era ? h->d_era : nullptr), (const uint8_t *)h->d_z, h->d_y, h->d_S[0],
                          (const CandRec *)h->d_cand, (const int *)h->d_cand_count, h->cfg.n_years, ept, (const int *)h->d_task_order,
                          h->d_work, btasks, (const int *)h->d_tlist, (const int *)(h->blk_active ? h->d_blockmode : nullptr)));
    return MP_OK;
}
// culled variants exist for 512 and 1024 threads per task (up to 31 slots per thread) and the large-landscape geometries
static int launch_cull_any(mp_engine *h, int cs, int tpt, int nl_max, int nclusters, const void *btasks_v)
{
    const BlockTask *btasks = (const BlockTask *)btasks_v;
    const int ept = (nl_max + tpt - 1) / tpt;
    if (tpt == 512) switch (cs) {
        case 1: return launch_cull<1, 512>(h, ept, nclusters, btasks);
        case 2: return launch_cull<2, 512>(h, ept, nclusters, btasks);
        case 4: return launch_cull<4, 512>(h, ept, nclusters, btasks);
        default: return launch_cull<8, 512>(h, ept, nclusters, btasks);
    }
    if (tpt == 1024) switch (cs) {
        case 1: return launch_cull<1, 1024>(h, ept, nclusters, btasks);
        case 2: return launch_cull<2, 1024>(h, ept, nclusters, btasks);
        case 4: return launch_cull<4, 1024>(h, ept, nclusters, btasks);
        default: return launch_cull<8, 1024>(h, ept, nclusters, btasks);
    }
    if (tpt == 2048) return launch_cull<8, 2048>(h, ept, nclusters, btasks);
    if (tpt == 4096) return cs == 16 ? launch_cull<16, 4096>(h, ept, nclusters, btasks) : launch_cull<8, 4096>(h, ept, nclusters, btasks);
    if (tpt == 8192) return cs == 16 ? launch_cull<16, 8192>(h, ept, nclusters, btasks) : launch_cull<8, 8192>(h, ept, nclusters, btasks);
    return MP_ERR_UNSUPPORTED;
}
}  // namespace mp
#endif
