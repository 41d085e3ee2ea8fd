// mp_capacity.cuh -- kernels of mp_capacity: the metapopulation capacity lambda_M of the landscape (Hanski & Ovaskainen 2000),
// the leading eigenvalue of the symmetric landscape matrix
//     M~_kl = sqrt(a_k a_l) exp(-alpha d_kl)  (k != l),  M~_kk = 0,  a = A^b,
// found by LOBPCG with block size 1 (the host loop in mp_engine.cu; DESIGN.md §2, §4).  One call holds a batch of parameter
// sets; every vector lives in layout (Morton) order, [set][vector][padded slot], FP64.
//
//  k_cap_prep   per (set, slot): the set's area constant h = (1/2) log2 A^b (FP32) / s = sqrt(A^b) (FP64), -inf / 0 for removed
//               patches, and the start vector (1 on kept patches); set 0 also writes the positions in layout order
//  k_cap_mv     u = M~ v for every active set in one launch: one target per thread, source tiles of CAP_NT staged in shared
//               memory, FP64 accumulation over the sources in ascending slot order (bit-identical for any grid).  The weight is
//               exactly symmetric in both precisions: FP32 ex2(fma(apre, d, h_k + h_l)), FP64 exp(-(alpha d)) (s_k s_l).
//               CULL (FP32 engines, landscapes with positions): a (target group, source group) tile of 32 x 32 slots is
//               skipped when the box32 bound of its largest weight is below the set's floor; the decision is symmetric in
//               the two groups, so the culled operator stays symmetric.  The row sum of the skipped weights of every target
//               group is bounded in the same pass (atomicMax of a non-negative float: order-independent).
//  k_cap_gram   the 2 x 6 inner products of the Rayleigh-Ritz step over {x, r, p} and {Ax, Ar, Ap}
//  k_cap_update x <- cx x + cr r + cp p (and Ax alike), p <- cr r + cp p (and Ap alike), r <- Ax - mu x; sums x.x, x.Ax, r.r
// The two reductions run over fixed chunks of CAP_CHUNK slots with a fixed block size and leave one partial per (set, chunk);
// the host adds the chunks in order.  No floating-point atomics anywhere: a set's results depend on nothing but its own inputs.
#pragma once
#include "mp_device.cuh"

namespace mp {

constexpr int CAP_NT = 128;        // threads (targets) per CTA of k_cap_mv and sources per shared-memory tile
constexpr int CAP_RT = 256;        // threads of the reduction kernels
constexpr int CAP_CHUNK = 4096;    // slots per partial sum of the reduction kernels
constexpr int CAP_NVEC = 6;        // x, r, p, Ax, Ar, Ap
enum { CAP_X = 0, CAP_R = 1, CAP_P = 2, CAP_AX = 3, CAP_AR = 4, CAP_AP = 5 };
constexpr int CAP_NGRAM = 12;      // x.Ax x.Ar x.Ap r.Ar r.Ap p.Ap | x.x x.r x.p r.r r.p p.p

// one active parameter set of a launch (uploaded by the host every iteration)
struct CapSet {
    double alpha;          // dispersal rate of the set
    double cx, cr, cp, mu; // k_cap_update: coefficients of the new x and Ritz value
    float thr;             // k_cap_mv: skip a tile when log2 of its distance factor is below thr (-inf: never)
    float lamax;           // log2 of max_l A_l^b (bound of the skipped weights)
    int set;               // the set's index in the call's batch
    int pad;
};

template <typename R> struct CapArgs {
    Landscape<R> ls;               // positions as uploaded (patch order); dist for dense landscapes
    const CapSet *cs;              // [active set]
    const R *lx, *ly;              // positions in layout order [npad]
    const R *hs;                   // area constants [set][npad]
    double *vec;                   // [set][CAP_NVEC][npad]
    const float4 *box32;           // bounding box of every group of 32 layout slots
    unsigned *bound;               // [set] bits of the largest row-sum bound of the skipped weights (non-negative float)
    unsigned long long *stats;     // MP_CNT_CONN_EXEC / MP_CNT_CONN_TOTAL
    int npad;
};

inline __host__ __device__ int cap_npad(int n) { return (n + CAP_NT - 1) / CAP_NT * CAP_NT; }

// grid (npad / 256, sets)
template <typename R>
__global__ void k_cap_prep(Landscape<R> ls, const int *__restrict__ perm, const double *__restrict__ area, const uint8_t *__restrict__ keep,
                           const double *__restrict__ b, int npad, R *__restrict__ lx, R *__restrict__ ly, R *__restrict__ hs,
                           double *__restrict__ vec)
{
    const int slot = blockIdx.x * blockDim.x + threadIdx.x, set = blockIdx.y;
    if (slot >= npad) return;
    const int q = slot < ls.n ? perm[slot] : -1;
    const bool kept = q >= 0 && (!keep || keep[q]);
    const double A = area && q >= 0 ? area[q] : 1.0;
    R hv;
    if (sizeof(R) == 4) hv = kept ? (R)(0.5 * b[set] * log2(A)) : (R)-INFINITY;
    else hv = kept ? (R)sqrt(pow(A, b[set])) : (R)0;
    hs[(size_t)set * npad + slot] = hv;
    vec[((size_t)set * CAP_NVEC + CAP_X) * npad + slot] = kept ? 1.0 : 0.0;
    if (set == 0) {
        lx[slot] = q >= 0 && ls.px ? ls.px[q] : (R)0;
        ly[slot] = q >= 0 && ls.py ? ls.py[q] : (R)0;
    }
}

template <typename R, int GEOM>
__device__ __forceinline__ double cap_weight(const Landscape<R> &ls, R apre, int k, int l, R tx, R ty, R hk, R sx, R sy, R hl)
{
    const R d = pair_distance<R, GEOM>(ls, k, l, tx, ty, sx, sy);
    if constexpr (sizeof(R) == 4) return (double)Num<float>::ex2(fmaf(apre, d, hk + hl));
    else return exp(-(apre * d)) * (hk * hl);
}

// grid (npad / CAP_NT, active sets); u[set][vout] = M~ v[set][vin]
template <typename R, int GEOM, bool CULL>
__global__ void __launch_bounds__(CAP_NT) k_cap_mv(CapArgs<R> a, int vin, int vout)
{
    constexpr int NG = CAP_NT / 32;                                   // groups of 32 sources per tile
    __shared__ R sx[CAP_NT], sy[CAP_NT], sh[CAP_NT];
    __shared__ double sv[CAP_NT];
    const CapSet cs = a.cs[blockIdx.y];
    const int n = a.ls.n, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int k = blockIdx.x * CAP_NT + tid, kc = min(k, n - 1);     // target slot (a thread past the end evaluates the last one)
    const R *hs = a.hs + (size_t)cs.set * a.npad;
    const double *v = a.vec + ((size_t)cs.set * CAP_NVEC + vin) * a.npad;
    const R apre = alpha_pre<R>(cs.alpha);
    const R tx = a.lx[kc], ty = a.ly[kc], hk = hs[kc];
    const int ngroups = (n + 31) / 32, g = blockIdx.x * NG + wid;   // the warp's target group
    const bool gvalid = g < ngroups;
    float4 gbox = make_float4(0.f, 0.f, 0.f, 0.f);
    if (CULL) gbox = a.box32[min(g, ngroups - 1)];
    double acc = 0.0;
    float bound = 0.f;                                                // row-sum bound of the weights this warp skips
    uint32_t nexec = 0;
    for (int l0 = 0; l0 < n; l0 += CAP_NT) {
        bool far[NG];
#pragma unroll
        for (int s = 0; s < NG; s++) far[s] = false;
        if (CULL) {
            bool need = false;
#pragma unroll
            for (int s = 0; s < NG; s++) {
                const int sg = l0 / 32 + s;
                if (sg >= ngroups) continue;
                const float4 sb = a.box32[sg];
                const float dx = fmaxf(0.f, fmaxf(sb.x - gbox.y, gbox.x - sb.y)), dy = fmaxf(0.f, fmaxf(sb.z - gbox.w, gbox.z - sb.w));
                const float r2 = (float)apre * (0.9999f * sqrtf(dx * dx + dy * dy));   // log2 of the largest exp(-alpha d), rounded up
                far[s] = r2 < cs.thr;
                if (far[s] && gvalid) bound += (float)min(32, n - 32 * sg) * exp2f(r2 + cs.lamax);
                need = need || (!far[s] && gvalid);
            }
            if (!__syncthreads_or(need)) continue;                    // also the barrier that frees the previous tile
        } else if (l0 > 0) {
            __syncthreads();
        }
        {
            const int l = l0 + tid;
            const bool in = l < n;
            sx[tid] = in ? a.lx[l] : (R)0; sy[tid] = in ? a.ly[l] : (R)0;
            sh[tid] = in ? hs[l] : (sizeof(R) == 4 ? (R)-INFINITY : (R)0);
            sv[tid] = in ? v[l] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int s = 0; s < NG; s++) {
            if (l0 + 32 * s >= n || far[s]) continue;                 // warp-uniform
            nexec += gvalid;
#pragma unroll 8
            for (int j = 32 * s; j < 32 * s + 32; j++) {
                const int l = l0 + j;                                  // padding sources (l >= n) weigh 0 through sh; min: in-bounds distances
                double w = cap_weight<R, GEOM>(a.ls, apre, kc, min(l, n - 1), tx, ty, hk, sx[j], sy[j], sh[j]);
                if (l == k) w = 0.0;                                  // M~_kk = 0
                acc = fma(w, sv[j], acc);
            }
        }
    }
    if (k < n) a.vec[((size_t)cs.set * CAP_NVEC + vout) * a.npad + k] = acc;
    if (lane == 0 && gvalid) {
        if (CULL && bound > 0.f) atomicMax(&a.bound[cs.set], __float_as_uint(bound));
        if (a.stats) {
            atomicAdd(&a.stats[MP_CNT_CONN_EXEC], (unsigned long long)nexec);
            atomicAdd(&a.stats[MP_CNT_CONN_TOTAL], (unsigned long long)ngroups);
        }
    }
}

// K partial sums of one (chunk, set) in a fixed order: warps by shuffles, then the warps' sums in order by thread i < K
template <int K>
__device__ __forceinline__ void cap_chunk_sum(double (&s)[K], double *__restrict__ out)
{
    __shared__ double ws[CAP_RT / 32][K];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < K; i++) {
        const double t = warp_sum(s[i]);
        if (lane == 0) ws[w][i] = t;
    }
    __syncthreads();
    if (threadIdx.x < K) {
        double t = 0.0;
        for (int j = 0; j < CAP_RT / 32; j++) t += ws[j][threadIdx.x];
        out[threadIdx.x] = t;
    }
}

// grid (chunks, active sets); part[active][chunk][CAP_NGRAM]
static __global__ void __launch_bounds__(CAP_RT) k_cap_gram(const CapSet *__restrict__ cs, const double *__restrict__ vec, int n, int npad,
                                                            double *__restrict__ part)
{
    const double *V = vec + (size_t)cs[blockIdx.y].set * CAP_NVEC * npad;
    double s[CAP_NGRAM];
#pragma unroll
    for (int i = 0; i < CAP_NGRAM; i++) s[i] = 0.0;
    const int i1 = min(n, (blockIdx.x + 1) * CAP_CHUNK);
    for (int i = blockIdx.x * CAP_CHUNK + threadIdx.x; i < i1; i += CAP_RT) {
        const double x = V[i], r = V[npad + i], p = V[2 * npad + i], ax = V[3 * npad + i], ar = V[4 * npad + i], ap = V[5 * npad + i];
        s[0] = fma(x, ax, s[0]); s[1] = fma(x, ar, s[1]); s[2] = fma(x, ap, s[2]);
        s[3] = fma(r, ar, s[3]); s[4] = fma(r, ap, s[4]); s[5] = fma(p, ap, s[5]);
        s[6] = fma(x, x, s[6]); s[7] = fma(x, r, s[7]); s[8] = fma(x, p, s[8]);
        s[9] = fma(r, r, s[9]); s[10] = fma(r, p, s[10]); s[11] = fma(p, p, s[11]);
    }
    cap_chunk_sum<CAP_NGRAM>(s, part + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * CAP_NGRAM);
}

// grid (chunks, active sets); part[active][chunk][3] = x.x, x.Ax, r.r of the updated vectors
static __global__ void __launch_bounds__(CAP_RT) k_cap_update(const CapSet *__restrict__ cs, double *__restrict__ vec, int n, int npad,
                                                              double *__restrict__ part)
{
    const CapSet c = cs[blockIdx.y];
    double *V = vec + (size_t)c.set * CAP_NVEC * npad;
    double s[3] = { 0.0, 0.0, 0.0 };
    const int i1 = min(n, (blockIdx.x + 1) * CAP_CHUNK);
    for (int i = blockIdx.x * CAP_CHUNK + threadIdx.x; i < i1; i += CAP_RT) {
        const double x = V[i], r = V[npad + i], p = V[2 * npad + i], ax = V[3 * npad + i], ar = V[4 * npad + i], ap = V[5 * npad + i];
        const double pn = c.cr * r + c.cp * p, apn = c.cr * ar + c.cp * ap;
        const double xn = c.cx * x + pn, axn = c.cx * ax + apn;
        const double rn = axn - c.mu * xn;
        V[i] = xn; V[npad + i] = rn; V[2 * npad + i] = pn; V[3 * npad + i] = axn; V[5 * npad + i] = apn;
        s[0] = fma(xn, xn, s[0]); s[1] = fma(xn, axn, s[1]); s[2] = fma(rn, rn, s[2]);
    }
    cap_chunk_sum<3>(s, part + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 3);
}

// dense landscapes: flag[0] = 1 when some d[i][j] != d[j][i]; grid (n / 256, rows i, i += gridDim.y)
template <typename R>
__global__ void k_cap_symcheck(const R *__restrict__ dist, int n, int *__restrict__ flag)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    for (int i = blockIdx.y; i < n; i += gridDim.y)
        if (j < n && j > i && dist[(size_t)i * n + j] != dist[(size_t)j * n + i]) atomicOr(flag, 1);
}

}  // namespace mp
