// mp_device.cuh -- device-side building blocks of the SPOM engine (sm_100a).
//
// Model (Appendix B of SURVEY.md; reference lines in /root/reference/sources/):
//   weight  w(k<-l) = exp(-alpha d_kl) A_l^b            main_MIDASPOM.c:184 (M), no areas there
//   S_tk    = sum_{l!=k} w(k<-l) y_tl                    main_MIDASPOM.c:351-355
//   E_t     = min(1, e/K_t)                              main_MIDASPOM.c:21-22, dieoff.c:56-57
//   C_tk    = min(1, c (K_t S_tk + Ksrc_t g_k))          main_MIDASPOM.c:356-357, dieoff.c:78-79, loss.c:98-100
//   g_k     = exp(-alpha u_k dsrc)                       loss.c:365, future.c:277
// with K_t = K, Ksrc_t = Ksrc on pre-event transitions (era flag) and 1, 0 otherwise.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/libmidaspom_cuda.h"

namespace mp {

// ------------------------------------------------------------------ Philox4x32-10
// Counter-based RNG (Salmon et al., SC'11): the stream of a chain depends only on
// (seed, global chain id, sweep, kind, cell) -- never on grid/block geometry.
enum : uint32_t { RK_INIT_PARAM = 1, RK_INIT_Z = 2, RK_SIM_EXT = 3, RK_SIM_COL = 4, RK_Z = 5, RK_Y = 6,
                  RK_AB = 7, RK_C = 8, RK_E = 9, RK_P = 10, RK_K = 11, RK_KSRC = 12, RK_DSRC = 13,
                  RK_PPC_DET = 14 };

__host__ __device__ inline uint32_t mulhi32(uint32_t a, uint32_t b)
{
#ifdef __CUDA_ARCH__
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
__host__ __device__ inline uint4 philox4x32_10(uint4 c, uint2 k)
{
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint32_t h0 = mulhi32(0xD2511F53u, c.x), l0 = 0xD2511F53u * c.x;
        const uint32_t h1 = mulhi32(0xCD9E8D57u, c.z), l1 = 0xCD9E8D57u * c.z;
        c = make_uint4(h1 ^ c.y ^ k.x, l1, h0 ^ c.w ^ k.y, l0);
        k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
    }
    return c;
}
__host__ __device__ inline uint4 rng(uint64_t seed, uint32_t chain, uint32_t sweep, uint32_t kind, uint32_t a, uint32_t b)
{
    return philox4x32_10(make_uint4(a, b, kind, sweep), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) + chain));
}
__host__ __device__ inline double u01(uint32_t x) { return ((double)x + 0.5) * (1.0 / 4294967296.0); }
// Gibbs draws compare logit(u) with the log-odds d:  u < 1/(1+exp(-d))  <=>  log(u/(1-u)) < d
__host__ __device__ inline double logit_u(uint32_t x) { const double u = u01(x); return log(u) - log1p(-u); }
__host__ __device__ inline void box_muller(uint32_t x0, uint32_t x1, double &n1, double &n2)
{
    const double r = sqrt(-2.0 * log(u01(x0)));
    const double th = 6.283185307179586476925286766559 * u01(x1);
    n1 = r * cos(th); n2 = r * sin(th);
}

// ------------------------------------------------------------------ arithmetic traits
// FP64: libdevice exp/log (<= 1 ulp) -- the 1e-9 parity path.
// FP32: MUFU.EX2 / MUFU.LG2 / MUFU.RSQ approximations -- the throughput path (1e-5).
template <typename R> struct Num;
template <> struct Num<double> {
    static __device__ __forceinline__ double exp_neg(double ax) { return exp(-ax); }          // exp(-ax)
    static __device__ __forceinline__ double logv(double x) { return log(x); }
    static __device__ __forceinline__ double log1m(double c) { return log1p(-c); }
    static __device__ __forceinline__ double sqrtv(double x) { return sqrt(x); }
    static __device__ __forceinline__ double powv(double a, double b) { return pow(a, b); }
};
template <> struct Num<float> {
    static __device__ __forceinline__ float ex2(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
    static __device__ __forceinline__ float lg2(float x) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
    static __device__ __forceinline__ float exp_neg(float ax) { return ex2(-1.4426950408889634f * ax); }
    static __device__ __forceinline__ float logv(float x) { return 0.6931471805599453f * lg2(x); }
    static __device__ __forceinline__ float log1m(float c) { return 0.6931471805599453f * lg2(1.0f - c); }
    static __device__ __forceinline__ float sqrtv(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
    static __device__ __forceinline__ float powv(float a, float b) { return (float)pow((double)a, (double)b); }
};

// ------------------------------------------------------------------ landscape view
template <typename R> struct Landscape {
    int n;
    R spacing;                 // MP_GEOM_LINEAR
    const R *px, *py;          // MP_GEOM_COORDS
    const R *dist;             // MP_GEOM_DENSE, [source][target]
    const double *src_unit;    // nullable => k+1
};

// Dispersal weight of a (target, source) pair, w = A_source^b exp(-alpha d(target, source)).
// The two per-chain / per-source constants are passed pre-transformed so that EVERY kernel of a
// precision evaluates the identical expression (a weight added by one kernel and removed by
// another must cancel exactly):
//   FP64: apre = alpha,            awv = A^b        w = exp(-(alpha d)) * A^b        (oracle order)
//   FP32: apre = -alpha log2(e),   awv = log2(A^b)  w = ex2(fma(apre, d, awv))        (one FFMA + MUFU.EX2)
template <typename R> __device__ __forceinline__ R alpha_pre(double alpha);
template <> __device__ __forceinline__ double alpha_pre<double>(double alpha) { return alpha; }
template <> __device__ __forceinline__ float alpha_pre<float>(double alpha) { return -1.4426950408889634f * (float)alpha; }
template <typename R> __device__ __forceinline__ R area_pre(double aw);
template <> __device__ __forceinline__ double area_pre<double>(double aw) { return aw; }
template <> __device__ __forceinline__ float area_pre<float>(double aw) { return (float)log2(aw); }

__device__ __forceinline__ double weight_of(double apre, double awv, double d) { return exp(-(apre * d)) * awv; }
__device__ __forceinline__ float weight_of(float apre, float awv, float d) { return Num<float>::ex2(fmaf(apre, d, awv)); }

template <typename R, int GEOM>
__device__ __forceinline__ R pair_distance(const Landscape<R> &ls, int target, int source, R tx, R ty, R sx, R sy)
{
    if (GEOM == MP_GEOM_LINEAR) {
        const int gap = target > source ? target - source : source - target;
        return (R)gap * ls.spacing;
    } else if (GEOM == MP_GEOM_COORDS) {
        const R dx = tx - sx, dy = ty - sy;
        return Num<R>::sqrtv(fma(dx, dx, dy * dy));      // explicit FMA: identical in every kernel
    } else {
        return ls.dist[(size_t)source * ls.n + target];
    }
}
// reference order for the linear geometry in FP64: exp(((-a)*(j-i))*d)  (main_MIDASPOM.c:184)
template <typename R, int GEOM>
__device__ __forceinline__ R pair_weight(const Landscape<R> &ls, R apre, R awv, int target, int source, R tx, R ty, R sx, R sy)
{
    if (GEOM == MP_GEOM_LINEAR && sizeof(R) == 8) {
        const int gap = target > source ? target - source : source - target;
        return (R)(exp(-((double)apre * (double)gap) * (double)ls.spacing) * (double)awv);
    }
    return weight_of(apre, awv, pair_distance<R, GEOM>(ls, target, source, tx, ty, sx, sy));
}

// per-chain derived constants of one transition
template <typename R> struct Trans {
    R c, Kt, Ks, E, logE, log1mE, alpha, dsrc;
    int src;     // external source active on this transition
};
template <typename R>
__device__ __forceinline__ Trans<R> make_trans(const mp_params &p, int pre)
{
    Trans<R> t;
    t.c = (R)p.c; t.alpha = (R)p.alpha; t.dsrc = (R)p.dsrc;
    t.Kt = pre ? (R)p.K : (R)1; t.Ks = pre ? (R)p.Ksrc : (R)0;
    double E = pre ? p.e / p.K : p.e;
    if (E > 1.0) E = 1.0;
    t.E = (R)E; t.logE = (R)log(E); t.log1mE = (R)log(1.0 - E);
    t.src = pre && p.Ksrc != 0.0;
    return t;
}
// branch-free choice between the post-event (a) and pre-event (b) constants of a chain
template <typename R>
__device__ __forceinline__ Trans<R> pick_trans(const Trans<R> &a, const Trans<R> &b, bool pre)
{
    Trans<R> t;
    t.c = a.c; t.alpha = a.alpha; t.dsrc = a.dsrc;
    t.Kt = pre ? b.Kt : a.Kt; t.Ks = pre ? b.Ks : a.Ks; t.E = pre ? b.E : a.E;
    t.logE = pre ? b.logE : a.logE; t.log1mE = pre ? b.log1mE : a.log1mE; t.src = pre ? b.src : a.src;
    return t;
}
template <typename R>
__device__ __forceinline__ R source_term(const Landscape<R> &ls, const Trans<R> &tr, int k)
{
    if (!tr.src) return (R)0;
    const R u = ls.src_unit ? (R)ls.src_unit[k] : (R)(k + 1);
    return Num<R>::exp_neg((tr.alpha * u) * tr.dsrc);
}
template <typename R>
__device__ __forceinline__ R col_prob(const Trans<R> &tr, R S, R g)
{
    R C = tr.src || tr.Kt != (R)1 ? tr.c * (tr.Kt * S + tr.Ks * g) : tr.c * S;
    return C > (R)1 ? (R)1 : C;
}
// log of the colonisation factor of a cell with y=0: z'=1 -> log C ; z'=0 -> log(1-C)
template <typename R>
__device__ __forceinline__ R log_col(int znext, R C) { return znext ? Num<R>::logv(C) : Num<R>::log1m(C); }

// (-inf) - (-inf) := 0, finite - (-inf) := +inf  (same convention as the oracle's ldiff)
template <typename R>
__device__ __forceinline__ R ldiff(R alt, R cur)
{
    if (cur == -INFINITY) return alt == -INFINITY ? (R)0 : (R)INFINITY;
    return alt - cur;
}

// ------------------------------------------------------------------ block reductions (fixed order => deterministic)
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// all threads receive the total; scratch must hold >= 32 doubles; contains one __syncthreads
__device__ __forceinline__ double block_sum(double v, double *scratch)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    if (lane == 0) scratch[w] = v;
    __syncthreads();
    double t = lane < nw ? scratch[lane] : 0.0;
    return warp_sum(t);
}

}  // namespace mp
