// mp_host.h -- host-side engine state shared by the translation units of libmidaspom_cuda.so.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_runtime.h>
#include "../../include/libmidaspom_cuda.h"
#include "mp_device.cuh"


struct mp_engine {
    mp_config cfg{};
    mp_sampler_config sc{};
    bool have_sc = false, have_landscape = false, have_obs = false, have_state = false;
    int geom = MP_GEOM_LINEAR;
    bool have_area = false;
    double spacing = 100.0;
    cudaStream_t stream = nullptr;
    std::string err;

    // landscape
    double *d_area = nullptr, *d_src_unit = nullptr;
    void *d_px = nullptr, *d_py = nullptr, *d_dist = nullptr;   // float or double per cfg.precision
    // data
    int8_t *d_obs = nullptr;
    uint8_t *d_era = nullptr;
    bool have_era = false;
    // chains
    mp_params *d_par = nullptr, *d_prop = nullptr;
    double *d_lsig = nullptr;
    uint8_t *d_z = nullptr, *d_y = nullptr;
    void *d_srec = nullptr;          // source records of k_conn (mp::SrcRec, [set][chain][word][padded slot], scan order)
    int nwords = 1;
    double *d_S[2] = { nullptr, nullptr };
    void *d_aw[2] = { nullptr, nullptr };
    double *d_partial[2] = { nullptr, nullptr };
    double *d_ljac = nullptr;        // log Jacobian of the ridge move (alpha, b, c) per chain
    double *d_llc = nullptr, *d_logu = nullptr, *d_parts = nullptr, *d_scalar = nullptr;
    int *d_flags = nullptr;
    unsigned long long *d_counts = nullptr;
    double *d_draws = nullptr;
    int ndraws = 0;
    uint32_t sweep = 0;              // host mirrors of d_ctr = {sweep, recorded draws}, the counters the kernels read
    uint32_t *d_ctr = nullptr;
    cudaGraphExec_t gexec[2] = { nullptr, nullptr };   // a captured sweep without / with the refresh of the resident S (mp_sweep)
    bool gwarm[2] = { false, false };                  // that kind of sweep has run once eagerly (lazy allocations done)
    long long glaunch[2][6] = { { 0 } };               // kernel launches per category inside each captured sweep (mp_get_timing counts them per replay)
    int use_graph = 1;               // replay captured sweeps (MP_GRAPH=0 disables)
    int nblk_col = 1;
    void *d_cand = nullptr;          // candidate records of the FP32 fast sweep (mp::CandRec, 32 B each)
    int *d_cand_count = nullptr;     // [task][2]: candidates, occupied
    bool any_src = false;            // some chain has an external source term (Ksrc != 0)
    int sm_count = 148;
    int refresh_every = 16;          // FP32 engine: sweeps between from-scratch recomputations of the resident S
    bool S_valid = false;            // resident S corresponds to the resident (y, alpha, b)
    bool S_exact = true;             // ... and was accumulated in FP64 (false after an evaluation call that took the tensor-core path or the
                                     // FP32 contraction: the next sweep recomputes it before the y scan applies rank-1 updates to it)
    int task_first = 0, task_stride = 1;   // (chain, year) tasks of the y sweep run by this engine (year sharding)
    int conn_lo = 0, conn_hi = -1;        // target patches of k_conn run by this engine (patch sharding); hi < 0 = all
    void *d_tile_box = nullptr;                // float4 {xmin, xmax, ymin, ymax} per group of 32 scan-order slots (culled k_conn)
    float *d_mlow = nullptr;                   // [chain][group] lower bound of S per group of 32 slots (k_group_min_S)
    double area_max = 1.0, area_min = 1.0;
    bool have_boxes = false; int conn_cull = 1;   // MP_CONN_CULL=0 disables the culling of k_conn
    void *d_gemm = nullptr; size_t gemm_bytes = 0;   // BF16 occupancy columns + source records of the tensor-core path (mp_conn_gemm.cu)
    bool have_params = false;                  // mp_set_params (or mp_init_chains) has run
    std::vector<mp_params> par_host;           // parameters as last uploaded by mp_set_params ...
    bool par_host_valid = false;               // ... still what the device holds (the sampler changes them on the device)
    int use_gemm = 1, gemm_min_n = 1024;       // tensor-core connectivity for chains sharing (alpha, b): MP_CONN_GEMM=0 disables, MP_CONN_GEMM_MIN_N
    int last_conn_path = 0;                    // 0: k_conn, 1: k_conn_gemm (mp_get_conn_path)
    int conn_acc32 = 1;   // FP32 engines, evaluation entry points: year contraction of k_conn on the FP32 pipe (mp_conn32.cu); MP_CONN_ACC32=0 keeps the DFMA form
    int conn_shape = 0;                        // CTA shape of k_conn: 0 choose, 1 = 128 threads x 2 targets, 2 = 64 x 2, 3 = 32 x 2 (MP_CONN_SHAPE)
    unsigned long long *d_work = nullptr;      // MP_CNT_* work counters (mp_get_work_counters)
    int *d_task_order = nullptr;               // scan tasks of this engine, longest first (k_order_tasks)
    int *d_perm = nullptr;                     // layout (Morton) order of the patches: perm[slot] = patch
    int *d_scan = nullptr, *d_minv = nullptr;  // visiting order of the y scan (position -> patch; = perm without a scan grid); patch -> layout slot
    int fast_cs = 0;                 // cluster size of the fast sweep (0 = choose); MP_FAST_CS overrides
    int fast_tpt = 0;                // threads per task of the fast sweep (0 = choose from N); MP_FAST_TPT overrides
    // block grid of the y scan (landscapes with coordinates; mp_set_scan_blocks): blk_nx x blk_ny cells, blk_k x blk_k colours
    int blk_nx = 1, blk_ny = 1, blk_k = 1;
    double blk_halo = 0.0;            // targets of a block: its own patches and every patch within this distance of its cell
    bool blk_active = false;          // more than one block: the scan runs colour by colour
    bool blk_tasks_dirty = true;      // the per-colour task lists depend on the chains and on the year sharding
    std::vector<double> hx, hy;       // the caller's coordinates (scan order and block lists are derived from them)
    double cx = 0.0, cy = 0.0, bb[4] = { 0, 0, 0, 0 };   // origin of the device coordinates; bounding box x0, x1, y0, y1 of the caller's
    std::vector<uint32_t> morton;     // Morton code of every patch
    std::vector<int> blk_of, scan_host;   // block of every patch; visiting order of the scan (position -> patch)
    int blk_tpt = 0, blk_cs = 0;      // threads per block task / cluster size (0 = choose); MP_BLK_TPT, MP_BLK_CS override
    std::vector<int> blk_slot_lo, blk_slot_hi, blk_tl_off, blk_tl_n;   // per block: own scan-order slots, target list
    std::vector<int> colour_off, colour_n;     // per colour: first block task and count in d_btasks
    int blk_nl_max = 0;               // largest target list
    int *d_tlist = nullptr;           // concatenated target lists (patch numbers)
    void *d_btasks = nullptr;         // mp::BlockTask of every (owned task, block), grouped by colour
    unsigned char *d_scan_work = nullptr;   // global scratch of the generic y scan on landscapes beyond one CTA's shared memory
    int *d_blockmode = nullptr;       // [chain] 1: this sweep's scan of the chain runs by blocks (k_block_valid)
    int last_scan[4] = { 0, 0, 0, 0 };   // geometry of the last y scan launched: threads per task, cluster size, candidates per trip, culled
    // communicator (mp_comm.cu): NCCL behind the C ABI
    void *comm = nullptr;             // ncclComm_t
    int comm_size = 1, comm_rank = 0, comm_per = 0;   // comm_per: scan-order slots per rank of the sharded connectivity
    double *d_comm_send = nullptr, *d_comm_recv = nullptr;   // packed connectivity columns of the sharded sweep
    int shard_flags = 0;              // what phase 0 of the current sharded sweep computed (bit 0: S, bit 1: S_prop)
    // posterior summaries of the latent state (mp_set_summaries): z_prob, S_sum, z_count, y_count and the sample counter
    unsigned char *d_sum = nullptr;
    int sum_first = 0, sum_thin = 0;  // sum_thin == 0: off
    unsigned long long sum_samples = 0;   // host mirror of the device sample counter, queued sweeps included
    // pointwise predictive densities for WAIC (mp_set_waic): lik, loglik, loglik_sq [T][N] and the uint64 sample counter
    unsigned char *d_waic = nullptr;
    int waic_first = 0, waic_thin = 0;    // waic_thin == 0: off
    // colonisation sources (mp_set_sources): per-sample lists and staging arrays, then the sums (mp_sources.cuh, src_layout)
    unsigned char *d_src = nullptr;
    int src_first = 0, src_thin = 0, src_nbins = 0;   // src_thin == 0: off
    double src_bin_width = 0.0;
    // timing
    bool timing = false;
    struct Span { cudaEvent_t a, b; int cat; };
    std::vector<Span> spans;
    std::vector<cudaEvent_t> pool;
    double t_ms[MP_K_NCAT] = { 0 };
    long long t_launch[MP_K_NCAT] = { 0 };
};

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                                 \
            return MP_ERR_CUDA;                                                                          \
        }                                                                                                \
    } while (0)
#define REQUIRE(cond, code, msg)                                                                         \
    do { if (!(cond)) { h->err = (msg); return (code); } } while (0)

inline size_t nN(const mp_engine *h) { return (size_t)h->cfg.n_patches; }
inline size_t nT(const mp_engine *h) { return (size_t)h->cfg.n_years; }
inline size_t nC(const mp_engine *h) { return (size_t)h->cfg.n_chains; }
inline size_t zcells(const mp_engine *h) { return nT(h) * nN(h); }
inline size_t ycells(const mp_engine *h) { return (nT(h) - 1) * nN(h); }
inline bool is64(const mp_engine *h) { return h->cfg.precision == MP_FP64; }
inline size_t rsz(const mp_engine *h) { return is64(h) ? sizeof(double) : sizeof(float); }

// ---- timing spans: CUDA events on the engine stream around every launch of a category
struct Timed {
    mp_engine *h; int cat; cudaEvent_t a = nullptr, b = nullptr;
    Timed(mp_engine *h_, int cat_) : h(h_), cat(cat_)
    {
        h->t_launch[cat]++;
        if (!h->timing) return;
        a = take(); b = take();
        cudaEventRecord(a, h->stream);
    }
    ~Timed()
    {
        if (!h->timing) return;
        cudaEventRecord(b, h->stream);
        h->spans.push_back({ a, b, cat });
    }
    cudaEvent_t take()
    {
        if (!h->pool.empty()) { cudaEvent_t e = h->pool.back(); h->pool.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
};
inline void drain_spans(mp_engine *h)
{
    for (auto &s : h->spans) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) h->t_ms[s.cat] += ms;
        h->pool.push_back(s.a); h->pool.push_back(s.b);
    }
    h->spans.clear();
}

template <typename R> inline mp::Landscape<R> view(const mp_engine *h)
{
    mp::Landscape<R> ls;
    ls.n = h->cfg.n_patches; ls.spacing = (R)h->spacing;
    ls.px = (const R *)h->d_px; ls.py = (const R *)h->d_py; ls.dist = (const R *)h->d_dist;
    ls.src_unit = h->d_src_unit;
    return ls;
}


// FP32 fast sweep (mp_sweep_fast_*.cu, one translation unit per geometry)
int mp_launch_sweep_fast_linear(mp_engine *h, int cs, int tpt);
int mp_launch_sweep_fast_coords(mp_engine *h, int cs, int tpt);
int mp_launch_sweep_fast_dense(mp_engine *h, int cs, int tpt);
// culled scan: nclusters whole (chain, year) tasks (btasks == nullptr) or block tasks (mp::BlockTask array on the device)
int mp_launch_sweep_cull_linear(mp_engine *h, int cs, int tpt, int nl_max, int nclusters, const void *btasks);
int mp_launch_sweep_cull_coords(mp_engine *h, int cs, int tpt, int nl_max, int nclusters, const void *btasks);
// k_conn of the FP32 engines with the year contraction on the FP32 pipe (mp_conn32.cu); args: the launch's mp::ConnArgs<float>
int mp_launch_conn32(mp_engine *h, const void *args, int geom, int ny, int shape, int cull, unsigned gx, unsigned gy, unsigned gz);
// tensor-core connectivity of every chain with one (alpha, b) (mp_conn_gemm.cu)
int mp_launch_conn_gemm(mp_engine *h, double alpha);
