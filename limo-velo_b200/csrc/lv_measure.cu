/*
 * lv_measure.cu — the kernels of one h-evaluation of the measurement model and of the IESKF step.
 *
 * Replaces, per input point, the chain (reference paths relative to the LIMO-Velo tree)
 *   Mapper::match                 src/Modules/Mapper.cpp:40-56       world transform
 *   KD_TREE::Nearest_Search       include/ikd-Tree/ikd_Tree/ikd_Tree.cpp:426-461   exact 5-NN
 *   Plane::Plane / estimate_plane src/Objects/Plane.cpp:19-55, src/Utils/Utils.cpp:32-66
 *   Match::Match                  src/Objects/Match.cpp:18-22
 *   Localizator::calculate_H      src/Modules/Localizator.cpp:29-57
 * the reduction IKFoM performs on its output,
 *   HTH = h_x^T h_x, h_x^T h      esekfom.hpp:1723,1727
 * and the 23x23 algebra between two evaluations (esekfom.hpp:1647-1817, csrc/lv_ieskf.h).
 *
 * Kernels of one evaluation (DESIGN.md 4): lv_reuse_kernel (evaluations after the first: keep the neighbours the
 * exact search provably returns again), lv_search_kernel (exact 5-NN at level 0, thin, 8 lanes per query),
 * lv_search_rings_kernel (the queries level 0 cannot certify, one warp each), lv_fit_kernel (plane fit, Jacobian
 * row, the 78 + 12 unique normal-equation sums per block in a fixed order; one spare block runs ieskf_prepare),
 * lv_ieskf_step_kernel (one block: reduction of the partials, gain, dx, next frame, loop control).  H (Nm x 12
 * fp64) is never materialised.  Inside an update every kernel is launched with programmatic dependent launch and
 * the whole update is replayed as one CUDA graph (lv_capi.cu).
 *
 * Bound: L2 / HBM gather LATENCY, not bandwidth (algorithmic traffic 72 B per point: 12 B query + 5 x 12 B
 * neighbours); no tensor-core-shaped work.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#ifdef LV_STEP_TIMING
__device__ unsigned long long g_probes[2];     /* total hash probes, number of lookups that needed more than 8 */
#ifdef __CUDA_ARCH__
#define LV_PROBE_COUNT() do { atomicAdd(&g_probes[0], 1ull); } while (0)
#endif
#endif
#ifdef LV_STEP_TIMING   /* tuning build only: per-phase clocks of the step kernel */
__device__ long long g_step_clk[64];
#ifdef __CUDA_ARCH__
#define LV_CK(k) do { if (threadIdx.x == 0) g_step_clk[k] = clock64(); } while (0)
#define LV_TK(k) do { g_step_clk[k] = clock64(); } while (0)
#define LV_FK(k) do { if (threadIdx.x == 0 && blockIdx.x == 1) g_step_clk[k] = clock64(); } while (0)
#endif
#endif
#ifndef LV_FK
#define LV_FK(k)
#endif

#include <cub/device/device_radix_sort.cuh>

#include "lv_internal.h"
#include "lv_predict.h"

#ifdef LV_STEP_TIMING   /* tuning build only: wall-clock timeline of the kernels of an update (graph + PDL included) */
__device__ unsigned long long g_tl[5][8][8];   /* [scheduled | past the wait | end (thread 0) | last block past the wait | end (any warp)][evaluation][kind], ns */
__device__ __forceinline__ unsigned long long lv_gt() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define LV_TL_SCHED() const unsigned long long tl_s_ = lv_gt()
#define LV_TL_WORK(c, kind) const int tl_e_ = (c)->n_evals & 7; if (threadIdx.x == 0) { atomicMin(&g_tl[0][tl_e_][kind], tl_s_); const unsigned long long tw_ = lv_gt(); atomicMin(&g_tl[1][tl_e_][kind], tw_); atomicMax(&g_tl[3][tl_e_][kind], tw_); }
#define LV_TL_END(kind) do { if (threadIdx.x == 0) atomicMax(&g_tl[2][tl_e_][kind], lv_gt()); if ((threadIdx.x & 31) == 0) atomicMax(&g_tl[4][tl_e_][kind], lv_gt()); } while (0)
#else
#define LV_TL_SCHED()
#define LV_TL_WORK(c, kind)
#define LV_TL_END(kind)
#endif

namespace lv {

/* the 90 (a, b) products each block accumulates: 78 upper-triangle entries of HTH, then 12 of HTh
 * (b = 12 selects h) */
__constant__ uint8_t c_pair_a[90];
__constant__ uint8_t c_pair_b[90];
static bool g_pairs_ready[64] = {false};    /* constant memory is per device */

static void init_pairs() {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (g_pairs_ready[dev]) return;
    uint8_t a[90], b[90];
    int e = 0;
    for (int i = 0; i < 12; ++i)
        for (int j = i; j < 12; ++j) { a[e] = (uint8_t)i; b[e] = (uint8_t)j; ++e; }
    for (int i = 0; i < 12; ++i) { a[e] = (uint8_t)i; b[e] = 12; ++e; }
    cudaMemcpyToSymbol(c_pair_a, a, sizeof(a));
    cudaMemcpyToSymbol(c_pair_b, b, sizeof(b));
    g_pairs_ready[dev] = true;
}

/* Programmatic dependent launch: every kernel of an update lets its successor's blocks be scheduled early
 * (pdl_trigger) and waits for its predecessor's results (pdl_wait) only after a prologue that touches nothing
 * the predecessor writes.  Every path through a kernel executes pdl_wait() and triggers only AFTER it, so
 * "this kernel runs past its wait" implies "its predecessor is complete", and a prologue may read whatever
 * was written two or more kernels ago.  Without the launch attribute both are no-ops. */
#ifdef LV_NO_GRIDDEP   /* diagnosis build: without the instructions every launch must be a plain one (LV_NO_PDL=1) */
__device__ __forceinline__ void pdl_wait() {}
__device__ __forceinline__ void pdl_trigger() {}
#else
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

/* the sweep of this launch: kernel arguments, or the device-side job of a graph replay */
struct JobView { const float* xyz; int n; int n_tiles; };
__device__ __forceinline__ JobView job_view(const MeasureArgs& a) {
    JobView j;
    if (a.job) { j.xyz = a.job->xyz; j.n = a.job->n; j.n_tiles = a.job->n_tiles; }
    else { j.xyz = a.xyz; j.n = a.n; j.n_tiles = a.n_tiles; }
    return j;
}

#define LV_ROW_STRIDE (kMeasureThreads + 4)   /* 132 doubles = 4 (mod 16): the 8 x 4 fragment loads of the fold below are conflict-free */
#define LV_SEARCH_THREADS 128
#define LV_GROUP 8                              /* lanes per query in K1 (LV_SEARCH_GROUP=1|8 overrides) */

__device__ __forceinline__ void store_neighbours(const MeasureArgs& a, int qi, const Top5& t) {
    a.nn_a[qi] = make_int4(t.i0, t.i1, t.i2, t.i3);                  /* positions in the arena, -1 = none */
    a.nn_b[qi] = make_int2(t.i4, __float_as_int(t.d4));
}
/* what a later evaluation needs to reuse this answer (lb <= 0: do not) */
__device__ __forceinline__ void store_ref(const MeasureArgs& a, int qi, const float* g, float lb) {
    if (a.ref) a.ref[qi] = make_float4(g[0], g[1], g[2], lb);
}

/*
 * K1 — search, level 0.  G lanes per query, ONE query per lane group, so the grid holds N * G / 32
 * warps and every SM keeps its full complement of warps in flight: the search is a chain of dependent
 * memory round trips (point -> hash slot -> halo bucket) and only resident warps hide them.  The
 * kernel is thin (no plane fit, ~50 registers).  Per group: one hash probe (all lanes, same address),
 * one contiguous scan of the home voxel's halo bucket (a request of the G lanes covers G x 16
 * contiguous bytes), shuffle merge, certification.  Queries level 0 cannot certify (sparse spot, no
 * slot) are appended to a work list for K1b.
 * History (ncu r1a..r1e + clock64 phase timers, profiles/): fused with the fit at 127 registers the
 * search phase alone cost 36-60 k cycles per 128-query tile; hard queries finished inside the warp
 * that found them serialised up to 13 ring searches in one warp (firing order clusters them).
 * Output, 24 B per query: positions of the 5 neighbours and the 5th squared distance.
 */
template <int G, bool LIST>
__global__ void __launch_bounds__(LV_SEARCH_THREADS) lv_search_kernel(const MeasureArgs a) {
    typedef GroupLanes<G> Grp;
    LV_TL_SCHED();
    pdl_wait();                 /* the predecessor (begin / step / reuse kernel) writes the frame and the lists */
    pdl_trigger();
    LV_TL_WORK(a.ctrl, 2);
    /* the search is a chain of dependent round trips (flags -> point -> slot -> bucket): everything that does
     * not depend on an earlier answer is requested up front, the `done` test included */
    const int done = a.ctrl->done;                      /* update already finished (uniform over the grid) */
    const Rt32 T = a.ctrl->frame.lidar_to_world;        /* uniform loads */
    const JobView jb = job_view(a);
    const int n_redo = LIST ? (int)a.hard_count[2] : 0;
    const int slot = (int)(((int64_t)blockIdx.x * LV_SEARCH_THREADS + threadIdx.x) / G);
    const int listed = LIST ? (int)a.redo_list[slot] : 0;   /* redo_list holds max_points entries: always readable */
    if (done) return;
    int qi = slot;
    bool have = slot < jb.n;
    if (LIST) {                 /* only the queries lv_reuse_kernel handed back */
        if ((int)blockIdx.x * (LV_SEARCH_THREADS / G) >= n_redo) return;
        have = slot < n_redo;
        qi = have ? listed : 0;
    }
    float g[3] = {0.f, 0.f, 0.f};
    uint32_t bs = 0, bc = 0, vox[3] = {0u, 0u, 0u};
    int st = 0;                       /* 0 no query / not finite, 1 bucket, 2 no level-0 slot */
    if (have) {
        rt_apply(T, jb.xyz[3 * qi], jb.xyz[3 * qi + 1], jb.xyz[3 * qi + 2], g);   /* Mapper.cpp:51 */
        const bool finite = (fabsf(g[0]) < 1e9f) && (fabsf(g[1]) < 1e9f) && (fabsf(g[2]) < 1e9f);
        if (finite) st = level0_probe(a.map, g[0], g[1], g[2], &bs, &bc, vox) >= 0 ? 1 : 2;
    }
    Top5 t;
    float region = 0.f;
    const bool settled = level0_scan<Grp>(a.map, g[0], g[1], g[2], a.max_d2, bs, bc, st == 1, t, &region, vox);
    if (have && (threadIdx.x & (G - 1)) == 0) {
        store_neighbours(a, qi, t);
        const bool hard = st == 2 || (st == 1 && !settled);
        store_ref(a, qi, g, (st == 1 && settled) ? outsider_bound(t.d5, region) : 0.f);
        if (hard) {
            const uint32_t b = blockIdx.x % kHardBuckets;
            a.hard_list[(size_t)b * a.hard_seg + atomicAdd(a.hard_count + 4 + b, 1u)] = (uint32_t)qi;
        }
    }
    LV_TL_END(2);
}

/*
 * K1c — search, level 0, query-per-lane prologue + 8-lane scans (LV_SEARCH_GROUP=32).  In K1 every instruction of a query's
 * prologue (world transform, three IEEE divisions for the voxel coordinate, hash, probe, face distances) is issued for a warp
 * that holds only FOUR queries: ncu puts 40 % of K1's instructions there.  Here a warp holds 32 queries: each lane does the
 * prologue of its own query (32 probes in flight per warp), then the warp walks its queries four at a time — the owner
 * lanes hand (point, bucket, certified radius) to the 8-lane groups by shuffle, which scan and merge exactly as K1 does.
 * Same candidates, same merge, same answers; an eighth of the prologue instructions.
 */
#define LV_COOP_THREADS 64
template <bool LIST>
__global__ void __launch_bounds__(LV_COOP_THREADS) lv_search_coop_kernel(const MeasureArgs a) {
    typedef GroupLanes<8> Grp;
    LV_TL_SCHED();
    pdl_wait();
    pdl_trigger();
    LV_TL_WORK(a.ctrl, 2);
    const int done = a.ctrl->done;
    const Rt32 T = a.ctrl->frame.lidar_to_world;
    const JobView jb = job_view(a);
    const int n_redo = LIST ? (int)a.hard_count[2] : 0;
    const int slot = (int)(blockIdx.x * LV_COOP_THREADS + threadIdx.x);
    const int listed = LIST ? (int)a.redo_list[slot < (int)a.n ? slot : 0] : 0;
    if (done) return;
    if (LIST && (int)(blockIdx.x * LV_COOP_THREADS) >= n_redo) return;
    const bool have = LIST ? slot < n_redo : slot < jb.n;
    const int qi = have ? (LIST ? listed : slot) : 0;
    /* 1. one query per lane */
    float g[3] = {0.f, 0.f, 0.f}, cert = 0.f;
    uint32_t bs = 0, bc = 0, vox[3] = {0u, 0u, 0u};
    int st = 0;                       /* 0 no query / not finite, 1 bucket, 2 no level-0 slot */
    if (have) {
        rt_apply(T, jb.xyz[3 * qi], jb.xyz[3 * qi + 1], jb.xyz[3 * qi + 2], g);   /* Mapper.cpp:51 */
        const bool finite = (fabsf(g[0]) < 1e9f) && (fabsf(g[1]) < 1e9f) && (fabsf(g[2]) < 1e9f);
        if (finite) st = level0_probe(a.map, g[0], g[1], g[2], &bs, &bc, vox) >= 0 ? 1 : 2;
        if (st == 1) cert = certified_d2(home_geom(a.map.grid, vox[0], vox[1], vox[2], g[0], g[1], g[2]));
    }
    /* 2. four queries at a time, 8 lanes each */
    const int lane = (int)(threadIdx.x & 31u);
#pragma unroll 1
    for (int r = 0; r < 8; ++r) {
        const int src = 4 * r + (lane >> 3);
        const int st_r = __shfl_sync(0xffffffffu, st, src);
        const bool have_r = __shfl_sync(0xffffffffu, have ? 1 : 0, src) != 0;
        if (!__ballot_sync(0xffffffffu, have_r)) break;           /* slots ascend with the lane: nothing further either */
        const float gx = __shfl_sync(0xffffffffu, g[0], src), gy = __shfl_sync(0xffffffffu, g[1], src), gz = __shfl_sync(0xffffffffu, g[2], src);
        const uint32_t bs_r = __shfl_sync(0xffffffffu, bs, src), bc_r = __shfl_sync(0xffffffffu, bc, src);
        const float cert_r = __shfl_sync(0xffffffffu, cert, src);
        const int qi_r = __shfl_sync(0xffffffffu, qi, src);
        Top5 t;
        float region = 0.f;
        const bool settled = level0_scan<Grp>(a.map, gx, gy, gz, a.max_d2, bs_r, bc_r, st_r == 1, t, &region, nullptr, &cert_r);
        if (have_r && (lane & 7) == 0) {
            store_neighbours(a, qi_r, t);
            const bool hard = st_r == 2 || (st_r == 1 && !settled);
            const float gq[3] = {gx, gy, gz};
            store_ref(a, qi_r, gq, (st_r == 1 && settled) ? outsider_bound(t.d5, region) : 0.f);
            if (hard) {
                const uint32_t b = blockIdx.x % kHardBuckets;
                a.hard_list[(size_t)b * a.hard_seg + atomicAdd(a.hard_count + 4 + b, 1u)] = (uint32_t)qi_r;
            }
        }
    }
    LV_TL_END(2);
}

/* ---- bulk copies into shared memory (TMA engine, 1-D form) and the mbarrier they complete on ---------------- */
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
/* global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; completes `bytes` of transaction on `bar` */
__device__ __forceinline__ void bulk_copy_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

/*
 * Kb — bin.  Once per update (the sweep does not change across its evaluations): the home voxel's slot of every
 * query at the propagated state.  A radix sort of the (slot, query) pairs follows (launch_bin), after which the
 * queries of one voxel sit next to each other and lv_search_staged_kernel fetches each halo bucket once per block.
 */
__global__ void __launch_bounds__(128) lv_bin_kernel(const MeasureArgs a) {
    pdl_wait();
    pdl_trigger();
    if (a.ctrl->done) return;
    const JobView jb = job_view(a);
    const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (i >= a.n) return;
    if (i >= jb.n) {            /* graph replay: the sort covers the capacity a.n; the padding sorts behind every query */
        a.bin_key_in[i] = 0xFFFFFFFFu;
        a.bin_val_in[i] = 0xFFFFFFFFu;
        return;
    }
    const Rt32& T = a.ctrl->frame.lidar_to_world;
    float g[3];
    rt_apply(T, jb.xyz[3 * i], jb.xyz[3 * i + 1], jb.xyz[3 * i + 2], g);
    uint32_t key = 0xFFFFFFFFu, bs, bc;
    const bool finite = (fabsf(g[0]) < 1e9f) && (fabsf(g[1]) < 1e9f) && (fabsf(g[2]) < 1e9f);
    if (finite) {
        const int slot = level0_probe(a.map, g[0], g[1], g[2], &bs, &bc);
        if (slot >= 0) key = (uint32_t)slot;
    }
    a.bin_key_in[i] = key;
    a.bin_val_in[i] = (uint32_t)i;
}

/*
 * K1s — search, level 0, from shared memory.  One block = LV_STAGE_QUERIES consecutive queries of the binned order,
 * i.e. a handful of voxel runs.  Per block: the run heads read their voxel's slot (one 32-byte sector: key, bucket
 * start and count), a block scan places the buckets in shared memory, each head issues ONE bulk copy
 * (cp.async.bulk, completing on an mbarrier) for its bucket, and after the wait every thread scans its query's
 * bucket out of shared memory: no per-lane merge, no shuffles, one global fetch per bucket instead of one per query
 * (a 65 536-point Velodyne sweep has ~6 queries per home voxel).  Buckets beyond the staging budget are scanned from
 * global memory by the same loop.
 *   Certification is relative to the voxel the query was BINNED in (at the propagated state): the bucket holds every
 * map point of that voxel's 3x3x3 neighbourhood, so whatever lies closer to the query than the neighbourhood's
 * boundary is exact — also when a later iterate has moved the query into a neighbouring voxel.  What cannot be
 * certified goes to lv_search_rings_kernel, as in the per-query kernel.  Results are identical to lv_search_kernel's.
 *   With REDO (evaluations after the first, reuse on) the queries lv_reuse_kernel vouched for are skipped.
 */
#define LV_STAGE_QUERIES 128
#define LV_STAGE_PTS 2560                      /* float4 of staged buckets per block: 40 KB */
/* one thread scans a whole bucket: p[0 .. n) are the points, ids are bstart + j */
__device__ __forceinline__ void scan_bucket(const float4* p, uint32_t n, uint32_t bstart, const float* g, Top5& t) {
    uint32_t j = 0;
    for (; j + 4 <= n; j += 4) {
        const float4 q0 = p[j], q1 = p[j + 1], q2 = p[j + 2], q3 = p[j + 3];
        top5_insert(t, sq_dist(g[0], g[1], g[2], q0.x, q0.y, q0.z), (int)(bstart + j));
        top5_insert(t, sq_dist(g[0], g[1], g[2], q1.x, q1.y, q1.z), (int)(bstart + j + 1));
        top5_insert(t, sq_dist(g[0], g[1], g[2], q2.x, q2.y, q2.z), (int)(bstart + j + 2));
        top5_insert(t, sq_dist(g[0], g[1], g[2], q3.x, q3.y, q3.z), (int)(bstart + j + 3));
    }
    for (; j < n; ++j) {
        const float4 q = p[j];
        top5_insert(t, sq_dist(g[0], g[1], g[2], q.x, q.y, q.z), (int)(bstart + j));
    }
}
__device__ __noinline__ void scan_bucket_global(const float4* p, uint32_t n, uint32_t bstart, const float* g, Top5& t) {
    for (uint32_t j = 0; j < n; ++j) {
        const float4 q = load_point(p + j);
        top5_insert(t, sq_dist(g[0], g[1], g[2], q.x, q.y, q.z), (int)(bstart + j));
    }
}
template <bool REDO>
__global__ void __launch_bounds__(LV_STAGE_QUERIES) lv_search_staged_kernel(const MeasureArgs a) {
    __shared__ __align__(16) float4 s_pts[LV_STAGE_PTS];
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ uint32_t s_key[LV_STAGE_QUERIES];
    __shared__ uint32_t s_run_start[LV_STAGE_QUERIES];    /* bucket position in the arena                         */
    __shared__ uint32_t s_run_count[LV_STAGE_QUERIES];
    __shared__ uint32_t s_run_off[LV_STAGE_QUERIES];      /* position in s_pts, 0xFFFFFFFF: read from the arena   */
    __shared__ uint32_t s_run_vox[LV_STAGE_QUERIES][3];   /* biased voxel coordinates of the run's voxel          */
    __shared__ uint32_t s_run_need[LV_STAGE_QUERIES];
    __shared__ uint32_t s_warp_heads[LV_STAGE_QUERIES / 32], s_warp_pts[LV_STAGE_QUERIES / 32];
    LV_TL_SCHED();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) mbar_init(&s_bar, 1);
    s_run_need[tid] = 0u;
    pdl_wait();                 /* frame (step kernel), binned order (sort), redo flags (reuse kernel) */
    pdl_trigger();
    LV_TL_WORK(a.ctrl, 2);
    const int done = a.ctrl->done;
    const Rt32 T = a.ctrl->frame.lidar_to_world;
    const JobView jb = job_view(a);
    if (done || (int)blockIdx.x * LV_STAGE_QUERIES >= jb.n) return;
    const int pos = (int)blockIdx.x * LV_STAGE_QUERIES + tid;
    const bool have = pos < jb.n;
    const uint32_t key = have ? a.bin_key[pos] : 0xFFFFFFFFu;
    const int qi = have ? (int)a.bin_val[pos] : 0;
    bool active = have;
    if (REDO && have) active = a.redo_flag[qi] != 0;
    s_key[tid] = key;
    __syncthreads();
    /* runs of equal keys inside the block */
    const bool binned = key != 0xFFFFFFFFu;
    const bool head = binned && (tid == 0 || s_key[tid - 1] != key);
    const unsigned hb = __ballot_sync(0xffffffffu, head);
    if (lane == 0) s_warp_heads[warp] = (uint32_t)__popc(hb);
    __syncthreads();
    uint32_t run = (uint32_t)__popc(hb & (0xffffffffu >> (31 - lane)));      /* heads at or before this lane */
    for (int w = 0; w < warp; ++w) run += s_warp_heads[w];
    run = binned ? run - 1u : 0u;                                             /* a binned query's run index */
    uint32_t n_runs = 0;
    for (int w = 0; w < LV_STAGE_QUERIES / 32; ++w) n_runs += s_warp_heads[w];
    if (binned && active) s_run_need[run] = 1u;                               /* benign race: everybody writes 1 */
    __syncthreads();
    /* the head of a run fetches its voxel's slot */
    uint32_t my_count = 0;
    if (head) {
        const uint4 e0 = load_slot(a.map.table + 2 * (size_t)key), e1 = load_slot(a.map.table + 2 * (size_t)key + 1);
        const uint64_t vk = (uint64_t)e0.x | ((uint64_t)e0.y << 32);
        s_run_vox[run][0] = (uint32_t)vk & 0x1FFFFFu;
        s_run_vox[run][1] = (uint32_t)(vk >> 21) & 0x1FFFFFu;
        s_run_vox[run][2] = (uint32_t)(vk >> 42) & 0x1FFFFFu;
        s_run_start[run] = e1.x;
        s_run_count[run] = e1.y;
        my_count = s_run_need[run] ? e1.y : 0u;
    }
    /* block-wide exclusive scan of the heads' counts -> staging offsets */
    uint32_t incl = my_count;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) s_warp_pts[warp] = incl;
    __syncthreads();
    uint32_t off = incl - my_count;
    for (int w = 0; w < warp; ++w) off += s_warp_pts[w];
    const bool staged = head && my_count > 0u && off + my_count <= (uint32_t)LV_STAGE_PTS;
    if (head) s_run_off[run] = staged ? off : 0xFFFFFFFFu;
    /* bytes in flight: the sum over the staged runs */
    uint32_t my_bytes = staged ? my_count * 16u : 0u;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) my_bytes += __shfl_xor_sync(0xffffffffu, my_bytes, d);
    __syncthreads();                              /* s_warp_pts is reused below: everybody has read it */
    if (lane == 0) s_warp_pts[warp] = my_bytes;
    __syncthreads();
    if (tid == 0) {
        uint32_t total = 0;
        for (int w = 0; w < LV_STAGE_QUERIES / 32; ++w) total += s_warp_pts[w];
        mbar_arrive_expect_tx(&s_bar, total);     /* the one arrival the barrier waits for + the bytes the copies bring */
    }
    if (staged) bulk_copy_g2s(s_pts + off, a.map.arena + s_run_start[run], my_count * 16u, &s_bar);
    /* meanwhile: this thread's query */
    float g[3] = {0.f, 0.f, 0.f};
    bool finite = false;
    if (active) {
        rt_apply(T, jb.xyz[3 * qi], jb.xyz[3 * qi + 1], jb.xyz[3 * qi + 2], g);   /* Mapper.cpp:51 */
        finite = (fabsf(g[0]) < 1e9f) && (fabsf(g[1]) < 1e9f) && (fabsf(g[2]) < 1e9f);
    }
    {   /* wait for the buckets (bounded: a lost transaction must not hang the GPU) */
        uint32_t spins = 0;
        while (!mbar_try_wait(&s_bar, 0u)) {
            if (++spins > (1u << 24)) { __trap(); }
        }
    }
    if (!active) return;
    Top5 t;
    top5_init(t, a.max_d2);
    float cert = 0.f;
    int st = 0;                                    /* 0 not finite, 1 bucket, 2 no bin */
    if (finite) st = binned ? 1 : 2;
    if (st == 1) {
        const uint32_t bstart = s_run_start[run], n = s_run_count[run], so = s_run_off[run];
        if (so != 0xFFFFFFFFu) scan_bucket(s_pts + so, n, bstart, g, t);          /* shared memory: LDS.128 */
        else scan_bucket_global(a.map.arena + bstart, n, bstart, g, t);             /* did not fit the staging budget */
        cert = neighbourhood_certified_d2(a.map.grid, s_run_vox[run][0], s_run_vox[run][1], s_run_vox[run][2], g[0], g[1], g[2]);
    }
    const bool settled = st == 1 && t.d4 <= cert;
    store_neighbours(a, qi, t);
    store_ref(a, qi, g, settled ? outsider_bound(t.d5, cert) : 0.f);
    if (st == 2 || (st == 1 && !settled)) {
        const uint32_t b = blockIdx.x % kHardBuckets;
        a.hard_list[(size_t)b * a.hard_seg + atomicAdd(a.hard_count + 4 + b, 1u)] = (uint32_t)qi;
    }
    LV_TL_END(2);
}

/*
 * Kv — reuse.  Evaluations after the first of an update: the iterate moved by millimetres, the map not at all.
 * One thread per query re-measures its five stored neighbours from the new world position and keeps them when
 * query_reusable() proves the exact search would return the same five (lv_voxel_search.h); the others go to
 * the redo list and through the search kernels as usual.  Results are identical either way.
 */
__global__ void __launch_bounds__(128) lv_reuse_kernel(const MeasureArgs a) {
    /* Before the wait: everything but the new frame.  The sweep, the stored neighbours (written by the previous
     * evaluation's search kernels, three or more kernels ago) and the map are fetched while the step kernel
     * still runs; after the wait only the frame is missing. */
    LV_TL_SCHED();
    const JobView jb = job_view(a);
    const int qi = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    const bool have = qi < jb.n;
    float p[3] = {0.f, 0.f, 0.f}, q[5][3];
    float ref[4] = {0.f, 0.f, 0.f, 0.f};
    int id[5] = {-1, -1, -1, -1, -1};
    bool cand = false;
    if (have) {
        p[0] = jb.xyz[3 * qi]; p[1] = jb.xyz[3 * qi + 1]; p[2] = jb.xyz[3 * qi + 2];
        const float4 r4 = a.ref[qi];
        const int4 na = a.nn_a[qi];
        const int2 nb = a.nn_b[qi];
        ref[0] = r4.x; ref[1] = r4.y; ref[2] = r4.z; ref[3] = r4.w;
        cand = r4.w > 0.f && nb.x >= 0;
        if (cand) {
            id[0] = na.x; id[1] = na.y; id[2] = na.z; id[3] = na.w; id[4] = nb.x;
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const float4 v = load_point(a.map.arena + id[k]);
                q[k][0] = v.x; q[k][1] = v.y; q[k][2] = v.z;
            }
        }
    }
    pdl_wait();                 /* the step kernel before us writes the frame and the done flag */
    pdl_trigger();
    LV_TL_WORK(a.ctrl, 1);
    if (a.ctrl->done) return;
    bool redo = false;
    if (have) {
        const Rt32& T = a.ctrl->frame.lidar_to_world;
        float g[3];
        rt_apply(T, p[0], p[1], p[2], g);
        redo = true;
        Top5 t;
        if (cand && query_reusable(ref, g, q, id, a.max_d2, t)) {
            store_neighbours(a, qi, t);
            redo = false;
        }
    }
    if (have && a.redo_flag) a.redo_flag[qi] = redo ? 1 : 0;       /* the staged search walks the binned order and skips the rest */
    /* one atomic per warp */
    const unsigned m = __ballot_sync(0xffffffffu, redo);
    if (m) {
        const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
        uint32_t base = 0;
        if (lane == leader) base = atomicAdd(a.hard_count + 2, (uint32_t)__popc(m));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (redo) a.redo_list[base + (uint32_t)__popc(m & ((1u << lane) - 1u))] = (uint32_t)qi;
    }
    LV_TL_END(1);
}

/* One warp per hard query and a query costs ~10 dependent memory round trips, so the grid gives every hard query of a sweep its
 * own warp (a 65 536-point sweep has ~1 200): 5 blocks of 4 warps are resident per SM (38 KB of scratch each). */
enum { kRingsGrid = 148 * 5 };
/*
 * K1b — search beyond ring 1: one WARP per query K1 could not certify (knn5_rings).  The work list
 * length lives on the device; a fixed grid strides over it, so no host round trip is needed.
 */
__global__ void __launch_bounds__(128) lv_search_rings_kernel(const MeasureArgs a) {
    /* flags, frame and job were written two or more kernels ago: safe to fetch while the search still runs
     * (a kernel triggers its successor only after its own wait, so "two kernels ago" is complete by now) */
    LV_TL_SCHED();
    const int done = a.ctrl->done;
    const JobView jb = job_view(a);
    const Rt32 T = a.ctrl->frame.lidar_to_world;
    pdl_wait();                 /* the search kernel's work list and uncertified answers */
    pdl_trigger();
    LV_TL_WORK(a.ctrl, 3);
    if (done) return;
    /* the 32 segment lengths, one per lane, and their prefix sums */
    const int lane = threadIdx.x & 31;
    const uint32_t cnt = a.hard_count[4 + lane];
    uint32_t incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    const uint32_t n_hard = __shfl_sync(0xffffffffu, incl, 31);
    __shared__ RingScratch s_ring[4];                  /* one per warp of the block */
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t h = warp; h < n_hard; h += n_warps) {
        int lo = 0;                                     /* first segment whose inclusive prefix exceeds h */
#pragma unroll
        for (int step = 16; step > 0; step >>= 1) {
            const uint32_t v = __shfl_sync(0xffffffffu, incl, lo + step - 1);
            if (v <= h) lo += step;
        }
        const uint32_t before = __shfl_sync(0xffffffffu, incl - cnt, lo);
        const int qi = (int)a.hard_list[(size_t)lo * a.hard_seg + (h - before)];
        float g[3];
        rt_apply(T, jb.xyz[3 * qi], jb.xyz[3 * qi + 1], jb.xyz[3 * qi + 2], g);
        const int2 prev = a.nn_b[qi];   /* level 0's (uncertified) 5th distance bounds the answer from above */
        Top5 u;
        float region = 0.f;
        __syncwarp();
        knn5_rings_warp(a.map, g[0], g[1], g[2], a.max_d2, prev.x >= 0 ? __int_as_float(prev.y) : a.max_d2, u, &region,
                        &s_ring[threadIdx.x >> 5]);
        if ((threadIdx.x & 31) == 0) {
            store_neighbours(a, qi, u);
            store_ref(a, qi, g, outsider_bound(u.d5, region));
        }
    }
    LV_TL_END(3);
}

/*
 * K2 — fit, row, reduce.  One thread per query, one tile = kMeasureThreads queries.
 *   fit + row   gates (Plane.cpp:36-43), 5x3 QR plane fit, residual, Jacobian row
 *   reduce      the 90 unique sums of H^T H and H^T h over the tile, fixed order; H (Nm x 12 fp64) is
 *               never materialised
 */
/* ieskf_prepare() of the iterate being measured, in one spare block (see lv_ieskf.h) */
__device__ __noinline__ void prepare_block(UpdateCtrl* c) {
    __shared__ PrepWork s_prep;
    ExecBlock ex;
    ieskf_prepare(ex, c, &s_prep);
}

__global__ void __launch_bounds__(kMeasureThreads, 4) lv_fit_kernel(const MeasureArgs a) {
    LV_TL_SCHED();
    /* prologue on data written two or more kernels ago (flags, frame, iterate): runs while the searches finish */
    const int done = a.ctrl->done;
    /* with a.prep the grid has one extra block in front; it is dispatched first and is done long before
     * the measurement blocks, so the iterate-only algebra costs the update no time of its own */
    const int n_blocks = a.prep ? (int)gridDim.x - 1 : (int)gridDim.x;
    const int bid = a.prep ? (int)blockIdx.x - 1 : (int)blockIdx.x;
    if (bid < 0) {
        if (!done) prepare_block(a.prep);
        pdl_wait();
        pdl_trigger();
#ifdef LV_STEP_TIMING
        if (threadIdx.x < 32) {   /* tuning build: how many queries this evaluation searched again, how many went to the ring search */
            unsigned v = a.hard_count[4 + threadIdx.x];
            for (int s_ = 16; s_ > 0; s_ >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s_);
            if (threadIdx.x == 0) { g_tl[2][a.ctrl->n_evals & 7][6] = v; g_tl[2][a.ctrl->n_evals & 7][7] = a.hard_count[2]; }
        }
        __syncthreads();
#endif
        /* the searches of this evaluation are over: reset their counters for the next one */
        if (threadIdx.x < kCounters) a.hard_count[threadIdx.x] = 0u;
        return;
    }

    __shared__ Frame s_frame;
    __shared__ double s_rows[16 * LV_ROW_STRIDE];   /* 13 columns of the tile's rows (12 of H, then h), padded to 16 with zeros */
    __shared__ double s_part[4 * 192];              /* per warp: its share of the three 8 x 8 tiles of [H h]^T [H h] */
    for (int i = threadIdx.x; i < 3 * LV_ROW_STRIDE; i += kMeasureThreads) s_rows[13 * LV_ROW_STRIDE + i] = 0.0;

    {   /* the frame of the current iterate: written by the step kernel, broadcast via smem */
        const uint32_t* src = reinterpret_cast<const uint32_t*>(&a.ctrl->frame);
        uint32_t* dst = reinterpret_cast<uint32_t*>(&s_frame);
        for (int i = threadIdx.x; i < (int)(sizeof(Frame) / 4); i += kMeasureThreads) dst[i] = src[i];
    }
    __syncthreads();
    const int tid = threadIdx.x;
    const JobView jb = job_view(a);
    /* the first tile's world points need only the sweep and the frame: transform them before the wait too */
    float g0[3] = {0.f, 0.f, 0.f};
    {
        const int i = bid * kMeasureThreads + tid;
        if (bid < jb.n_tiles && i < jb.n)
            rt_apply(s_frame.lidar_to_world, jb.xyz[3 * i], jb.xyz[3 * i + 1], jb.xyz[3 * i + 2], g0);
    }
    LV_FK(56);
    pdl_wait();                 /* the neighbour lists */
    pdl_trigger();
    LV_TL_WORK(a.ctrl, 4);
    if (done) return;
    LV_FK(57);

    double acc = 0.0;
    int count = 0;

    for (int tile = bid; tile < jb.n_tiles; tile += n_blocks) {
        const int i = tile * kMeasureThreads + tid;
        bool chosen = false;
        double row[12], hval = 0.0;
        if (i < jb.n) {
            float g[3] = {g0[0], g0[1], g0[2]};
            if (tile != bid) rt_apply(s_frame.lidar_to_world, jb.xyz[3 * i], jb.xyz[3 * i + 1], jb.xyz[3 * i + 2], g);
            const int4 na = a.nn_a[i];
            const int2 nb = a.nn_b[i];
            const float d4 = __int_as_float(nb.y);
            float abcd[4] = {0.f, 0.f, 0.f, 0.f};
            float dist = 0.f;
            float q[5][3];
            float dsq[5] = {INFINITY, INFINITY, INFINITY, INFINITY, INFINITY};
            int orig[5] = {-1, -1, -1, -1, -1};
            const bool full = nb.x >= 0;
            if (full) {
                const float4* src = a.map.arena;
                const float4 q0 = load_point(src + na.x), q1 = load_point(src + na.y), q2 = load_point(src + na.z),
                             q3 = load_point(src + na.w), q4 = load_point(src + nb.x);
                q[0][0] = q0.x; q[0][1] = q0.y; q[0][2] = q0.z;
                q[1][0] = q1.x; q[1][1] = q1.y; q[1][2] = q1.z;
                q[2][0] = q2.x; q[2][1] = q2.y; q[2][2] = q2.z;
                q[3][0] = q3.x; q[3][1] = q3.y; q[3][2] = q3.z;
                q[4][0] = q4.x; q[4][1] = q4.y; q[4][2] = q4.z;
                orig[0] = __float_as_int(q0.w); orig[1] = __float_as_int(q1.w); orig[2] = __float_as_int(q2.w);
                orig[3] = __float_as_int(q3.w); orig[4] = __float_as_int(q4.w);
                for (int k = 0; k < 5; ++k) dsq[k] = sq_dist(g[0], g[1], g[2], q[k][0], q[k][1], q[k][2]);
                LV_FK(58);
                canonical_neighbour_order(q, dsq, orig);             /* equidistant neighbours: the reference's (distance, x) order */
                /* Plane.cpp:36-43: 5 neighbours and the farthest closer than MAX_DIST_PLANE */
                if ((double)d4 < a.gate_d2) {
                    chosen = plane_fit(q, a.planes_threshold, abcd);               /* Plane.cpp:45-55 */
                    if (chosen) {
                        dist = plane_dist(abcd, g);                                /* Match.cpp:21 */
                        jacobian_row(s_frame, g, abcd, dist, a.estimate_extrinsics != 0, row, &hval);
                    } else {
                        abcd[0] = abcd[1] = abcd[2] = abcd[3] = 0.f;
                    }
                }
            }
            if (a.valid) a.valid[i] = chosen ? 1 : 0;
            if (a.g_world) { a.g_world[3 * i] = g[0]; a.g_world[3 * i + 1] = g[1]; a.g_world[3 * i + 2] = g[2]; }
            if (a.nn_idx || a.nn_sqd) {
                for (int k = 0; k < 5; ++k) {
                    if (a.nn_idx) a.nn_idx[5 * i + k] = orig[k];
                    if (a.nn_sqd) a.nn_sqd[5 * i + k] = dsq[k];
                }
            }
            if (a.plane) { for (int k = 0; k < 4; ++k) a.plane[4 * i + k] = abcd[k]; }
            if (a.dist) a.dist[i] = dist;
            if (a.rows) {
                for (int k = 0; k < 12; ++k) a.rows[13 * (size_t)i + k] = chosen ? row[k] : 0.0;
                a.rows[13 * (size_t)i + 12] = chosen ? hval : 0.0;
            }
        }
        LV_FK(59);
        /* stage the row (zeros when rejected), fold the tile into the block's 90 sums */
#pragma unroll
        for (int k = 0; k < 12; ++k) s_rows[k * LV_ROW_STRIDE + tid] = chosen ? row[k] : 0.0;
        s_rows[12 * LV_ROW_STRIDE + tid] = chosen ? hval : 0.0;
        count += __syncthreads_count(chosen ? 1 : 0);
        LV_FK(60);
        {
            /* The tile's 13 x 13 Gram matrix on the fp64 tensor cores (mma.m8n8k4: D = A B + C, A 8x4, B 4x8): 16 x 16 with
             * the padding, three 8 x 8 tiles (00, 01, 11 — it is symmetric), each warp a quarter of the 128 rows.  A lane's A
             * fragment of column-tile I is element (column I*8 + lane/4, row k0 + lane%4) and the B fragment of column-tile J
             * is the same expression with J: two loads feed three MMAs of 256 multiply-adds each.  (The scalar fold — 90
             * threads x 128 x two 8-byte shared loads per multiply-add — spent 4 400 cycles per tile waiting for the four
             * resident blocks' 6 000 shared-memory wavefronts; clock64, tools/step_timing.py.) */
            const int lane = tid & 31, w = tid >> 5;
            const double* f0 = s_rows + (lane >> 2) * LV_ROW_STRIDE + 32 * w + (lane & 3);
            const double* f1 = f0 + 8 * LV_ROW_STRIDE;
            double c00a = 0.0, c00b = 0.0, c01a = 0.0, c01b = 0.0, c11a = 0.0, c11b = 0.0;
#pragma unroll
            for (int ks = 0; ks < 8; ++ks) {
                const double a0 = f0[4 * ks], a1 = f1[4 * ks];
                asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c00a), "+d"(c00b) : "d"(a0), "d"(a0));
                asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c01a), "+d"(c01b) : "d"(a0), "d"(a1));
                asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c11a), "+d"(c11b) : "d"(a1), "d"(a1));
            }
            double* pt = s_part + w * 192 + (lane >> 2) * 8 + 2 * (lane & 3);   /* C fragment: row lane/4, columns 2 (lane%4), +1 */
            pt[0] = c00a; pt[1] = c00b;
            pt[64] = c01a; pt[65] = c01b;
            pt[128] = c11a; pt[129] = c11b;
        }
        __syncthreads();
        if (tid < 90) {   /* entry (a, b), a <= b: tile 00 / 01 / 11; the warps' shares in warp order */
            const int pa = c_pair_a[tid], pb = c_pair_b[tid];
            const int idx = (pa < 8 ? (pb < 8 ? 0 : 64) : 128) + (pa & 7) * 8 + (pb & 7);
            acc += (s_part[idx] + s_part[192 + idx]) + (s_part[384 + idx] + s_part[576 + idx]);
        }
        __syncthreads();
    }
    LV_FK(61);
    double* out = a.partials + (size_t)bid * kPartialStride;
    if (tid < 90) out[tid] = acc;
    if (tid == 90) out[90] = (double)count;
    /* Pre-reduction: the blocks form groups of kPartialGroup consecutive rows; the block of a group that finishes LAST
     * (a ticket per group) adds the group's rows in row order into one group row.  Which block that is varies, the
     * order of the additions does not, so the result is deterministic; the groups finish at different times and are
     * summed on different SMs while other blocks still work, and the step kernel is left with <= 19 rows instead of 592
     * (it used to spend a quarter of its time pulling 400 KB of partials through one SM's L2 port). */
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    const int grp = bid / kPartialGroup, r0 = grp * kPartialGroup;
    const int r1 = r0 + kPartialGroup < n_blocks ? r0 + kPartialGroup : n_blocks;
    if (tid == 0) {
        const unsigned ticket = atomicAdd(a.group_tickets + grp, 1u);
        s_last = ticket == (unsigned)(r1 - r0) - 1u ? 1 : 0;
        if (s_last) a.group_tickets[grp] = 0u;          /* nobody else touches it before the next evaluation */
    }
    __syncthreads();
    LV_FK(62);
    if (s_last) {
        __threadfence();
        if (tid < 91) {
            double v[kPartialGroup];
#pragma unroll
            for (int r = 0; r < kPartialGroup; ++r) v[r] = r0 + r < r1 ? __ldcg(a.partials + (size_t)(r0 + r) * kPartialStride + tid) : 0.0;
            double sum = 0.0;
#pragma unroll
            for (int r = 0; r < kPartialGroup; ++r) sum += v[r];
            a.group_rows[(size_t)grp * kPartialStride + tid] = sum;
        }
    }
    LV_FK(63);
    LV_TL_END(4);
}

/* ---- fixed-order reduction of the per-block partials ---------------------------------------- */
/* Warp w of the block owns rows w, w + nwarps, ...; lanes own elements lane, lane+32, lane+64.  Rows are
 * fetched 8 at a time (24 independent loads per lane) and
 * added in row order; then the warp sums are added in warp order.  Deterministic for a given grid. */
__device__ void reduce_partials_block(const double* partials, int n_partials, double* s_tmp /*nwarps*96*/,
                                      double* HTH, double* HTh, int64_t* nm) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    double a0 = 0, a1 = 0, a2 = 0;
    for (int b = warp; b < n_partials; b += 8 * nwarps) {
        double v[8][3];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int row = b + r * nwarps;
            const double* p = partials + (size_t)row * kPartialStride;
            const bool in = row < n_partials;
            v[r][0] = in ? p[lane] : 0.0;
            v[r][1] = in ? p[lane + 32] : 0.0;
            v[r][2] = in ? p[lane + 64] : 0.0;
        }
#pragma unroll
        for (int r = 0; r < 8; ++r) { a0 += v[r][0]; a1 += v[r][1]; a2 += v[r][2]; }
    }
    s_tmp[warp * 96 + lane] = a0;
    s_tmp[warp * 96 + lane + 32] = a1;
    s_tmp[warp * 96 + lane + 64] = a2;
    __syncthreads();
    if (threadIdx.x < 91) {
        double s = 0;
        for (int w = 0; w < nwarps; ++w) s += s_tmp[w * 96 + threadIdx.x];
        const int e = threadIdx.x;
        if (e < 78) {
            const int i = c_pair_a[e], j = c_pair_b[e];
            HTH[i * 12 + j] = s;
            HTH[j * 12 + i] = s;
        } else if (e < 90) {
            HTh[e - 78] = s;
        } else {
            *nm = (int64_t)(s + 0.5);
        }
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kStepThreads, 1) lv_ieskf_step_kernel(UpdateCtrl* c, const IeskfParams prm,
                                                                     const double* partials, int n_partials) {
    /* (min. blocks 1: the kernel runs as a single block, so ptxas may use up to 255 registers; with the default bound it
     * stopped at 128 and spilled) */
    /* before the wait: what the previous step (or begin) kernel left, two or more kernels ago */
    constexpr int kPrepWords = (int)(sizeof(StepPrep) / sizeof(double));
    constexpr int kPrepLoads = (kPrepWords + kStepThreads - 1) / kStepThreads;
    static_assert(kStepThreads >= 99, "one pass for the state and the counters");
    LV_TL_SCHED();
    const int t = threadIdx.x;
    const int done = c->done;
    double sv = 0.0;
    if (t < 26) sv = c->x[t];
    else if (t < 52) sv = c->x_prop[t - 26];
    int cv = 0;
    if (t >= 96 && t < 99) cv = t == 96 ? c->n_evals : (t == 97 ? c->t : c->iter);
    pdl_wait();                 /* partials and c->prep, written by the fit kernel */
    pdl_trigger();
    LV_TL_WORK(c, 5);
    if (done) return;
    __shared__ IeskfWork w;
    __shared__ double s_tmp[(kStepThreads / 32) * 96];
    ExecBlock ex;
    LV_CK(0);
    /* ieskf_load(), split: the loads are issued here and parked in shared memory after the reduction, so
     * they are in flight together with the partials */
    const double* src = reinterpret_cast<const double*>(&c->prep);
    double pv[kPrepLoads];
#pragma unroll
    for (int r = 0; r < kPrepLoads; ++r) pv[r] = t + r * kStepThreads < kPrepWords ? src[t + r * kStepThreads] : 0.0;
    LV_CK(1);
    reduce_partials_block(partials, n_partials, s_tmp, w.HTH, w.HTh, &w.n_matches);
    double* dst = reinterpret_cast<double*>(&w.p);
#pragma unroll
    for (int r = 0; r < kPrepLoads; ++r)
        if (t + r * kStepThreads < kPrepWords) dst[t + r * kStepThreads] = pv[r];
    if (t < 26) w.x[t] = sv;
    else if (t < 52) w.xp[t - 26] = sv;
    if (t == 96) { w.n_evals = cv; w.eval_idx = cv < kMaxEvals ? cv : kMaxEvals - 1; }
    if (t == 97) w.t = cv;
    if (t == 98) w.iter = cv;
    __syncthreads();
    LV_CK(2);
    ieskf_step(ex, prm, c, &w);
    LV_TL_END(5);
}

__global__ void __launch_bounds__(kStepThreads) lv_reduce_partials_kernel(const double* partials, int n_partials,
                                                                          double* out) {
    __shared__ double s_tmp[(kStepThreads / 32) * 96];
    __shared__ double HTH[144], HTh[12];
    __shared__ int64_t nm;
    reduce_partials_block(partials, n_partials, s_tmp, HTH, HTh, &nm);
    for (int i = threadIdx.x; i < 144; i += blockDim.x) out[i] = HTH[i];
    if (threadIdx.x < 12) out[144 + threadIdx.x] = HTh[threadIdx.x];
    if (threadIdx.x == 0) out[156] = (double)nm;
}

__global__ void __launch_bounds__(256) lv_ieskf_begin_kernel(UpdateCtrl* c, MeasureJob* job, const float* xyz, int n,
                                                             uint32_t* counters) {
    pdl_trigger();
    if (counters && threadIdx.x < kCounters) counters[threadIdx.x] = 0u;    /* work-list lengths of the measurement kernels */
    if (job && threadIdx.x == 0) {
        job->xyz = xyz;
        job->n = n;
        job->n_tiles = (n + kMeasureThreads - 1) / kMeasureThreads;
    }
    ExecBlock ex;
    ieskf_begin(ex, c);
}

/* Localizator::propagate_to (Localizator.cpp:59-75): every IMU sample between two sweeps through esekf::predict, one launch,
 * one thread block; imu = k x 7 doubles (acc, gyro, dt).  The state stays in UpdateCtrl: update -> propagate -> update needs
 * no host round trip. */
__global__ void __launch_bounds__(256) lv_predict_kernel(UpdateCtrl* c, const PredictNoise noise, const double* __restrict__ imu, int k) {
    __shared__ PredictWork w;
    ExecBlock ex;
    LV_PAR(i, kStateLen) w.x[i] = c->x[i];
    LV_PAR(i, kN * kN) w.P[i] = c->P[i];
    ex.sync();
    for (int s = 0; s < k; ++s) predict_step(ex, noise, imu + 7 * s, imu + 7 * s + 3, imu[7 * s + 6], &w);
    LV_PAR(i, kStateLen) c->x[i] = w.x[i];
    LV_PAR(i, kN * kN) c->P[i] = w.P[i];
}

__global__ void lv_set_frame_kernel(UpdateCtrl* c) {
    if (threadIdx.x == 0) {
        make_frame(c->x, &c->frame);
        c->done = 0;
    }
}

__global__ void lv_l2_flush_kernel(uint4* buf, size_t n16) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride)
        buf[i] = make_uint4((unsigned)i, 1u, 2u, 3u);
}

/* ---- launchers ------------------------------------------------------------------------------- */
int measure_grid(int n) {
    const int tiles = (n + kMeasureThreads - 1) / kMeasureThreads;
    const int cap = 148 * 4;   /* one B200: 148 SMs, 4 blocks of 128 threads resident per SM is ample */
    return tiles < cap ? (tiles > 0 ? tiles : 1) : cap;
}

void measure_init() { init_pairs(); }

/* K1 variant of one launch: lanes per query (1, 4, 8) or 32 = lv_search_coop_kernel.
 * Measured (profiles/r2_bench_*group*.json, r2_timeline*.txt): 4 lanes per query issue a quarter fewer instructions per query than
 * 8 (the prologue is shared by eight queries of a warp instead of four) and win when a launch has tens of thousands of queries;
 * 8 lanes have the shorter chain per query (a bucket of 36 points is one batch of loads instead of two) and win on the short
 * work lists of late evaluations and on small sweeps.  So the choice follows the number of queries the launch can expect:
 * all of them in the first evaluation, ~90 % / 45 % / 12 % in evaluations 2 / 3 / 4 of an update with neighbour reuse (cfg1).
 * LV_SEARCH_GROUP overrides for tuning runs and tests (read at every direct launch and when a handle's graph is built). */
static int search_group(const MeasureArgs& a, int eval) {
    const char* e = getenv("LV_SEARCH_GROUP");
    if (e) {
        const int group = atoi(e);
        if (group == 1 || group == 4 || group == 8 || group == 32) return group;
    }
    static const double kRedoShare[4] = {1.0, 0.9, 0.45, 0.12};
    const double share = (eval > 0 && a.ref) ? kRedoShare[eval < 3 ? eval : 3] : 1.0;
    return (double)a.n * share >= 40000.0 ? 4 : 8;
}
static int search_block(int group) { return group == 32 ? LV_COOP_THREADS : LV_SEARCH_THREADS; }
static int search_grid(const MeasureArgs& a, int group) {
    const int sgrid = group == 32 ? (int)(((int64_t)a.n + LV_COOP_THREADS - 1) / LV_COOP_THREADS)
                                  : (int)(((int64_t)a.n * group + LV_SEARCH_THREADS - 1) / LV_SEARCH_THREADS);
    return sgrid < 1 ? 1 : sgrid;
}
/* <<<>>> with the programmatic-dependent-launch attribute when `pdl` (see pdl_wait above) */
template <class... Params, class... Args>
static cudaError_t launch_k(void (*kernel)(Params...), unsigned grid, unsigned block, cudaStream_t st, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid, 1, 1);
    cfg.blockDim = dim3(block, 1, 1);
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = pdl ? at : nullptr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, Params(args)...);
}

template <bool LIST>
static void launch_search(const MeasureArgs& a, int group, int sgrid, cudaStream_t st, bool pdl) {
    switch (group) {
        case 1: launch_k(lv_search_kernel<1, LIST>, sgrid, LV_SEARCH_THREADS, st, pdl, a); break;
        case 32: launch_k(lv_search_coop_kernel<LIST>, sgrid, LV_COOP_THREADS, st, pdl, a); break;
        case 4: launch_k(lv_search_kernel<4, LIST>, sgrid, LV_SEARCH_THREADS, st, pdl, a); break;
        default: launch_k(lv_search_kernel<8, LIST>, sgrid, LV_SEARCH_THREADS, st, pdl, a); break;
    }
}

cudaError_t launch_measure(const MeasureArgs& a, int grid, cudaStream_t st, const MeasureProbe* probe, int reuse, int pdl) {
    init_pairs();
    const int group = search_group(a, reuse);          /* reuse = index of the evaluation within its update */
    const int sgrid = search_grid(a, group);
    /* work-list length, a spare word, redo-list length; inside an update with pdl the kernels
     * reset them themselves (begin kernel, fit kernel) so that every node of the update is a kernel */
    if (!pdl) cudaMemsetAsync(a.hard_count, 0, kCounters * sizeof(uint32_t), st);
    const unsigned qgrid = (unsigned)((a.n + LV_STAGE_QUERIES - 1) / LV_STAGE_QUERIES > 0 ? (a.n + LV_STAGE_QUERIES - 1) / LV_STAGE_QUERIES : 1);
    if (reuse && a.ref) {
        if (probe) probe->at(probe->ctx, 4);
        launch_k(lv_reuse_kernel, (a.n + 127) / 128 > 0 ? (a.n + 127) / 128 : 1, 128, st, pdl != 0, a);
        if (probe) probe->at(probe->ctx, 0);
        if (a.bin_key) launch_k(lv_search_staged_kernel<true>, qgrid, LV_STAGE_QUERIES, st, pdl != 0, a);
        else launch_search<true>(a, group, sgrid, st, pdl != 0);
    } else {
        if (probe) probe->at(probe->ctx, 0);
        if (a.bin_key) launch_k(lv_search_staged_kernel<false>, qgrid, LV_STAGE_QUERIES, st, pdl != 0, a);
        else launch_search<false>(a, group, sgrid, st, pdl != 0);
    }
    static const bool dbg_sync = getenv("LV_DEBUG_SYNC") != nullptr;   /* diagnosis: name the kernel that does not finish */
    if (dbg_sync) { cudaStreamSynchronize(st); fprintf(stderr, "[lv] search done\n"); fflush(stderr); }
    if (probe) probe->at(probe->ctx, 1);
    launch_k(lv_search_rings_kernel, kRingsGrid, 128, st, pdl != 0, a);
    if (dbg_sync) { cudaStreamSynchronize(st); fprintf(stderr, "[lv] search-rings done\n"); fflush(stderr); }
    if (probe) probe->at(probe->ctx, 2);
    launch_k(lv_fit_kernel, grid + (a.prep ? 1 : 0), kMeasureThreads, st, pdl != 0, a);
    if (dbg_sync) { cudaStreamSynchronize(st); fprintf(stderr, "[lv] fit done\n"); fflush(stderr); }
    if (probe) probe->at(probe->ctx, 3);
    return cudaGetLastError();
}
size_t bin_sort_tmp_bytes(int64_t max_points) {
    size_t bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const uint32_t*)nullptr,
                                    (uint32_t*)nullptr, (int)max_points, 0, 32);
    return bytes;
}
cudaError_t launch_bin(const MeasureArgs& a, cudaStream_t st, int pdl, int* launches) {
    launch_k(lv_bin_kernel, (unsigned)((a.n + 127) / 128 > 0 ? (a.n + 127) / 128 : 1), 128, st, pdl != 0, a);
    size_t tmp = a.sort_tmp_bytes;
    /* with a device-side job (graph replay) the sort covers the capacity a.n: positions past the sweep's n hold the
     * previous sweep's pairs, which lv_search_staged_kernel never reads (keys are sorted per launch over [0, a.n)) */
    cudaError_t e = cub::DeviceRadixSort::SortPairs(a.sort_tmp, tmp, a.bin_key_in, const_cast<uint32_t*>(a.bin_key), a.bin_val_in,
                                                    const_cast<uint32_t*>(a.bin_val), a.n, 0, a.sort_bits, st);
    if (launches) *launches += 1 + 4;
    return e != cudaSuccess ? e : cudaGetLastError();
}
cudaError_t launch_ieskf_begin(UpdateCtrl* c, MeasureJob* job, const float* xyz, int n, uint32_t* counters, cudaStream_t st) {
    lv_ieskf_begin_kernel<<<1, 256, 0, st>>>(c, job, xyz, n, counters);
    return cudaGetLastError();
}
const void* ieskf_begin_kernel_ptr() { return (const void*)lv_ieskf_begin_kernel; }
cudaError_t launch_ieskf_step(UpdateCtrl* c, const IeskfParams& prm, const double* partials, int n_partials,
                              cudaStream_t st, int pdl) {
    init_pairs();
    launch_k(lv_ieskf_step_kernel, 1, kStepThreads, st, pdl != 0, c, prm, partials, n_partials);
    return cudaGetLastError();
}
cudaError_t launch_reduce_partials(const double* partials, int n_partials, double* out, cudaStream_t st) {
    init_pairs();
    lv_reduce_partials_kernel<<<1, kStepThreads, 0, st>>>(partials, n_partials, out);
    return cudaGetLastError();
}
cudaError_t launch_predict(UpdateCtrl* c, const PredictNoise& noise, const double* d_imu, int k, cudaStream_t st) {
    lv_predict_kernel<<<1, 256, 0, st>>>(c, noise, d_imu, k);
    return cudaGetLastError();
}
cudaError_t launch_set_frame(UpdateCtrl* c, cudaStream_t st) {
    lv_set_frame_kernel<<<1, 32, 0, st>>>(c);
    return cudaGetLastError();
}
cudaError_t launch_l2_flush(void* buf, size_t bytes, cudaStream_t st) {
    lv_l2_flush_kernel<<<148 * 8, 256, 0, st>>>(reinterpret_cast<uint4*>(buf), bytes / 16);
    return cudaGetLastError();
}

}  // namespace lv

#ifdef LV_STEP_TIMING
extern "C" int lv_debug_step_clocks(long long* out) {
    return (int)cudaMemcpyFromSymbol(out, g_step_clk, sizeof(long long) * 64);
}
extern "C" int lv_debug_probes(unsigned long long* out) {
    cudaDeviceSynchronize();
    int e = (int)cudaMemcpyFromSymbol(out, g_probes, sizeof(unsigned long long) * 2);
    unsigned long long z[2] = {0, 0};
    cudaMemcpyToSymbol(g_probes, z, sizeof(z));
    return e;
}
/* out[5][8][8]; resets the table (starts to ~0, ends to 0) */
extern "C" int lv_debug_timeline(unsigned long long* out) {
    cudaDeviceSynchronize();
    int e = (int)cudaMemcpyFromSymbol(out, g_tl, sizeof(unsigned long long) * 320);
    unsigned long long init[320];
    for (int i = 0; i < 64; ++i) { init[i] = ~0ull; init[64 + i] = ~0ull; init[128 + i] = 0ull; init[192 + i] = 0ull; init[256 + i] = 0ull; }
    cudaMemcpyToSymbol(g_tl, init, sizeof(init));
    return e;
}
#endif
