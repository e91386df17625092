/*
 * lv_capi.cu — context object and the C ABI of liblimovelo_b200.so (include/limovelo_b200.h).
 *
 * One lv_context replaces the Localizator + Mapper singletons of the reference
 * (src/Modules/Localizator.cpp:100-103, include/Headers/Mapper.hpp:35-38): it owns the IKFoM
 * state mirror, the device map and the device buffers of one sequence, on one CUDA stream.
 * No CPU fallback exists: without a usable CUDA device every compute call returns LV_ERR_CUDA.
 */
#include <math.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/limovelo_b200.h"
#include "lv_host.h"
#include "lv_internal.h"
#include "lv_predict.h"

using namespace lv;

static_assert(sizeof(lv_iter_log) == sizeof(IterLog), "lv_iter_log must mirror lv::IterLog");
static_assert(LV_MAX_EVALS == kMaxEvals, "log capacity");
static_assert(LV_STATE_LEN == kStateLen && LV_DOF == kDof, "state layout");

static thread_local std::string g_last_error;
static void set_error(const std::string& s) { g_last_error = s; }

#define LV_CUDA(call)                                                                            \
    do {                                                                                         \
        cudaError_t e__ = (call);                                                                \
        if (e__ != cudaSuccess) {                                                                \
            char buf__[512];                                                                     \
            snprintf(buf__, sizeof(buf__), "%s:%d: %s -> %s", __FILE__, __LINE__, #call,         \
                     cudaGetErrorString(e__));                                                   \
            set_error(buf__);                                                                    \
            return LV_ERR_CUDA;                                                                  \
        }                                                                                        \
    } while (0)

struct EventPair { cudaEvent_t a, b; int kind; int upd; int slot; };   /* kind 0 measure, 1 solve, 2 build, 3 search, 4 search-upper, 5 fit */
enum { kNevalsRing = 4096 };

struct lv_context {
    lv_params prm;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    MapBuffers map;
    float* d_sweep = nullptr;          /* max_points x 3 */
    UpdateCtrl* d_ctrl = nullptr;
    UpdateCtrl* h_ctrl = nullptr;      /* pinned mirror for the D2H of results */
    double* d_partials = nullptr;
    double* d_group_rows = nullptr;    /* partials pre-reduced in groups of kPartialGroup rows (fit kernel) */
    uint32_t* d_group_tickets = nullptr;
    int4* d_nn_a = nullptr;            /* max_points: K1 -> K2 hand-over */
    int2* d_nn_b = nullptr;
    uint32_t* d_hard_list = nullptr;   /* kHardBuckets segments of hard_segment(max_points) entries, then kCounters counters */
    float4* d_ref = nullptr;           /* max_points: reuse reference (lv_reuse_kernel) */
    uint32_t* d_redo = nullptr;        /* max_points */
    uint32_t *d_bin_key = nullptr, *d_bin_val = nullptr, *d_bin_key_in = nullptr, *d_bin_val_in = nullptr;   /* sort_queries */
    uint8_t* d_redo_flag = nullptr;
    void* d_bin_tmp = nullptr;
    size_t bin_tmp_bytes = 0;
    double* d_imu = nullptr;           /* kImuBatch x 7: lv_propagate_device */
    double* h_imu = nullptr;           /* pinned */
    int64_t last_sweep_n = 0;          /* points of the sweep d_sweep holds (lv_correct / lv_measure*), for lv_map_add_last_sweep */
    const float* last_sweep = nullptr; /* device pointer of the sweep of the last update */
    bool use_reuse = true;
    bool use_pdl = true;               /* programmatic dependent launch between the kernels of an update */
    /* Compensator (deskew) staging: lazily allocated */
    lv_state32* d_path = nullptr;      /* deskew_max_states() */
    lv_state32* h_path = nullptr;      /* pinned */
    double* d_times = nullptr;         /* max_points */
    float* d_deskew_in = nullptr;      /* max_points x 3 */
    int* d_bad = nullptr;
    int* h_bad = nullptr;              /* pinned */
    DownsampleScratch ds;              /* downsamplers: grows with the largest cloud seen */
    float* d_ds_in = nullptr;          /* staging for the host-buffer variants */
    float* d_ds_out = nullptr;
    int64_t ds_stage_cap = 0;
    double* d_reduced = nullptr;       /* 157 doubles */
    double* h_reduced = nullptr;       /* pinned */
    void* d_flush = nullptr;
    /* per-point debug outputs (lazily allocated, max_points) */
    uint8_t* d_valid = nullptr; int32_t* d_nn_idx = nullptr; float* d_nn_sqd = nullptr;
    float* d_plane = nullptr; float* d_dist = nullptr; float* d_gworld = nullptr; double* d_rows = nullptr;
    /* host mirror of the filter (get_x / get_P) */
    double x[LV_STATE_LEN];
    double P[LV_DOF * LV_DOF];
    bool state_dirty = true;           /* host mirror newer than d_ctrl->x/P */
    bool pending_fetch = false;        /* device holds results not yet mirrored (lv_correct_device) */
    double last_time_updated = -1;
    lv_iter_log logs[LV_MAX_EVALS];
    int32_t n_evals = 0;
    int32_t last_status = LV_OK;
    /* profiling */
    bool profile = false;
    std::vector<EventPair> pending;
    std::vector<EventPair> pool;
    lv_profile prof;
    int32_t* h_nevals = nullptr;       /* pinned ring: n_evals of profiled updates */
    uint32_t update_seq = 0;
    IeskfParams iprm;
    /* one update = begin + (MAX_NUM_ITERS + 1) x (search, search-upper, fit, step): replayed as a CUDA graph
     * (one per sweep-capacity bucket) so that the host pays one launch instead of ~21 */
    struct UpdateGraph {
        int64_t cap;
        cudaGraph_t graph;
        cudaGraphExec_t exec;
        cudaGraphNode_t begin_node;
    };
    std::vector<UpdateGraph> graphs;
    MeasureJob* d_job = nullptr;
    bool use_graph = true;
};

static lv_status drain_events(lv_context* h) {
    if (h->pending.empty()) return LV_OK;
    LV_CUDA(cudaStreamSynchronize(h->stream));
    for (auto& e : h->pending) {
        float ms = 0;
        LV_CUDA(cudaEventElapsedTime(&ms, e.a, e.b));
        /* launches enqueued after the update had already finished return immediately: keep them apart */
        const bool idle = e.upd >= 0 && e.slot >= h->h_nevals[e.upd % kNevalsRing];
        if (idle) { h->prof.idle_ms += ms; h->prof.idle_launches++; }
        else if (e.kind == 0) { h->prof.measure_ms += ms; h->prof.measure_launches++; }
        else if (e.kind == 3) {
            h->prof.search_ms += ms; h->prof.measure_ms += ms; h->prof.measure_launches++;
            if (e.slot <= 0) { h->prof.search_first_ms += ms; h->prof.search_first_launches++; }
        }
        else if (e.kind == 4) { h->prof.search_upper_ms += ms; h->prof.measure_ms += ms; }
        else if (e.kind == 5) { h->prof.fit_ms += ms; h->prof.measure_ms += ms; }
        else if (e.kind == 6) { h->prof.reuse_ms += ms; h->prof.measure_ms += ms; }
        else if (e.kind == 1) { h->prof.solve_ms += ms; h->prof.solve_launches++; }
        else { h->prof.build_ms += ms; h->prof.build_launches++; }
        h->pool.push_back(e);
    }
    h->pending.clear();
    return LV_OK;
}
static bool prof_begin(lv_context* h, int kind, EventPair* ep) {
    if (!h->profile) return false;
    if (h->pending.size() > 2048) drain_events(h);
    if (h->pool.empty()) {
        EventPair e;
        if (cudaEventCreate(&e.a) != cudaSuccess || cudaEventCreate(&e.b) != cudaSuccess) return false;
        h->pool.push_back(e);
    }
    *ep = h->pool.back();
    h->pool.pop_back();
    ep->kind = kind;
    ep->upd = -1;
    ep->slot = 0;
    cudaEventRecord(ep->a, h->stream);
    return true;
}
static void prof_end(lv_context* h, EventPair* ep) {
    cudaEventRecord(ep->b, h->stream);
    h->pending.push_back(*ep);
}

static void fill_iprm(lv_context* h) {
    h->iprm.R = h->prm.LiDAR_noise;
    h->iprm.D = h->prm.degeneracy_threshold;
    for (int i = 0; i < kN; ++i) h->iprm.limits[i] = h->prm.LIMITS[i];
    h->iprm.max_iter = h->prm.MAX_NUM_ITERS;
    h->iprm.estimate_extrinsics = h->prm.estimate_extrinsics;
}

static MeasureArgs make_measure_args(lv_context* h, const float* d_xyz, int64_t n) {
    MeasureArgs a;
    memset(&a, 0, sizeof(a));
    a.xyz = d_xyz;
    a.n = (int32_t)n;
    a.n_tiles = (int32_t)((n + kMeasureThreads - 1) / kMeasureThreads);
    a.map = map_view(h->map);
    a.ctrl = h->d_ctrl;
    const double md = h->prm.MAX_DIST_PLANE;
    a.gate_d2 = md * md;
    float f = (float)a.gate_d2;
    if ((double)f < a.gate_d2) f = nextafterf(f, INFINITY);
    a.max_d2 = f;
    a.planes_threshold = h->prm.PLANES_THRESHOLD;
    a.estimate_extrinsics = h->prm.estimate_extrinsics;
    a.partials = h->d_partials;
    a.group_rows = h->d_group_rows;
    a.group_tickets = h->d_group_tickets;
    a.nn_a = h->d_nn_a;
    a.nn_b = h->d_nn_b;
    a.hard_list = h->d_hard_list;
    a.hard_seg = hard_segment(h->prm.max_points);
    a.hard_count = h->d_hard_list + (size_t)kHardBuckets * a.hard_seg;
    if (h->prm.sort_queries) {
        a.bin_key = h->d_bin_key; a.bin_val = h->d_bin_val; a.bin_key_in = h->d_bin_key_in; a.bin_val_in = h->d_bin_val_in;
        a.redo_flag = h->d_redo_flag;
        a.sort_tmp = h->d_bin_tmp; a.sort_tmp_bytes = h->bin_tmp_bytes;
        a.sort_bits = 0;
        for (uint32_t sl = h->map.slots; sl > 1; sl >>= 1) a.sort_bits++;
    }
    return a;
}

template <class T>
static cudaError_t ensure(T** p, size_t count) {
    if (*p) return cudaSuccess;
    return cudaMalloc(p, sizeof(T) * count);
}

extern "C" {

const char* lv_last_error(void) { return g_last_error.c_str(); }
const char* lv_version(void) { return "limovelo_b200 0.1 (sm_100a)"; }
/* the results are UpdateCtrl up to `prep`, which only the kernels of an update read */
static const size_t kResultBytes = offsetof(UpdateCtrl, prep);
int64_t lv_result_bytes(void) { return (int64_t)kResultBytes; }

/* every failure after `new lv_context` goes through here: nothing of a half-built context survives */
#define LV_CREATE_CUDA(call)                                                                     \
    do {                                                                                         \
        cudaError_t e__ = (call);                                                                \
        if (e__ != cudaSuccess) {                                                                \
            char buf__[512];                                                                     \
            snprintf(buf__, sizeof(buf__), "%s:%d: %s -> %s", __FILE__, __LINE__, #call,         \
                     cudaGetErrorString(e__));                                                   \
            lv_destroy(h);                                                                       \
            set_error(buf__);                                                                    \
            return LV_ERR_CUDA;                                                                  \
        }                                                                                        \
    } while (0)

lv_status lv_create(const lv_params* p, lv_handle* out) {
    if (!p || !out) return LV_ERR_ARG;
    *out = nullptr;
    /* all argument checks come before the first allocation */
    if (p->NUM_MATCH_POINTS != 5) { set_error("NUM_MATCH_POINTS must be 5 (5x3 plane fit)"); return LV_ERR_ARG; }
    if (p->MAX_NUM_ITERS < 0 || p->MAX_NUM_ITERS + 1 > LV_MAX_EVALS) {   /* 0: a single h-evaluation (esekfom.hpp:1634 runs i = -1 .. max-1) */
        set_error("MAX_NUM_ITERS out of range");
        return LV_ERR_ARG;
    }
    if (!(p->voxel_size > 0.f) || !(p->map_downsample_size > 0.f) || p->max_map_points <= 0 || p->max_points <= 0) {
        set_error("bad capacity / voxel_size / map_downsample_size");
        return LV_ERR_ARG;
    }
    if (p->max_map_points > (1ll << 24) || p->max_points > (1ll << 24)) { set_error("capacity beyond 2^24 points"); return LV_ERR_ARG; }
    if (!(p->MAX_DIST_PLANE > 0.0) || p->MAX_DIST_PLANE > 48.0 * (double)p->map_downsample_size) {
        set_error("MAX_DIST_PLANE must be positive and at most 48 map_downsample_size (ring search bound)");
        return LV_ERR_ARG;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        set_error("no CUDA device available (there is no CPU fallback)");
        return LV_ERR_CUDA;
    }
    LV_CUDA(cudaSetDevice(p->device));
    lv_context* h = new lv_context();
    h->prm = *p;
    memset(&h->prof, 0, sizeof(h->prof));
    memset(h->logs, 0, sizeof(h->logs));
    memset(&h->map, 0, sizeof(h->map));
    fill_iprm(h);
    if (p->stream) { h->stream = (cudaStream_t)p->stream; h->own_stream = false; }
    else { LV_CREATE_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)); h->own_stream = true; }
    LV_CREATE_CUDA(map_alloc(h->map, p->max_map_points, p->max_points, p->voxel_size, p->map_downsample_size));
    { int l = 0; LV_CREATE_CUDA(map_clear(h->map, h->stream, &l)); }
    LV_CREATE_CUDA(cudaMalloc(&h->d_sweep, sizeof(float) * 3 * p->max_points));
    LV_CREATE_CUDA(cudaMalloc(&h->d_nn_a, sizeof(int4) * p->max_points));
    LV_CREATE_CUDA(cudaMalloc(&h->d_nn_b, sizeof(int2) * p->max_points));
    LV_CREATE_CUDA(cudaMalloc(&h->d_hard_list, sizeof(uint32_t) * ((size_t)kHardBuckets * hard_segment(p->max_points) + kCounters)));
    LV_CREATE_CUDA(cudaMalloc(&h->d_ref, sizeof(float4) * p->max_points));
    LV_CREATE_CUDA(cudaMalloc(&h->d_redo, sizeof(uint32_t) * (p->max_points + 64)));   /* + one block of slack: read speculatively */
    /* hand-over buffers start defined: lv_search_kernel<.., LIST> reads redo_list[] before it knows the list's length, and a
     * first update's reuse kernel must not see stale neighbours (also keeps compute-sanitizer initcheck quiet) */
    LV_CREATE_CUDA(cudaMemset(h->d_redo, 0, sizeof(uint32_t) * (p->max_points + 64)));
    LV_CREATE_CUDA(cudaMemset(h->d_nn_a, 0xFF, sizeof(int4) * p->max_points));
    LV_CREATE_CUDA(cudaMemset(h->d_nn_b, 0xFF, sizeof(int2) * p->max_points));
    LV_CREATE_CUDA(cudaMemset(h->d_ref, 0, sizeof(float4) * p->max_points));
    LV_CREATE_CUDA(cudaMemset(h->d_hard_list, 0, sizeof(uint32_t) * ((size_t)kHardBuckets * hard_segment(p->max_points) + kCounters)));
    if (p->sort_queries) {
        LV_CREATE_CUDA(cudaMalloc(&h->d_bin_key, sizeof(uint32_t) * p->max_points));
        LV_CREATE_CUDA(cudaMalloc(&h->d_bin_val, sizeof(uint32_t) * p->max_points));
        LV_CREATE_CUDA(cudaMalloc(&h->d_bin_key_in, sizeof(uint32_t) * p->max_points));
        LV_CREATE_CUDA(cudaMalloc(&h->d_bin_val_in, sizeof(uint32_t) * p->max_points));
        LV_CREATE_CUDA(cudaMalloc(&h->d_redo_flag, p->max_points));
        LV_CREATE_CUDA(cudaMemset(h->d_redo_flag, 1, p->max_points));
        h->bin_tmp_bytes = bin_sort_tmp_bytes(p->max_points);
        LV_CREATE_CUDA(cudaMalloc(&h->d_bin_tmp, h->bin_tmp_bytes));
    }
    h->use_reuse = getenv("LV_NO_REUSE") == nullptr;
    h->use_pdl = getenv("LV_NO_PDL") == nullptr;
    LV_CREATE_CUDA(cudaMalloc(&h->d_job, sizeof(MeasureJob)));
    measure_init();
    h->use_graph = getenv("LV_NO_GRAPH") == nullptr;
    LV_CREATE_CUDA(cudaMalloc(&h->d_ctrl, sizeof(UpdateCtrl)));
    LV_CREATE_CUDA(cudaMemset(h->d_ctrl, 0, sizeof(UpdateCtrl)));
    LV_CREATE_CUDA(cudaMallocHost(&h->h_ctrl, sizeof(UpdateCtrl)));
    LV_CREATE_CUDA(cudaMalloc(&h->d_partials, sizeof(double) * kPartialStride * (148 * 4 + 8)));
    LV_CREATE_CUDA(cudaMemset(h->d_partials, 0, sizeof(double) * kPartialStride * (148 * 4 + 8)));
    LV_CREATE_CUDA(cudaMalloc(&h->d_group_rows, sizeof(double) * kPartialStride * 32));
    LV_CREATE_CUDA(cudaMemset(h->d_group_rows, 0, sizeof(double) * kPartialStride * 32));
    LV_CREATE_CUDA(cudaMalloc(&h->d_group_tickets, sizeof(uint32_t) * 32));
    LV_CREATE_CUDA(cudaMemset(h->d_group_tickets, 0, sizeof(uint32_t) * 32));
    LV_CREATE_CUDA(cudaMalloc(&h->d_reduced, sizeof(double) * 160));
    LV_CREATE_CUDA(cudaMallocHost(&h->h_reduced, sizeof(double) * 160));
    LV_CREATE_CUDA(cudaMallocHost(&h->h_nevals, sizeof(int32_t) * kNevalsRing));
    /* default filter state: identity pose, P = I (esekf constructor); callers normally follow
     * with lv_init_state or lv_set_state */
    for (int i = 0; i < LV_STATE_LEN; ++i) h->x[i] = 0;
    h->x[kRot + 3] = 1; h->x[kOffR + 3] = 1; h->x[kGrav] = LV_S2_LEN;
    for (int i = 0; i < LV_DOF * LV_DOF; ++i) h->P[i] = (i % (LV_DOF + 1) == 0) ? 1.0 : 0.0;
    *out = h;
    return LV_OK;
}

void lv_destroy(lv_handle h) {
    if (!h) return;
    cudaSetDevice(h->prm.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (auto& e : h->pending) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
    for (auto& e : h->pool) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
    for (auto& u : h->graphs) { cudaGraphExecDestroy(u.exec); cudaGraphDestroy(u.graph); }
    cudaFree(h->d_job); cudaFree(h->d_ref); cudaFree(h->d_redo); cudaFree(h->d_imu); cudaFreeHost(h->h_imu);
    cudaFree(h->d_bin_key); cudaFree(h->d_bin_val); cudaFree(h->d_bin_key_in); cudaFree(h->d_bin_val_in); cudaFree(h->d_redo_flag); cudaFree(h->d_bin_tmp);
    cudaFree(h->d_path); cudaFreeHost(h->h_path); cudaFree(h->d_times); cudaFree(h->d_deskew_in); cudaFree(h->d_bad); cudaFreeHost(h->h_bad);
    ds_free(h->ds); cudaFree(h->d_ds_in); cudaFree(h->d_ds_out);
    map_free(h->map);
    cudaFree(h->d_sweep); cudaFree(h->d_nn_a); cudaFree(h->d_nn_b); cudaFree(h->d_hard_list); cudaFree(h->d_ctrl); cudaFreeHost(h->h_ctrl); cudaFree(h->d_partials); cudaFree(h->d_group_rows); cudaFree(h->d_group_tickets);
    cudaFree(h->d_reduced); cudaFreeHost(h->h_reduced); cudaFreeHost(h->h_nevals); cudaFree(h->d_flush);
    cudaFree(h->d_valid); cudaFree(h->d_nn_idx); cudaFree(h->d_nn_sqd); cudaFree(h->d_plane);
    cudaFree(h->d_dist); cudaFree(h->d_gworld); cudaFree(h->d_rows);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

/* ---- Mapper ---------------------------------------------------------------------------------- */
/* device-side error flags of the map (table / arena exhausted) -> status.  Call after a stream synchronisation that
 * followed map_fetch_counters(). */
static lv_status map_status_from_mirror(lv_context* h) {
    const uint32_t err = h->map.h_counters[kCtrError];
    if (!err) return LV_OK;
    char buf[256];
    snprintf(buf, sizeof(buf), "device map out of capacity (flags 0x%x: 1 voxel table, 2 arena, 4 extent too large, 8 list, 16 block table): raise max_map_points",
             err);
    set_error(buf);
    return LV_ERR_CAPACITY;
}
static void count_map_launches(lv_context* h, int launches) { h->prof.total_launches += launches; }

static lv_status map_build_device_impl(lv_context* h, const float* d_xyz, int64_t m) {
    EventPair ep;
    const bool pr = prof_begin(h, 2, &ep);
    int launches = 0;
    LV_CUDA(map_clear(h->map, h->stream, &launches));
    LV_CUDA(map_add(h->map, d_xyz, m, 0, h->stream, &launches));              /* Build: no downsampling (Mapper.cpp:68-71) */
    if (pr) prof_end(h, &ep);
    count_map_launches(h, launches);
    return LV_OK;
}
static lv_status map_add_device_impl(lv_context* h, const float* d_xyz, int64_t n, int downsample) {
    EventPair ep;
    const bool pr = prof_begin(h, 2, &ep);
    int launches = 0;
    LV_CUDA(map_add(h->map, d_xyz, n, downsample ? 1 : 0, h->stream, &launches));
    if (pr) prof_end(h, &ep);
    count_map_launches(h, launches);
    return LV_OK;
}

lv_status lv_map_build(lv_handle h, const float* xyz, int64_t m) {
    if (!h || (!xyz && m > 0)) return LV_ERR_ARG;
    if (m <= 0) return LV_OK;                                    /* Mapper.cpp:23 */
    if (m > h->map.cap) { set_error("map capacity exceeded"); return LV_ERR_CAPACITY; }
    LV_CUDA(cudaSetDevice(h->prm.device));
    LV_CUDA(cudaMemcpyAsync(h->map.stage_xyz, xyz, sizeof(float) * 3 * m, cudaMemcpyHostToDevice, h->stream));
    return map_build_device_impl(h, h->map.stage_xyz, m);
}
lv_status lv_map_build_device(lv_handle h, const float* d_xyz, int64_t m) {
    if (!h || (!d_xyz && m > 0)) return LV_ERR_ARG;
    if (m <= 0) return LV_OK;
    if (m > h->map.cap) { set_error("map capacity exceeded"); return LV_ERR_CAPACITY; }
    LV_CUDA(cudaSetDevice(h->prm.device));
    return map_build_device_impl(h, d_xyz, m);
}
int64_t lv_map_size(lv_handle h) {
    if (!h || h->map.empty) return 0;
    if (cudaSetDevice(h->prm.device) != cudaSuccess) return -1;
    if (map_fetch_counters(h->map, h->stream) != cudaSuccess || cudaStreamSynchronize(h->stream) != cudaSuccess) return -1;
    map_status_from_mirror(h);
    return (int64_t)(int32_t)h->map.h_counters[kCtrPoints];
}
int lv_map_exists(lv_handle h) { return (h && !h->map.empty) ? 1 : 0; }
lv_status lv_map_status(lv_handle h) {
    if (!h) return LV_ERR_ARG;
    LV_CUDA(cudaSetDevice(h->prm.device));
    LV_CUDA(map_fetch_counters(h->map, h->stream));
    LV_CUDA(cudaStreamSynchronize(h->stream));
    return map_status_from_mirror(h);
}
int64_t lv_map_points(lv_handle h, float* out, int64_t cap) {
    if (!h || h->map.empty) return 0;
    if (cudaSetDevice(h->prm.device) != cudaSuccess) return -1;
    int64_t n = 0;
    if (map_points_sorted(h->map, out, cap, &n, h->stream) != cudaSuccess) return -1;
    return n;
}

lv_status lv_map_add(lv_handle h, const float* xyz, int64_t n, int downsample) {
    if (!h || (!xyz && n > 0)) return LV_ERR_ARG;
    if (n <= 0) return LV_OK;                                    /* Mapper.cpp:23 */
    if (h->map.empty) return lv_map_build(h, xyz, n);            /* Mapper.cpp:26 */
    if (n > h->map.add_cap) { set_error("more points than one lv_map_add can take (max_map_points)"); return LV_ERR_CAPACITY; }
    LV_CUDA(cudaSetDevice(h->prm.device));
    LV_CUDA(cudaMemcpyAsync(h->map.stage_xyz, xyz, sizeof(float) * 3 * n, cudaMemcpyHostToDevice, h->stream));
    return map_add_device_impl(h, h->map.stage_xyz, n, downsample);
}
lv_status lv_map_add_device(lv_handle h, const float* d_xyz, int64_t n, int downsample) {
    if (!h || (!d_xyz && n > 0)) return LV_ERR_ARG;
    if (n <= 0) return LV_OK;
    if (n > h->map.add_cap) { set_error("more points than one lv_map_add can take (max_map_points)"); return LV_ERR_CAPACITY; }
    LV_CUDA(cudaSetDevice(h->prm.device));
    if (h->map.empty) return map_build_device_impl(h, d_xyz, n);
    return map_add_device_impl(h, d_xyz, n, downsample);
}

/* ---- the tick on the device: main.cpp:99-105 ------------------------------------------------- */
static lv_status upload_state(lv_context* h, const double* x, const double* P);
static lv_status add_sweep_impl(lv_context* h, const float* d_xyz_lidar, int64_t n, int downsample) {
    if (h->state_dirty) {                                         /* the transform uses the device copy of the state */
        lv_status s = upload_state(h, h->x, h->P);
        if (s != LV_OK) return s;
        h->state_dirty = false;
    }
    EventPair ep;
    const bool pr = prof_begin(h, 2, &ep);
    int launches = 0;
    LV_CUDA(map_add_sweep(h->map, h->d_ctrl, d_xyz_lidar, n, downsample ? 1 : 0, h->stream, &launches));
    if (pr) prof_end(h, &ep);
    count_map_launches(h, launches);
    return LV_OK;
}
lv_status lv_map_add_sweep_device(lv_handle h, const float* d_xyz_lidar, int64_t n, int downsample) {
    if (!h || (!d_xyz_lidar && n > 0)) return LV_ERR_ARG;
    if (n <= 0) return LV_OK;
    if (n > h->map.add_cap) { set_error("more points than one lv_map_add can take (max_map_points)"); return LV_ERR_CAPACITY; }
    LV_CUDA(cudaSetDevice(h->prm.device));
    return add_sweep_impl(h, d_xyz_lidar, n, downsample);
}
lv_status lv_map_add_last_sweep(lv_handle h, int downsample) {
    if (!h) return LV_ERR_ARG;
    if (!h->last_sweep || h->last_sweep_n <= 0) { set_error("no sweep has been corrected yet"); return LV_ERR_ARG; }
    LV_CUDA(cudaSetDevice(h->prm.device));
    return add_sweep_impl(h, h->last_sweep, h->last_sweep_n, downsample);
}

/* ---- state ----------------------------------------------------------------------------------- */
static lv_status fetch_results(lv_context* h);
static lv_status sync_mirror(lv_context* h) {   /* bring the host mirror up to date after lv_correct_device */
    if (!h->pending_fetch) return LV_OK;
    if (cudaSetDevice(h->prm.device) != cudaSuccess) return LV_ERR_CUDA;
    fetch_results(h);
    return LV_OK;
}

lv_status lv_set_state(lv_handle h, const double* x, const double* P) {
    if (!h) return LV_ERR_ARG;
    if (!(x && P)) sync_mirror(h);
    if (x) memcpy(h->x, x, sizeof(h->x));
    if (P) memcpy(h->P, P, sizeof(h->P));
    h->state_dirty = true;
    return LV_OK;
}
lv_status lv_get_state(lv_handle h, double* x, double* P) {
    if (!h) return LV_ERR_ARG;
    sync_mirror(h);
    if (x) memcpy(x, h->x, sizeof(h->x));
    if (P) memcpy(P, h->P, sizeof(h->P));
    return LV_OK;
}
lv_status lv_init_state(lv_handle h, const float q_imu[4]) {
    if (!h || !q_imu) return LV_ERR_ARG;
    lvh_init_state(h->prm, q_imu, h->x, h->P);
    h->state_dirty = true;
    return LV_OK;
}
lv_status lv_predict(lv_handle h, const double acc[3], const double gyro[3], double dt) {
    if (!h || !acc || !gyro) return LV_ERR_ARG;
    sync_mirror(h);
    lvh_predict(h->prm, acc, gyro, dt, h->x, h->P);
    h->state_dirty = true;
    return LV_OK;
}
/* Localizator::propagate_to on the device (Localizator.cpp:59-75): k IMU samples, one launch, no host round trip */
lv_status lv_propagate_device(lv_handle h, const double* acc, const double* gyro, const double* dt, int32_t k) {
    enum { kImuBatch = 512 };
    if (!h || !acc || !gyro || !dt || k < 0) return LV_ERR_ARG;
    if (k == 0) return LV_OK;
    LV_CUDA(cudaSetDevice(h->prm.device));
    if (!h->d_imu) {
        LV_CUDA(cudaMalloc(&h->d_imu, sizeof(double) * 7 * kImuBatch));
        LV_CUDA(cudaMallocHost(&h->h_imu, sizeof(double) * 7 * kImuBatch));
    }
    if (h->state_dirty) {                                         /* the host mirror is newer (lv_set_state / lv_predict): bring it over */
        lv_status s = upload_state(h, h->x, h->P);
        if (s != LV_OK) return s;
        h->state_dirty = false;
    }
    const PredictNoise noise = {h->prm.covariance_gyroscope, h->prm.covariance_acceleration, h->prm.covariance_bias_gyroscope,
                                h->prm.covariance_bias_acceleration};
    for (int32_t s0 = 0; s0 < k; s0 += kImuBatch) {
        const int32_t kb = k - s0 < kImuBatch ? k - s0 : kImuBatch;
        if (s0 > 0) LV_CUDA(cudaStreamSynchronize(h->stream));    /* the pinned staging buffer is reused */
        for (int32_t i = 0; i < kb; ++i) {
            for (int a = 0; a < 3; ++a) { h->h_imu[7 * i + a] = acc[3 * (s0 + i) + a]; h->h_imu[7 * i + 3 + a] = gyro[3 * (s0 + i) + a]; }
            h->h_imu[7 * i + 6] = dt[s0 + i];
        }
        LV_CUDA(cudaMemcpyAsync(h->d_imu, h->h_imu, sizeof(double) * 7 * kb, cudaMemcpyHostToDevice, h->stream));
        LV_CUDA(launch_predict(h->d_ctrl, noise, h->d_imu, kb, h->stream));
        h->prof.total_launches += 1;
    }
    h->pending_fetch = true;                                      /* the device now holds the newest (x, P) */
    return LV_OK;
}
double lv_last_time_updated(lv_handle h) { return h ? h->last_time_updated : -1; }

static lv_status upload_state(lv_context* h, const double* x, const double* P) {
    /* x, P are staged through the pinned mirror so the copy is truly asynchronous */
    memcpy(h->h_ctrl->x, x, sizeof(double) * kStateLen);
    if (P) memcpy(h->h_ctrl->P, P, sizeof(double) * kN * kN);
    /* x and P are adjacent in UpdateCtrl: one copy (each small copy costs several microseconds of latency) */
    static_assert(offsetof(UpdateCtrl, P) == offsetof(UpdateCtrl, x) + sizeof(double) * kStateLen, "x, P adjacent");
    LV_CUDA(cudaMemcpyAsync(h->d_ctrl->x, h->h_ctrl->x, sizeof(double) * (kStateLen + (P ? kN * kN : 0)),
                            cudaMemcpyHostToDevice, h->stream));
    return LV_OK;
}

/* launch_measure() with one CUDA-event pair per kernel when profiling is on (never inside a capture) */
static cudaError_t launch_measure_timed(lv_context* h, const MeasureArgs& a, int grid, int allow_events, int reuse,
                                        int upd, int slot, int pdl = 0) {
    if (!h->profile || !allow_events) return launch_measure(a, grid, h->stream, nullptr, reuse, pdl);
    struct Ctx { lv_context* h; EventPair ep; bool on; int upd, slot; } ctx = {h, EventPair(), false, upd, slot};
    MeasureProbe probe;
    probe.ctx = &ctx;
    probe.at = [](void* p, int stage) {
        Ctx* c = static_cast<Ctx*>(p);
        if (c->on) prof_end(c->h, &c->ep);
        c->on = false;
        if (stage != 3) {         /* 4: reuse kernel follows, 0: search, 1: search-upper, 2: fit, 3: end */
            c->on = prof_begin(c->h, stage == 4 ? 6 : 3 + stage, &c->ep);
            c->ep.upd = c->upd; c->ep.slot = c->slot;
        }
    };
    return launch_measure(a, grid, h->stream, &probe, reuse, 0);   /* events between the kernels: no pdl */
}

/* ---- the update ------------------------------------------------------------------------------ */
static MeasureArgs update_measure_args(lv_context* h, const float* d_xyz, int64_t n, bool as_job) {
    MeasureArgs a = make_measure_args(h, d_xyz, n);
    a.prep = h->d_ctrl;                                           /* ieskf_prepare rides in the fit kernel */
    if (as_job) a.job = h->d_job;
    if (h->use_reuse) { a.ref = h->d_ref; a.redo_list = h->d_redo; }
    return a;
}

/* enqueue begin + all evaluations on h->stream; with `job` the sweep comes from device memory (graph capture) */
static lv_status enqueue_update_kernels(lv_context* h, const float* d_xyz, int64_t n, bool as_job);

static lv_status build_update_graph(lv_context* h, int64_t cap, lv_context::UpdateGraph* out) {
    cudaGraph_t graph = nullptr;
    LV_CUDA(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
    lv_status s = enqueue_update_kernels(h, nullptr, cap, true);
    cudaError_t e = cudaStreamEndCapture(h->stream, &graph);
    if (s != LV_OK || e != cudaSuccess) {
        if (graph) cudaGraphDestroy(graph);
        if (e != cudaSuccess) { set_error(cudaGetErrorString(e)); return LV_ERR_CUDA; }
        return s;
    }
    out->cap = cap;
    out->graph = graph;                 /* kept: the node handles below belong to it */
    LV_CUDA(cudaGraphInstantiate(&out->exec, graph, 0));
    /* the one node patched per launch is the begin kernel (sweep pointer and size); the measurement kernels' arguments
     * embed the map view, which never changes over the life of a handle (tables and arena are allocated once) */
    size_t n_nodes = 0;
    LV_CUDA(cudaGraphGetNodes(graph, nullptr, &n_nodes));
    std::vector<cudaGraphNode_t> nodes(n_nodes);
    LV_CUDA(cudaGraphGetNodes(graph, nodes.data(), &n_nodes));
    out->begin_node = nullptr;
    for (cudaGraphNode_t nd : nodes) {
        cudaGraphNodeType t;
        LV_CUDA(cudaGraphNodeGetType(nd, &t));
        if (t != cudaGraphNodeTypeKernel) continue;
        cudaKernelNodeParams kp;
        LV_CUDA(cudaGraphKernelNodeGetParams(nd, &kp));
        if (kp.func == ieskf_begin_kernel_ptr()) out->begin_node = nd;
    }
    if (!out->begin_node) { set_error("update graph: begin node not found"); return LV_ERR_CUDA; }
    return LV_OK;
}

static lv_status enqueue_update(lv_context* h, const float* d_xyz, int64_t n) {
    if (h->state_dirty) {
        lv_status s = upload_state(h, h->x, h->P);
        if (s != LV_OK) return s;
        h->state_dirty = false;
    }
    if (h->profile || !h->use_graph) return enqueue_update_kernels(h, d_xyz, n, false);
    int64_t cap = 4096;
    while (cap < n) cap <<= 1;
    if (cap > h->prm.max_points) cap = h->prm.max_points;
    lv_context::UpdateGraph* g = nullptr;
    for (auto& u : h->graphs) if (u.cap == cap) g = &u;
    if (!g) {
        lv_context::UpdateGraph u;
        lv_status s = build_update_graph(h, cap, &u);
        if (s != LV_OK) return s;
        h->graphs.push_back(u);
        g = &h->graphs.back();
    }
    UpdateCtrl* c = h->d_ctrl;
    MeasureJob* job = h->d_job;
    int n32 = (int)n;
    uint32_t* counters = h->d_hard_list + (size_t)kHardBuckets * hard_segment(h->prm.max_points);
    void* args[5] = {&c, &job, &d_xyz, &n32, &counters};
    cudaKernelNodeParams kp = {};
    kp.func = const_cast<void*>(ieskf_begin_kernel_ptr());
    kp.gridDim = dim3(1, 1, 1);
    kp.blockDim = dim3(256, 1, 1);
    kp.kernelParams = args;
    LV_CUDA(cudaGraphExecKernelNodeSetParams(g->exec, g->begin_node, &kp));
    LV_CUDA(cudaGraphLaunch(g->exec, h->stream));
    h->prof.total_launches += 1 + 4 * (h->prm.MAX_NUM_ITERS + 1) + (h->use_reuse ? h->prm.MAX_NUM_ITERS : 0) + (h->prm.sort_queries ? 5 : 0);
    return LV_OK;
}

static lv_status enqueue_update_kernels(lv_context* h, const float* d_xyz, int64_t n, bool as_job) {
    const int pdl = (h->use_pdl && !h->profile) ? 1 : 0;
    uint32_t* counters = h->d_hard_list + (size_t)kHardBuckets * hard_segment(h->prm.max_points);
    LV_CUDA(launch_ieskf_begin(h->d_ctrl, as_job ? h->d_job : nullptr, d_xyz, (int)n, counters, h->stream));
    if (!as_job) h->prof.total_launches += 1;
    MeasureArgs a = update_measure_args(h, d_xyz, n, as_job);
    const int grid = measure_grid((int)n);
    if (a.bin_key) {                                              /* once per update: the sweep binned by home voxel */
        int l = 0;
        LV_CUDA(launch_bin(a, h->stream, pdl, &l));
        if (!as_job) h->prof.total_launches += l;
    }
    for (int e = 0; e <= h->prm.MAX_NUM_ITERS; ++e) {            /* i = -1 .. max_iter-1, esekfom.hpp:1634 */
        EventPair ep;
        bool pr;
        LV_CUDA(launch_measure_timed(h, a, grid, as_job ? 0 : 1, e /* evaluation index: > 0 = reuse + work list */, (int)(h->update_seq % kNevalsRing), e, pdl));
        pr = prof_begin(h, 1, &ep);
        ep.upd = (int)(h->update_seq % kNevalsRing); ep.slot = e;
        LV_CUDA(launch_ieskf_step(h->d_ctrl, h->iprm, h->d_group_rows, partial_groups(grid), h->stream, pdl));
        if (pr) prof_end(h, &ep);
        if (!as_job) h->prof.total_launches += 4 + ((e > 0 && h->use_reuse) ? 1 : 0);
    }
    if (h->profile) {
        LV_CUDA(cudaMemcpyAsync(&h->h_nevals[h->update_seq % kNevalsRing], &h->d_ctrl->n_evals, sizeof(int32_t),
                                cudaMemcpyDeviceToHost, h->stream));
        h->update_seq++;
    }
    return LV_OK;
}

static lv_status fetch_results(lv_context* h) {
    LV_CUDA(cudaMemcpyAsync(h->h_ctrl, h->d_ctrl, kResultBytes, cudaMemcpyDeviceToHost, h->stream));
    LV_CUDA(map_fetch_counters(h->map, h->stream));       /* 64 bytes: the map's error flags ride along */
    LV_CUDA(cudaStreamSynchronize(h->stream));
    const UpdateCtrl* c = h->h_ctrl;
    memcpy(h->x, c->x, sizeof(h->x));
    if (c->status == LV_OK) memcpy(h->P, c->P, sizeof(h->P));
    h->n_evals = c->n_evals;
    memcpy(h->logs, c->logs, sizeof(h->logs));
    h->last_status = c->status;
    h->state_dirty = false;
    h->pending_fetch = false;
    if (c->status == LV_OK && map_status_from_mirror(h) != LV_OK) return LV_ERR_CAPACITY;
    return (lv_status)c->status;
}

lv_status lv_correct(lv_handle h, const float* xyz, int64_t n, double time, lv_iter_log* logs, int32_t* n_evals,
                     double* x_out, double* P_out) {
    if (!h || !xyz || n <= 0) return LV_ERR_ARG;
    if (n_evals) *n_evals = 0;
    if (h->map.empty) return LV_EMPTY_MAP;                       /* Localizator.cpp:24 */
    if (n > h->prm.max_points) { set_error("sweep capacity exceeded"); return LV_ERR_CAPACITY; }
    LV_CUDA(cudaSetDevice(h->prm.device));
    LV_CUDA(cudaMemcpyAsync(h->d_sweep, xyz, sizeof(float) * 3 * n, cudaMemcpyHostToDevice, h->stream));
    lv_status s = enqueue_update(h, h->d_sweep, n);
    if (s != LV_OK) return s;
    h->last_sweep = h->d_sweep; h->last_sweep_n = n;
    s = fetch_results(h);
    h->last_time_updated = time;                                  /* Localizator.cpp:26 */
    if (logs) memcpy(logs, h->logs, sizeof(lv_iter_log) * (size_t)h->n_evals);
    if (n_evals) *n_evals = h->n_evals;
    if (x_out) memcpy(x_out, h->x, sizeof(h->x));
    if (P_out) memcpy(P_out, h->P, sizeof(h->P));
    return s;
}

lv_status lv_correct_device(lv_handle h, const float* d_xyz, int64_t n, double time) {
    if (!h || !d_xyz || n <= 0) return LV_ERR_ARG;
    if (h->map.empty) return LV_EMPTY_MAP;
    LV_CUDA(cudaSetDevice(h->prm.device));
    lv_status s = enqueue_update(h, d_xyz, n);
    h->last_sweep = d_xyz; h->last_sweep_n = n;
    h->last_time_updated = time;
    h->pending_fetch = true;
    return s;
}

lv_status lv_last_logs(lv_handle h, lv_iter_log* logs, int32_t* n_evals) {
    if (!h) return LV_ERR_ARG;
    LV_CUDA(cudaSetDevice(h->prm.device));
    lv_status s = fetch_results(h);
    if (logs) memcpy(logs, h->logs, sizeof(lv_iter_log) * (size_t)h->n_evals);
    if (n_evals) *n_evals = h->n_evals;
    return s;
}

/* ---- operator boundary ----------------------------------------------------------------------- */
static lv_status run_measure_once(lv_context* h, const double* x, const float* xyz, int64_t n, bool want_rows,
                                  bool want_debug) {
    if (n > h->prm.max_points) { set_error("sweep capacity exceeded"); return LV_ERR_CAPACITY; }
    LV_CUDA(cudaSetDevice(h->prm.device));
    LV_CUDA(cudaMemcpyAsync(h->d_sweep, xyz, sizeof(float) * 3 * n, cudaMemcpyHostToDevice, h->stream));
    lv_status s = upload_state(h, x, nullptr);
    if (s != LV_OK) return s;
    h->state_dirty = true;   /* d_ctrl->x no longer mirrors the filter */
    LV_CUDA(launch_set_frame(h->d_ctrl, h->stream));
    MeasureArgs a = make_measure_args(h, h->d_sweep, n);
    const size_t mp = (size_t)h->prm.max_points;
    if (want_rows) { LV_CUDA(ensure(&h->d_rows, 13 * mp)); LV_CUDA(ensure(&h->d_valid, mp)); a.rows = h->d_rows; a.valid = h->d_valid; }
    if (want_debug) {
        LV_CUDA(ensure(&h->d_valid, mp)); LV_CUDA(ensure(&h->d_nn_idx, 5 * mp)); LV_CUDA(ensure(&h->d_nn_sqd, 5 * mp));
        LV_CUDA(ensure(&h->d_plane, 4 * mp)); LV_CUDA(ensure(&h->d_dist, mp)); LV_CUDA(ensure(&h->d_gworld, 3 * mp));
        a.valid = h->d_valid; a.nn_idx = h->d_nn_idx; a.nn_sqd = h->d_nn_sqd; a.plane = h->d_plane; a.dist = h->d_dist;
        a.g_world = h->d_gworld;
    }
    const int grid = measure_grid((int)n);
    if (a.bin_key) { int l = 0; LV_CUDA(launch_bin(a, h->stream, 0, &l)); h->prof.total_launches += l; }
    LV_CUDA(launch_measure_timed(h, a, grid, 1, 0, -1, 0));
    LV_CUDA(launch_reduce_partials(h->d_group_rows, partial_groups(grid), h->d_reduced, h->stream));
    LV_CUDA(cudaMemcpyAsync(h->h_reduced, h->d_reduced, sizeof(double) * 157, cudaMemcpyDeviceToHost, h->stream));
    h->prof.total_launches += 5;
    return LV_OK;
}

lv_status lv_measure_reduced(lv_handle h, const double* x, const float* xyz, int64_t n, double* HTH, double* HTh,
                             int64_t* nm) {
    if (!h || !x || !xyz || n <= 0) return LV_ERR_ARG;
    if (nm) *nm = 0;
    if (h->map.empty) return LV_EMPTY_MAP;
    lv_status s = run_measure_once(h, x, xyz, n, false, false);
    if (s != LV_OK) return s;
    LV_CUDA(cudaStreamSynchronize(h->stream));
    if (HTH) memcpy(HTH, h->h_reduced, sizeof(double) * 144);
    if (HTh) memcpy(HTh, h->h_reduced + 144, sizeof(double) * 12);
    if (nm) *nm = (int64_t)h->h_reduced[156];
    return LV_OK;
}

lv_status lv_measure(lv_handle h, const double* x, const float* xyz, int64_t n, double* h_x, double* h_vec, int64_t* nm) {
    if (!h || !x || !xyz || n <= 0 || !nm) return LV_ERR_ARG;
    *nm = 0;
    if (h->map.empty) return LV_EMPTY_MAP;
    lv_status s = run_measure_once(h, x, xyz, n, true, false);
    if (s != LV_OK) return s;
    std::vector<double> rows(13 * (size_t)n);
    std::vector<uint8_t> valid((size_t)n);
    LV_CUDA(cudaMemcpyAsync(rows.data(), h->d_rows, sizeof(double) * 13 * n, cudaMemcpyDeviceToHost, h->stream));
    LV_CUDA(cudaMemcpyAsync(valid.data(), h->d_valid, (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    LV_CUDA(cudaStreamSynchronize(h->stream));
    /* compaction in input order = the single-thread order of Mapper::match (Mapper.cpp:46-53);
     * layout: column-major Nm x 12 like Eigen::MatrixXd (Localizator.cpp:31) */
    int64_t cnt = 0;
    for (int64_t i = 0; i < n; ++i) cnt += valid[i] ? 1 : 0;
    int64_t k = 0;
    for (int64_t i = 0; i < n; ++i) {
        if (!valid[i]) continue;
        if (h_x)
            for (int c = 0; c < 12; ++c) h_x[(size_t)c * cnt + k] = rows[13 * (size_t)i + c];
        if (h_vec) h_vec[k] = rows[13 * (size_t)i + 12];
        ++k;
    }
    *nm = cnt;
    return LV_OK;
}

lv_status lv_match_all(lv_handle h, const double* x, const float* xyz, int64_t n, uint8_t* valid, int32_t* nn_idx,
                       float* nn_sqd, float* plane, float* dist, float* g_world) {
    if (!h || !x || !xyz || n <= 0) return LV_ERR_ARG;
    if (h->map.empty) return LV_EMPTY_MAP;
    lv_status s = run_measure_once(h, x, xyz, n, false, true);
    if (s != LV_OK) return s;
    if (valid) LV_CUDA(cudaMemcpyAsync(valid, h->d_valid, (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    if (nn_idx) LV_CUDA(cudaMemcpyAsync(nn_idx, h->d_nn_idx, sizeof(int32_t) * 5 * n, cudaMemcpyDeviceToHost, h->stream));
    if (nn_sqd) LV_CUDA(cudaMemcpyAsync(nn_sqd, h->d_nn_sqd, sizeof(float) * 5 * n, cudaMemcpyDeviceToHost, h->stream));
    if (plane) LV_CUDA(cudaMemcpyAsync(plane, h->d_plane, sizeof(float) * 4 * n, cudaMemcpyDeviceToHost, h->stream));
    if (dist) LV_CUDA(cudaMemcpyAsync(dist, h->d_dist, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    if (g_world) LV_CUDA(cudaMemcpyAsync(g_world, h->d_gworld, sizeof(float) * 3 * n, cudaMemcpyDeviceToHost, h->stream));
    LV_CUDA(cudaStreamSynchronize(h->stream));
    return LV_OK;
}


/* the neighbours the LAST evaluation of the last update (or operator call) handed to the plane fit, as map point ids:
 * after an update with neighbour reuse these are the stored five where lv_reuse_kernel vouched for them and the fresh
 * search's elsewhere — what lv_match_all (always a fresh search) cannot show */
__global__ void lv_neighbour_ids_kernel(const int4* nn_a, const int2* nn_b, const float4* arena, int n, int32_t* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int4 a = nn_a[i];
    const int2 b = nn_b[i];
    const int id[5] = {a.x, a.y, a.z, a.w, b.x};
    for (int k = 0; k < 5; ++k) out[5 * i + k] = (b.x >= 0 && id[k] >= 0) ? __float_as_int(arena[id[k]].w) : -1;
}
lv_status lv_last_neighbours(lv_handle h, int64_t n, int32_t* nn_idx) {
    if (!h || !nn_idx || n <= 0 || n > h->prm.max_points) return LV_ERR_ARG;
    if (h->map.empty) return LV_EMPTY_MAP;
    LV_CUDA(cudaSetDevice(h->prm.device));
    LV_CUDA(ensure(&h->d_nn_idx, 5 * (size_t)h->prm.max_points));
    lv_neighbour_ids_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(h->d_nn_a, h->d_nn_b, h->map.arena, (int)n, h->d_nn_idx);
    LV_CUDA(cudaGetLastError());
    LV_CUDA(cudaMemcpyAsync(nn_idx, h->d_nn_idx, sizeof(int32_t) * 5 * (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    LV_CUDA(cudaStreamSynchronize(h->stream));
    return LV_OK;
}

/* ---- utilities ------------------------------------------------------------------------------- */
void* lv_host_alloc(int64_t bytes) {
    void* p = nullptr;
    if (bytes <= 0 || cudaMallocHost(&p, (size_t)bytes) != cudaSuccess) return nullptr;
    return p;
}
void lv_host_free(void* p) { if (p) cudaFreeHost(p); }
void* lv_device_alloc(lv_handle h, int64_t bytes) {
    if (!h || bytes <= 0) return nullptr;
    void* p = nullptr;
    cudaSetDevice(h->prm.device);
    if (cudaMalloc(&p, (size_t)bytes) != cudaSuccess) return nullptr;
    return p;
}
void lv_device_free(lv_handle h, void* p) { if (h && p) { cudaSetDevice(h->prm.device); cudaFree(p); } }
lv_status lv_memcpy_h2d(lv_handle h, void* dst, const void* src, int64_t bytes) {
    if (!h || !dst || !src || bytes < 0) return LV_ERR_ARG;
    LV_CUDA(cudaSetDevice(h->prm.device));
    LV_CUDA(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyHostToDevice, h->stream));
    LV_CUDA(cudaStreamSynchronize(h->stream));
    return LV_OK;
}
/* ---- Compensator::compensate ------------------------------------------------------------------ */
static lv_status deskew_common(lv_context* h, const lv_state32* path, int32_t ns, const lv_state32* Xt2,
                               const float* d_xyz, const double* d_t, int64_t n, float* d_out) {
    if (!h->d_path) {
        LV_CUDA(cudaMalloc(&h->d_path, sizeof(lv_state32) * deskew_max_states()));
        LV_CUDA(cudaMallocHost(&h->h_path, sizeof(lv_state32) * deskew_max_states()));
        LV_CUDA(cudaMalloc(&h->d_bad, sizeof(int)));
        LV_CUDA(cudaMallocHost(&h->h_bad, sizeof(int)));
    }
    memcpy(h->h_path, path, sizeof(lv_state32) * (size_t)ns);
    LV_CUDA(cudaMemcpyAsync(h->d_path, h->h_path, sizeof(lv_state32) * (size_t)ns, cudaMemcpyHostToDevice, h->stream));
    LV_CUDA(launch_deskew(h->d_path, ns, *Xt2, path[0].time, path[ns - 1].time, d_xyz, d_t, n, d_out, h->d_bad, h->stream));
    LV_CUDA(cudaMemcpyAsync(h->h_bad, h->d_bad, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    h->prof.total_launches += 2;
    return LV_OK;
}
static lv_status deskew_args_ok(lv_context* h, const lv_state32* path, int32_t ns, const lv_state32* Xt2, const void* a,
                                const void* b, int64_t n, const void* c) {
    if (!h || !path || !Xt2 || !a || !b || !c || n <= 0 || ns < 2) return LV_ERR_ARG;
    if (ns > deskew_max_states()) { set_error("deskew path too long"); return LV_ERR_CAPACITY; }
    if (n > h->prm.max_points) { set_error("sweep capacity exceeded"); return LV_ERR_CAPACITY; }
    for (int32_t s = 1; s < ns; ++s)
        if (!(path[s - 1].time <= path[s].time)) { set_error("deskew path not sorted by time"); return LV_ERR_ARG; }
    return LV_OK;
}
lv_status lv_compensate_device(lv_handle h, const lv_state32* path, int32_t ns, const lv_state32* Xt2,
                               const float* d_xyz, const double* d_t, int64_t n, float* d_xyz_out) {
    lv_status s = deskew_args_ok(h, path, ns, Xt2, d_xyz, d_t, n, d_xyz_out);
    if (s != LV_OK) return s;
    LV_CUDA(cudaSetDevice(h->prm.device));
    s = deskew_common(h, path, ns, Xt2, d_xyz, d_t, n, d_xyz_out);
    if (s != LV_OK) return s;
    LV_CUDA(cudaStreamSynchronize(h->stream));
    if (*h->h_bad) { set_error("deskew: a timestamp lies outside the path or the points are not time-sorted"); return LV_ERR_ARG; }
    return LV_OK;
}
lv_status lv_compensate(lv_handle h, const lv_state32* path, int32_t ns, const lv_state32* Xt2, const float* xyz,
                        const double* t, int64_t n, float* xyz_out) {
    lv_status s = deskew_args_ok(h, path, ns, Xt2, xyz, t, n, xyz_out);
    if (s != LV_OK) return s;
    LV_CUDA(cudaSetDevice(h->prm.device));
    if (!h->d_times) {
        LV_CUDA(cudaMalloc(&h->d_times, sizeof(double) * h->prm.max_points));
        LV_CUDA(cudaMalloc(&h->d_deskew_in, sizeof(float) * 3 * h->prm.max_points));
    }
    LV_CUDA(cudaMemcpyAsync(h->d_deskew_in, xyz, sizeof(float) * 3 * n, cudaMemcpyHostToDevice, h->stream));
    LV_CUDA(cudaMemcpyAsync(h->d_times, t, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
    s = deskew_common(h, path, ns, Xt2, h->d_deskew_in, h->d_times, n, h->d_deskew_in);
    if (s != LV_OK) return s;
    LV_CUDA(cudaMemcpyAsync(xyz_out, h->d_deskew_in, sizeof(float) * 3 * n, cudaMemcpyDeviceToHost, h->stream));
    LV_CUDA(cudaStreamSynchronize(h->stream));
    if (*h->h_bad) { set_error("deskew: a timestamp lies outside the path or the points are not time-sorted"); return LV_ERR_ARG; }
    return LV_OK;
}

/* ---- downsamplers ------------------------------------------------------------------------------- */
static lv_status ds_stage(lv_context* h, int64_t n) {
    if (n <= h->ds_stage_cap) return LV_OK;
    cudaFree(h->d_ds_in); cudaFree(h->d_ds_out);
    h->d_ds_in = h->d_ds_out = nullptr;
    h->ds_stage_cap = 0;
    const int64_t cap = n + n / 4 + 1024;
    LV_CUDA(cudaMalloc(&h->d_ds_in, sizeof(float) * 3 * cap));
    LV_CUDA(cudaMalloc(&h->d_ds_out, sizeof(float) * 3 * cap));
    h->ds_stage_cap = cap;
    return LV_OK;
}
lv_status lv_voxelgrid_downsample_device(lv_handle h, const float* d_xyz, int64_t n, float leaf, float* d_xyz_out, int64_t* n_out) {
    if (!h || !d_xyz || !d_xyz_out || !n_out || n < 0 || !(leaf > 0.f) || n > 0x7fffffff) return LV_ERR_ARG;
    *n_out = 0;
    if (n == 0) return LV_OK;
    LV_CUDA(cudaSetDevice(h->prm.device));
    LV_CUDA(ds_reserve(h->ds, n));
    int launches = 0;
    LV_CUDA(launch_voxelgrid(h->ds, d_xyz, n, leaf, d_xyz_out, h->stream, &launches));
    h->prof.total_launches += launches;
    LV_CUDA(cudaStreamSynchronize(h->stream));
    if (h->ds.h_count[1]) {
        /* pcl::VoxelGrid::applyFilter warns "Leaf size is too small for the input dataset. Integer indices would overflow."
         * and hands the input on unchanged; Compensator::voxelgrid_downsample carries on with it.  Same here. */
        set_error("voxel grid: leaf size too small for the extent of the cloud (cell index overflows): input passed through");
        if (d_xyz_out != d_xyz) LV_CUDA(cudaMemcpyAsync(d_xyz_out, d_xyz, sizeof(float) * 3 * (size_t)n, cudaMemcpyDeviceToDevice, h->stream));
        LV_CUDA(cudaStreamSynchronize(h->stream));
        *n_out = n;
        return LV_OK;
    }
    *n_out = h->ds.h_count[0];
    return LV_OK;
}
lv_status lv_voxelgrid_downsample(lv_handle h, const float* xyz, int64_t n, float leaf, float* xyz_out, int64_t* n_out) {
    if (!h || !xyz || !xyz_out || !n_out || n < 0 || !(leaf > 0.f) || n > 0x7fffffff) return LV_ERR_ARG;
    *n_out = 0;
    if (n == 0) return LV_OK;
    LV_CUDA(cudaSetDevice(h->prm.device));
    lv_status s = ds_stage(h, n);
    if (s != LV_OK) return s;
    LV_CUDA(cudaMemcpyAsync(h->d_ds_in, xyz, sizeof(float) * 3 * n, cudaMemcpyHostToDevice, h->stream));
    s = lv_voxelgrid_downsample_device(h, h->d_ds_in, n, leaf, h->d_ds_out, n_out);
    if (s != LV_OK) return s;
    LV_CUDA(cudaMemcpyAsync(xyz_out, h->d_ds_out, sizeof(float) * 3 * (size_t)*n_out, cudaMemcpyDeviceToHost, h->stream));
    LV_CUDA(cudaStreamSynchronize(h->stream));
    return LV_OK;
}
lv_status lv_temporal_downsample(lv_handle h, const float* xyz, int64_t n, int32_t rate, double min_dist, float* xyz_out,
                                 int32_t* idx_out, int64_t* n_out) {
    if (!h || !xyz || !xyz_out || !n_out || n < 0 || n > 0x7fffffff) return LV_ERR_ARG;
    *n_out = 0;
    if (n == 0) return LV_OK;
    LV_CUDA(cudaSetDevice(h->prm.device));
    lv_status s = ds_stage(h, n);
    if (s != LV_OK) return s;
    LV_CUDA(ds_reserve(h->ds, n));
    LV_CUDA(cudaMemcpyAsync(h->d_ds_in, xyz, sizeof(float) * 3 * n, cudaMemcpyHostToDevice, h->stream));
    int launches = 0;
    LV_CUDA(launch_temporal(h->ds, h->d_ds_in, n, rate, min_dist, h->d_ds_out, nullptr, h->stream, &launches));
    h->prof.total_launches += launches;
    LV_CUDA(cudaStreamSynchronize(h->stream));
    const int64_t m = h->ds.h_count[0];
    LV_CUDA(cudaMemcpyAsync(xyz_out, h->d_ds_out, sizeof(float) * 3 * (size_t)m, cudaMemcpyDeviceToHost, h->stream));
    if (idx_out) LV_CUDA(cudaMemcpyAsync(idx_out, h->ds.sel, sizeof(int32_t) * (size_t)m, cudaMemcpyDeviceToHost, h->stream));
    LV_CUDA(cudaStreamSynchronize(h->stream));
    *n_out = m;
    return LV_OK;
}

lv_status lv_synchronize(lv_handle h) {
    if (!h) return LV_ERR_ARG;
    LV_CUDA(cudaSetDevice(h->prm.device));
    LV_CUDA(cudaStreamSynchronize(h->stream));
    return LV_OK;
}
lv_status lv_profile_enable(lv_handle h, int on) {
    if (!h) return LV_ERR_ARG;
    h->profile = on != 0;
    return LV_OK;
}
lv_status lv_profile_get(lv_handle h, lv_profile* out, int reset) {
    if (!h || !out) return LV_ERR_ARG;
    LV_CUDA(cudaSetDevice(h->prm.device));
    lv_status s = drain_events(h);
    if (s != LV_OK) return s;
    *out = h->prof;
    if (reset) memset(&h->prof, 0, sizeof(h->prof));
    return LV_OK;
}
lv_status lv_flush_l2(lv_handle h) {
    if (!h) return LV_ERR_ARG;
    LV_CUDA(cudaSetDevice(h->prm.device));
    const size_t bytes = 256ull << 20;
    if (!h->d_flush) LV_CUDA(cudaMalloc(&h->d_flush, bytes));
    LV_CUDA(launch_l2_flush(h->d_flush, bytes, h->stream));
    h->prof.total_launches += 1;
    return LV_OK;
}

}  // extern "C"
