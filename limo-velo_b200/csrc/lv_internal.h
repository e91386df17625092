/*
 * lv_internal.h — launcher declarations shared by the translation units of liblimovelo_b200.so.
 */
#ifndef LV_INTERNAL_H_
#define LV_INTERNAL_H_

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/limovelo_b200.h"
#include "lv_ieskf.h"
#include "lv_voxel_search.h"

namespace lv {

enum { kMeasureThreads = 128, kPartialStride = 96, kStepThreads = 256, kPartialGroup = 32 };
inline int partial_groups(int grid) { return (grid + kPartialGroup - 1) / kPartialGroup; }
/* The search kernel appends its uncertified queries to one of 32 lists picked by block index: thousands of atomics on
 * ONE counter cost it a 9 us tail on the first evaluation of an update (tools/timeline.py). */
enum { kHardBuckets = 32, kCounters = 4 + kHardBuckets };
/* a bucket receives the queries of every 32nd block: at most n / 32 + (queries per block <= 128) of them */
inline uint32_t hard_segment(int64_t n) { return (uint32_t)((n + kHardBuckets - 1) / kHardBuckets + 160); }

/* the sweep of an update replayed from a CUDA graph: written by the begin kernel (whose arguments are the
 * only thing patched per launch), read by the measurement kernels instead of MeasureArgs::xyz / n / n_tiles */
struct MeasureJob {
    const float* xyz;
    int32_t n;
    int32_t n_tiles;
};

/* per-launch constants of the measurement kernels (reuse, search, search-upper, fit) */
struct MeasureArgs {
    const float* xyz;          /* n x 3 packed, LiDAR frame                               */
    int32_t n;                 /* with `job`: the capacity the grids were sized for       */
    int32_t n_tiles;           /* ceil(n / kMeasureThreads)                               */
    const MeasureJob* job;     /* non-NULL: xyz / n / n_tiles come from device memory      */
    VoxelMapView map;
    const UpdateCtrl* ctrl;    /* frame + done flag                                       */
    UpdateCtrl* prep;          /* non-NULL: block 0 of the fit kernel runs ieskf_prepare() */
    float max_d2;              /* smallest float >= MAX_DIST_PLANE^2 (search radius^2)    */
    double gate_d2;            /* MAX_DIST_PLANE^2 in double (Plane.cpp:42)               */
    float planes_threshold;
    int32_t estimate_extrinsics;
    double* partials;          /* [grid][kPartialStride]: 78 + 12 sums, count             */
    double* group_rows;        /* [partial_groups(grid)][kPartialStride]: the partials summed in groups of kPartialGroup rows */
    uint32_t* group_tickets;   /* [partial_groups(grid)]: blocks of the group that have finished (fit kernel)                  */
    /* optional per-point outputs (NULL on the hot path) */
    uint8_t* valid;
    int32_t* nn_idx;
    float* nn_sqd;
    float* plane;
    float* dist;
    float* g_world;
    double* rows;              /* n x 13 (row[12], h)                                     */
    int4* nn_a;                /* n: search result handed from K1 to K2 (neighbours 0..3)      */
    int2* nn_b;                /* n: (neighbour 4, bits of the 5th squared distance)         */
    uint32_t* hard_list;       /* queries level 0 could not certify (K1 -> K1b): kHardBuckets segments of hard_seg entries */
    uint32_t hard_seg;         /* capacity of one segment                                      */
    uint32_t* hard_count;      /* [2] length of redo_list, [4 .. 4 + kHardBuckets) lengths of the segments; kCounters words */
    /* reuse of neighbours across the evaluations of one update (NULL: off) */
    float4* ref;               /* n: world position the stored neighbours were searched from + outsider bound */
    uint32_t* redo_list;       /* n: queries whose neighbours could not be reused (Kv -> K1)  */
    /* binned order of the sweep (lv_params.sort_queries; NULL: per-query search from global memory) */
    const uint32_t* bin_key;   /* n: home-voxel slot at the propagated state, ascending (0xFFFFFFFF: none) */
    const uint32_t* bin_val;   /* n: the query at that position                                            */
    uint32_t* bin_key_in;      /* n: unsorted, written by lv_bin_kernel                                    */
    uint32_t* bin_val_in;
    uint8_t* redo_flag;        /* n: 1 = search again (written by lv_reuse_kernel)                         */
    void* sort_tmp;            /* cub::DeviceRadixSort scratch for n pairs                                 */
    size_t sort_tmp_bytes;
    int32_t sort_bits;         /* significant bits of a slot index                                         */
};

/* device map storage (layout: lv_voxel_map.h) + scratch of one add */
struct MapBuffers {
    MapGrid grid;
    uint4* table;              /* voxel slots (2 x uint4 each)                               */
    uint32_t slots;
    uint4* btable;             /* block slots                                                 */
    uint32_t bslots;
    float4* arena;             /* own extents + halo buckets                                  */
    uint32_t arena_cap;
    uint32_t* counters;        /* kMapCounters device words                                   */
    uint32_t* h_counters;      /* pinned mirror (map_fetch_counters)                          */
    uint32_t* touched;
    uint32_t* dirty;
    uint32_t list_cap;
    float* stage_xyz;          /* device copy of host points handed to lv_map_build / lv_map_add: add_cap x 3 */
    uint32_t *skeys, *skeys_alt, *svals, *svals_alt;   /* sort of the new points (add_cap each) */
    void* sort_tmp;
    size_t sort_tmp_bytes;
    int sort_bits;
    int64_t cap;               /* max_map_points (sizes the tables and the arena)             */
    int64_t add_cap;           /* most points one build / add can take                        */
    int64_t n_inserted;        /* ids handed out so far                                       */
    bool empty;                /* nothing was ever added (Mapper::exists, Mapper.cpp:32-34)   */
};

cudaError_t map_alloc(MapBuffers& b, int64_t max_map_points, int64_t max_points, float voxel_size, float ds);
void map_free(MapBuffers& b);
/* empty the map (table, block table, counters); asynchronous */
cudaError_t map_clear(MapBuffers& b, cudaStream_t st, int* launches);
/* KD_TREE::Build (downsample = 0 on an empty map) / Add_Points: n points in DEVICE memory; asynchronous, no host round trip */
cudaError_t map_add(MapBuffers& b, const float* d_xyz, int64_t n, int downsample, cudaStream_t st, int* launches);
/* the sweep (LiDAR frame, device) transformed by the state in d_ctrl->x, then map_add: main.cpp:99-105 without leaving the GPU */
cudaError_t map_add_sweep(MapBuffers& b, const UpdateCtrl* d_ctrl, const float* d_xyz_lidar, int64_t n, int downsample, cudaStream_t st,
                          int* launches);
cudaError_t map_fetch_counters(MapBuffers& b, cudaStream_t st);
cudaError_t map_points_sorted(MapBuffers& b, float* host_out, int64_t cap, int64_t* n_out, cudaStream_t st);
VoxelMapView map_view(const MapBuffers& b);

int measure_grid(int n);
/* `probe` (optional) is called on the launching thread before the search (stage 0), after it (1), after the
 * upper-level search (2) and after the fit (3): the profiler records its events there */
struct MeasureProbe { void (*at)(void* ctx, int stage); void* ctx; };
/* reuse = index of the evaluation within its update; != 0 (needs a.ref): lv_reuse_kernel first, then the search only
 * over the queries it could not vouch for; the probe then sees stage 4 before the reuse kernel.  The index also picks
 * the shape of the level-0 search kernel (search_group() in lv_measure.cu). */
cudaError_t launch_measure(const MeasureArgs& a, int grid, cudaStream_t st, const MeasureProbe* probe = nullptr,
                           int reuse = 0, int pdl = 0);
/* once per update when a.bin_key is set: lv_bin_kernel + radix sort of the (slot, query) pairs */
cudaError_t launch_bin(const MeasureArgs& a, cudaStream_t st, int pdl, int* launches);
size_t bin_sort_tmp_bytes(int64_t max_points);
cudaError_t launch_ieskf_begin(UpdateCtrl* c, MeasureJob* job, const float* xyz, int n, uint32_t* counters, cudaStream_t st);
const void* ieskf_begin_kernel_ptr();
void measure_init();                          /* constant tables; call once before any capture           */
cudaError_t launch_ieskf_step(UpdateCtrl* c, const IeskfParams& prm, const double* partials, int n_partials,
                              cudaStream_t st, int pdl = 0);
/* stand-alone reduction of the partials (operator-boundary calls): out[0:144) HTH, [144:156) HTh, [156] Nm */
cudaError_t launch_reduce_partials(const double* partials, int n_partials, double* out, cudaStream_t st);
struct PredictNoise;
cudaError_t launch_predict(UpdateCtrl* c, const PredictNoise& noise, const double* d_imu, int k, cudaStream_t st);
cudaError_t launch_set_frame(UpdateCtrl* c, cudaStream_t st);   /* frame from c->x, done = 0 */
cudaError_t launch_l2_flush(void* buf, size_t bytes, cudaStream_t st);

/* lv_downsample.cu: PointCloudProcessor::temporal_downsample and Compensator::voxelgrid_downsample */
struct DownsampleScratch {
    int64_t cap = 0;
    uint32_t *keys = nullptr, *keys_sorted = nullptr, *vals = nullptr, *vals_sorted = nullptr;
    uint8_t* flags = nullptr;
    int32_t* sel = nullptr;
    void* tmp = nullptr;
    size_t tmp_bytes = 0;
    void* box = nullptr;           /* GridBox */
    int* count = nullptr;
    int* h_count = nullptr;        /* pinned: [0] output count, [1] overflow flag */
};
cudaError_t ds_reserve(DownsampleScratch& s, int64_t n);
void ds_free(DownsampleScratch& s);
cudaError_t launch_voxelgrid(DownsampleScratch& s, const float* d_xyz, int64_t n, float leaf, float* d_out, cudaStream_t st,
                             int* launches);
cudaError_t launch_temporal(DownsampleScratch& s, const float* d_xyz, int64_t n, int rate, double min_dist, float* d_out,
                            int32_t* d_idx_out, cudaStream_t st, int* launches);

/* lv_deskew.cu: Compensator::compensate.  d_bad (one int) is set when a timestamp is out of range / out of order */
int deskew_max_states();
cudaError_t launch_deskew(const lv_state32* d_path, int ns, const lv_state32& Xt2, double t_lo, double t_hi,
                          const float* d_xyz, const double* d_t, int64_t n, float* d_out, int* d_bad, cudaStream_t st);

}  // namespace lv
#endif
