// Shared host/device helpers for libradarb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <utility>
#include <vector>

#include "radarb200.h"

#define RB_WARP 32

struct rb_scratch {
    void* ptr = nullptr;
    size_t cap = 0;
};

// Named scratch slots; each grows on demand and is reused across calls.
enum rb_slot {
    RB_S_TILE_STATUS = 0,   // spoke: tile survivor counts, in-sweep tile prefixes, sweep totals
    RB_S_SWEEP_FLAGS,       // spoke: self-cleaning counters (done, ticket)
    RB_S_SPOKE_MASK,        // spoke: survivor bitmask, 1 bit per cell
    RB_S_REDUCE,            // bounds partials
    RB_S_KEEP,              // land filter keep flags
    RB_S_BLOCKSUM,          // scan block sums
    RB_S_BLOCKSUM2,
    RB_S_CELL_ID,           // dbscan: cell id per point
    RB_S_CELL_START,        // dbscan: cell start table
    RB_S_CELL_FILL,
    RB_S_SORT_IDX,
    RB_S_SX, RB_S_SY, RB_S_SZ, RB_S_ST,
    RB_S_CORE,
    RB_S_PARENT,
    RB_S_MINORIG,
    RB_S_FLAGS,
    RB_S_RANK,
    RB_S_SLABEL,
    RB_S_STATS,
    RB_S_MISC,
    RB_S_FUSE_GRID,         // max fusion: the dense grids of one group of frames
    RB_S_FUSE_FRAMES,       // max fusion: per-frame bounds, grid sizes and offsets
    RB_S_FUSE_TILES,        // max fusion: occupied cells per grid tile, their scan
    RB_S_COMP_KEY,          // dbscan: component key per point (original order)
    RB_S_PIPE, RB_S_PIPE_EDGES, RB_S_PIPE_TIMES,   // rb_detect_block: sweep bases + bounds, device edges, times
    RB_S_B_NCORE, RB_S_B_PARENT, RB_S_B_LABEL, RB_S_B_MINKEY, RB_S_CORE_START, RB_S_CB_LIST,   // dbscan, tight: per-bucket arrays
    RB_S_CSV,               // csv ingest: newline counts per chunk, their scan, newline offsets
    RB_S_CLUSTERS,          // cluster records: (frame, label) slot tables, tile lists, segment scans
    RB_S_LAND_FLAG,         // land accumulate: "an intensity is not a small integer" flag
    RB_S_SHARD_IDS, RB_S_SHARD_LOCAL, RB_S_SHARD_KEYS,   // time-sharded driver: staged frame ids, local frame list, key flags / ranks
    RB_S_GROUP_TMP,         // rb_stable_group: frame offsets of its single frame
    RB_S_LAND_ORDERED,      // land accumulate, ordered path: cell ids, grouped intensities, segment table
    RB_S_REC_FRAMES,        // windowed ST-DBSCAN: frame offsets, frame ids
    RB_S_REC_LOCAL,         // windowed ST-DBSCAN: times, global index, keys, labels, core flags of one window
    RB_S_REC_KEYS,          // windowed ST-DBSCAN: every window's run-length encoded zone keys
    RB_S_REC_KEYS_BIG,      // windowed ST-DBSCAN: encodings of the windows that outgrew the capacity guess
    RB_S_REC_TABLE,         // windowed ST-DBSCAN: the stitched key -> cluster id table
    RB_S_REC_CORE,          // windowed ST-DBSCAN: recording-wide core flags when the caller passes none
    RB_S_REC_FLAG,          // windowed ST-DBSCAN: hint-violation flag, kept from pass 1 to pass 3
    RB_S_PLY_TILES,         // PLY formatter: bytes of each block of lines, then their scan
    RB_S_COUNT
};

struct rb_db_plan;
struct rb_comm;

struct rb_ctx {
    int device = 0;
    int sm_count = 0;
    int cc_major = 0, cc_minor = 0;
    int64_t l2_bytes = 0;
    int64_t launches = 0;
    rb_scratch slots[RB_S_COUNT];
    std::vector<void*> retired;      // outgrown scratch buffers, freed in rb_destroy (never while work may be in flight)
    void* pinned = nullptr;          // small pinned staging buffer (host)
    size_t pinned_cap = 0;
    rb_dbscan_stats last_stats;
    rb_db_plan* db_plan = nullptr;   // state shared by the rb_stdbscan_* phases (dbscan.cu)
    rb_comm* comm = nullptr;         // NCCL communicator of this context (comm.cu, rb_comm_init)
    int64_t rec_key_cap = 0;         // windowed ST-DBSCAN: zone-encoding capacity guess (largest seen, bounded; recording.cu)
    int opt_dbscan_mode = 0;         // 0 = auto, 1 = always the general algorithm, 2 = require the tight one
    int opt_spoke_mask_variant = 0;  // 0 = auto, 1 = register-staged mask kernel, 2 = require the TMA-staged one
    int spoke_last_variant = 0;      // mask kernel the last rb_spoke_to_points launched (1 / 2)
    int land_last_variant = 0;       // accumulation the last rb_land_accumulate[_ordered] ran (1 = shared, 2 = global, 3 = ordered)
    int opt_spoke_profile = 0;       // 1: record events around the three spoke-to-point kernels
    int opt_spoke_ring = 2;          // TMA ring of the mask kernel: 0 = 64 KiB x 3, 1 = 32 KiB x 4, 2 = 32 KiB x 3 (default), 3 = 48 KiB x 2
    int opt_spoke_l2_hint = 1;       // 1: the mask kernel's bulk loads carry an L2 evict-first policy
    int opt_mask_priority = 1;       // 1: the mask kernel is launched with the device's highest launch priority
    int prio_high = 0;               // that priority (cudaDeviceGetStreamPriorityRange)
    int opt_mask_gate = 1;           // 1: the mask kernels of all contexts of a device run one after the other (see spoke.cu)
    int64_t opt_fuse_group_cells = 0; // > 0: grid cells one group of rb_fuse_max_frames may hold (0 = 2^28)
    int opt_carveout = -1;           // >= 0: every launch asks for this shared-memory carve-out (percent), see rb_launch
    unsigned attr_spoke_mask = 0;    // per-context "function attribute set" flags (a context = one device)
    bool attr_land = false;
    cudaEvent_t spoke_ev[4] = {nullptr, nullptr, nullptr, nullptr};
};

void rb_set_error(const char* fmt, ...);
void rb_db_plan_free(rb_ctx* ctx);
void rb_comm_free(rb_ctx* ctx);
int rb_scratch_get(rb_ctx* ctx, rb_slot slot, size_t bytes, void** out);

#define RB_CUDA(call)                                                                      \
    do {                                                                                   \
        cudaError_t _e = (call);                                                           \
        if (_e != cudaSuccess) {                                                           \
            rb_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
            return RB_ERR_CUDA;                                                            \
        }                                                                                  \
    } while (0)

#define RB_LAUNCH_CHECK(ctx)                                                               \
    do {                                                                                   \
        (ctx)->launches++;                                                                 \
        cudaError_t _e = cudaGetLastError();                                               \
        if (_e != cudaSuccess) {                                                           \
            rb_set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return RB_ERR_CUDA;                                                            \
        }                                                                                  \
    } while (0)

#define RB_REQUIRE(cond, msg)                                                              \
    do {                                                                                   \
        if (!(cond)) {                                                                     \
            rb_set_error("%s:%d: %s", __FILE__, __LINE__, msg);                            \
            return RB_ERR_ARG;                                                             \
        }                                                                                  \
    } while (0)

#define RB_TRY(expr)                                                                       \
    do {                                                                                   \
        int _rc = (expr);                                                                  \
        if (_rc != RB_OK) return _rc;                                                      \
    } while (0)

static inline int64_t rb_div_up(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Every kernel of the library is launched through here. With the "carveout" option set, each launch carries the same
// preferred shared-memory carve-out: an SM runs CTAs of different kernels side by side only when they agree on its
// L1 / shared-memory split, so this is what lets the latency-bound clustering kernels of one block be resident next to
// the HBM-bound mask kernel of the next (blocks in flight on different streams).
#ifdef __CUDACC__
template <typename... KArgs, typename... Args>
inline cudaError_t rb_launch_prio(rb_ctx* ctx, bool high_priority, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                  cudaStream_t stream, Args&&... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    unsigned na = 0;
    if (ctx->opt_carveout >= 0) {
        attr[na].id = cudaLaunchAttributePreferredSharedMemoryCarveout;
        attr[na].val.sharedMemCarveout = (unsigned)ctx->opt_carveout;
        ++na;
    }
    if (high_priority && ctx->opt_mask_priority) {
        // CTAs of a higher-priority launch are dispatched before the waiting CTAs of the other grids: the 148 persistent
        // CTAs of the HBM-bound mask kernel must not queue behind the thousands of CTAs of another block's kernels
        attr[na].id = cudaLaunchAttributePriority;
        attr[na].val.priority = ctx->prio_high;
        ++na;
    }
    if (na) { cfg.attrs = attr; cfg.numAttrs = na; }
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
template <typename... KArgs, typename... Args>
inline cudaError_t rb_launch(rb_ctx* ctx, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                             Args&&... args) {
    return rb_launch_prio(ctx, false, kernel, grid, block, smem, stream, std::forward<Args>(args)...);
}
#endif

// ---- device helpers ---------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ unsigned rb_lane() { return threadIdx.x & 31u; }
__device__ __forceinline__ unsigned rb_lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}
// streaming 128-bit load: read-only path, do not allocate in L1
__device__ __forceinline__ float4 rb_ld_stream4(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ unsigned long long rb_ld_acquire_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void rb_st_release_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ int rb_ld_acquire_s32(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void rb_st_release_s32(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int rb_ld_relaxed_s32(const int* p) {
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
#endif

// device-wide exclusive scan of int32 -> int32 (n < 2^31); total written to *total_out (device, optional)
int rb_exclusive_scan_i32(rb_ctx* ctx, const int32_t* in, int32_t* out, int64_t n,
                          int32_t* total_out, cudaStream_t stream);

// ST-DBSCAN without the final counter read-back (dbscan.cu); with a hint nothing in it syncs. min_frames > 0: the
// PointCloudWorkF variant (rb_stdbscan_wf)
int rb_stdbscan_enqueue(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride, const float* times,
                        int64_t n, double eps_space, float eps_time, int min_samples, int32_t* labels, uint8_t* core,
                        const rb_stdbscan_hint* hint, void* stream, int min_frames = 0);
int rb_stdbscan_fetch_stats(rb_ctx* ctx, int64_t* n_clusters, void* stream);
// phases for the windowed driver (recording.cu): set every core flag right after a plan; the plan's hint-violation word
int rb_stdbscan_set_cores_planned(rb_ctx* ctx, const uint8_t* core_in, void* stream);
int rb_stdbscan_hint_flag(rb_ctx* ctx, const unsigned long long** flag);
// ... and for its min_frames variant: switch the current plan to it (0 = back to the T4 rules); the WF border rule with
// recording-wide indices gidx[plan's n] and per cluster id the smallest core index of the whole cluster, start_of
int rb_stdbscan_set_min_frames(rb_ctx* ctx, int min_frames);
int rb_stdbscan_assign_global(rb_ctx* ctx, const int32_t* core_label, int32_t* labels, const int64_t* gidx, const int64_t* start_of,
                              void* stream);
// device flag "rb_land_accumulate saw an intensity that is not a small integer" of this context (land.cu)
int rb_land_inexact_flag(rb_ctx* ctx, int32_t** flag, cudaStream_t stream);
// bounds of the first *n_dev points (n_dev on the device, at most n_max): no host knowledge of n needed (land.cu)
int rb_bounds_devn(rb_ctx* ctx, const float* x, const float* y, const int64_t* n_dev, int64_t n_max, float* out4, cudaStream_t stream);
