// Context, error text, scratch arena and the device-wide exclusive scan used by the other stages.
#include <stdarg.h>
#include <stdlib.h>

#include "common.cuh"

static thread_local char g_err[512] = "";

void rb_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

extern "C" const char* rb_last_error(void) { return g_err; }
extern "C" int rb_version(void) { return 1; }

extern "C" int rb_create(int device, rb_ctx** out) {
    if (!out) { rb_set_error("rb_create: out is NULL"); return RB_ERR_ARG; }
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        rb_set_error("rb_create: no CUDA device (%s); this library has no CPU fallback",
                     e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return RB_ERR_CUDA;
    }
    if (device < 0 || device >= n) { rb_set_error("rb_create: bad device %d of %d", device, n); return RB_ERR_ARG; }
    // the caller's current device is left as it was: every entry point works on the device of the buffers / stream it is
    // given (one process per GPU is the norm; a caller that drives several devices sets the current device itself)
    int prev = -1;
    RB_CUDA(cudaGetDevice(&prev));
    struct Restore { int d; ~Restore() { if (d >= 0) cudaSetDevice(d); } } restore{prev == device ? -1 : prev};
    RB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    RB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        rb_set_error("rb_create: device %d is sm_%d%d; this build is sm_100a only", device, prop.major, prop.minor);
        return RB_ERR_CUDA;
    }
    rb_ctx* ctx = new rb_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->cc_major = prop.major;
    ctx->cc_minor = prop.minor;
    ctx->l2_bytes = prop.l2CacheSize;
    int prio_low = 0, prio_high = 0;
    if (cudaDeviceGetStreamPriorityRange(&prio_low, &prio_high) == cudaSuccess) ctx->prio_high = prio_high;
    memset(&ctx->last_stats, 0, sizeof ctx->last_stats);
    ctx->pinned_cap = 1 << 20;                     // 1 MiB: frame offsets of 130k frames fit without a re-allocation
    e = cudaMallocHost(&ctx->pinned, ctx->pinned_cap);
    if (e != cudaSuccess) {
        rb_set_error("rb_create: cudaMallocHost -> %s", cudaGetErrorString(e));
        delete ctx;
        return RB_ERR_NOMEM;
    }
    // diagnostic defaults from the environment (experiments that must reach every context of a process, worker threads'
    // included): RB_OPT_<NAME>=<integer> is rb_set_option(ctx, "<name>", value)
    static const char* const env_opts[] = {"carveout", "spoke_ring", "spoke_l2_hint", "dbscan_mode", "spoke_mask_variant", "mask_gate", "mask_priority"};
    for (const char* name : env_opts) {
        char var[64] = "RB_OPT_";
        size_t k = strlen(var);
        for (const char* c = name; *c && k + 1 < sizeof var; ++c) var[k++] = (char)(*c >= 'a' && *c <= 'z' ? *c - 32 : *c);
        var[k] = 0;
        const char* v = getenv(var);
        if (v && *v && rb_set_option(ctx, name, atoll(v)) != RB_OK) { rb_destroy(ctx); return RB_ERR_ARG; }
    }
    *out = ctx;
    return RB_OK;
}

extern "C" void rb_destroy(rb_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    for (int i = 0; i < RB_S_COUNT; ++i)
        if (ctx->slots[i].ptr) cudaFree(ctx->slots[i].ptr);
    for (void* p : ctx->retired) cudaFree(p);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    for (int i = 0; i < 4; ++i)
        if (ctx->spoke_ev[i]) cudaEventDestroy(ctx->spoke_ev[i]);
    rb_db_plan_free(ctx);
    rb_comm_free(ctx);
    delete ctx;
}

extern "C" int rb_device_info(rb_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, int64_t* l2_bytes) {
    RB_REQUIRE(ctx, "ctx is NULL");
    if (sm_count) *sm_count = ctx->sm_count;
    if (cc_major) *cc_major = ctx->cc_major;
    if (cc_minor) *cc_minor = ctx->cc_minor;
    if (l2_bytes) *l2_bytes = ctx->l2_bytes;
    return RB_OK;
}

extern "C" int rb_set_option(rb_ctx* ctx, const char* name, int64_t value) {
    RB_REQUIRE(ctx && name, "NULL argument");
    if (!strcmp(name, "spoke_profile")) { ctx->opt_spoke_profile = value != 0; return RB_OK; }
    if (!strcmp(name, "dbscan_mode")) {
        RB_REQUIRE(value >= 0 && value <= 2, "dbscan_mode: 0 = auto, 1 = general algorithm, 2 = require the tight-cell algorithm");
        ctx->opt_dbscan_mode = (int)value;
        return RB_OK;
    }
    if (!strcmp(name, "spoke_mask_variant")) {
        RB_REQUIRE(value >= 0 && value <= 2, "spoke_mask_variant: 0 = auto, 1 = register-staged, 2 = TMA-staged");
        ctx->opt_spoke_mask_variant = (int)value;
        return RB_OK;
    }
    if (!strcmp(name, "spoke_ring")) {
        RB_REQUIRE(value >= 0 && value <= 3, "spoke_ring: 0 = 64 KiB x 3, 1 = 32 KiB x 4, 2 = 32 KiB x 3 (default), 3 = 48 KiB x 2");
        ctx->opt_spoke_ring = (int)value;
        return RB_OK;
    }
    if (!strcmp(name, "spoke_l2_hint")) { ctx->opt_spoke_l2_hint = value != 0; return RB_OK; }
    if (!strcmp(name, "mask_gate")) { ctx->opt_mask_gate = value != 0; return RB_OK; }
    if (!strcmp(name, "mask_priority")) { ctx->opt_mask_priority = value != 0; return RB_OK; }
    if (!strcmp(name, "carveout")) {
        RB_REQUIRE(value >= -1 && value <= 100, "carveout: -1 = the driver's choice per kernel, 0..100 = percent of the SM's shared memory");
        ctx->opt_carveout = (int)value;
        return RB_OK;
    }
    if (!strcmp(name, "fuse_group_cells")) {
        RB_REQUIRE(value >= 0, "fuse_group_cells: 0 = default (2^28), else the grid cells one group of frames may hold");
        ctx->opt_fuse_group_cells = value;
        return RB_OK;
    }
    rb_set_error("rb_set_option: unknown option '%s'", name);
    return RB_ERR_ARG;
}

extern "C" int64_t rb_get_info(rb_ctx* ctx, const char* name) {
    if (!ctx || !name) return -1;
    if (!strcmp(name, "launches")) return ctx->launches;
    if (!strcmp(name, "spoke_profile")) return ctx->opt_spoke_profile;
    if (!strcmp(name, "spoke_mask_variant")) return ctx->opt_spoke_mask_variant;
    if (!strcmp(name, "dbscan_mode")) return ctx->opt_dbscan_mode;
    if (!strcmp(name, "spoke_last_variant")) return ctx->spoke_last_variant;
    if (!strcmp(name, "land_last_variant")) return ctx->land_last_variant;
    if (!strcmp(name, "spoke_ring")) return ctx->opt_spoke_ring;
    if (!strcmp(name, "spoke_l2_hint")) return ctx->opt_spoke_l2_hint;
    if (!strcmp(name, "mask_gate")) return ctx->opt_mask_gate;
    if (!strcmp(name, "mask_priority")) return ctx->opt_mask_priority;
    if (!strcmp(name, "carveout")) return ctx->opt_carveout;
    if (!strcmp(name, "fuse_group_cells")) return ctx->opt_fuse_group_cells;
    // device time of the last profiled rb_spoke_to_points, per kernel, in nanoseconds (syncs on its last event)
    int k = !strcmp(name, "spoke_mask_ns") ? 0 : !strcmp(name, "spoke_offsets_ns") ? 1 : !strcmp(name, "spoke_emit_ns") ? 2 : -1;
    if (k >= 0) {
        if (!ctx->spoke_ev[3]) return -1;
        if (cudaEventSynchronize(ctx->spoke_ev[3]) != cudaSuccess) return -1;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->spoke_ev[k], ctx->spoke_ev[k + 1]) != cudaSuccess) return -1;
        return (int64_t)((double)ms * 1e6);
    }
    return -1;
}

extern "C" int64_t rb_launch_count(rb_ctx* ctx) { return ctx ? ctx->launches : -1; }

// Frees the scratch buffers this context has outgrown. Only for moments when NO work of the context is in flight (the
// caller has just synchronised its stream) and no collective of the process is waiting for a peer: cudaFree synchronises
// the whole device. rb_detect_block calls it after its final read-back; the time-sharded path never does.
extern "C" int rb_trim(rb_ctx* ctx) {
    RB_REQUIRE(ctx, "ctx is NULL");
    for (void* p : ctx->retired) cudaFree(p);
    ctx->retired.clear();
    return RB_OK;
}

int rb_scratch_get(rb_ctx* ctx, rb_slot slot, size_t bytes, void** out) {
    rb_scratch& s = ctx->slots[slot];
    if (bytes == 0) bytes = 16;
    if (s.cap < bytes) {
        if (s.ptr) {
            // The old buffer may still be in use by work queued on the caller's stream, and neither a device-wide
            // sync nor cudaFree (which syncs implicitly) is safe here: with several contexts per device (blocks in
            // flight, one NCCL communicator per worker) another thread's collective may be waiting for a peer that
            // is itself blocked in such a sync. Retire the buffer; it is freed with the context.
            ctx->retired.push_back(s.ptr);
            s.ptr = nullptr;
            s.cap = 0;
        }
        size_t want = bytes + bytes / 2;           // headroom: retired buffers stay allocated until rb_destroy
        want = (want + 255) & ~size_t(255);
        cudaError_t e = cudaMalloc(&s.ptr, want);
        if (e != cudaSuccess) {
            rb_set_error("scratch slot %d: cudaMalloc(%zu) -> %s", (int)slot, want, cudaGetErrorString(e));
            s.ptr = nullptr;
            return RB_ERR_NOMEM;
        }
        s.cap = want;
    }
    *out = s.ptr;
    return RB_OK;
}

// ---- exclusive scan (int32) --------------------------------------------------------------------
// Three phases: per-block sums, scan of the block sums by one block, rescan + add.
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ int warp_incl_scan(int v) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int o = __shfl_up_sync(0xffffffffu, v, d);
        if ((int)rb_lane() >= d) v += o;
    }
    return v;
}

// exclusive scan of one value per thread across the block; returns exclusive prefix, total in *total
__device__ __forceinline__ int block_excl_scan(int v, int* total) {
    __shared__ int warp_sums[SCAN_THREADS / 32];
    __shared__ int block_total;
    int incl = warp_incl_scan(v);
    int w = threadIdx.x >> 5;
    if (rb_lane() == 31) warp_sums[w] = incl;
    __syncthreads();
    if (w == 0) {
        int s = rb_lane() < SCAN_THREADS / 32 ? warp_sums[rb_lane()] : 0;
        int si = warp_incl_scan(s);
        if (rb_lane() < SCAN_THREADS / 32) warp_sums[rb_lane()] = si - s;
        if (rb_lane() == SCAN_THREADS / 32 - 1) block_total = si;
    }
    __syncthreads();
    int excl = incl - v + warp_sums[w];
    *total = block_total;
    __syncthreads();
    return excl;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_block_sums(const int32_t* in, int64_t n,
                                                               int32_t* __restrict__ sums) {
    int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    int s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k)
        if (base + k < n) s += in[base + k];
    int total;
    block_excl_scan(s, &total);
    if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

// single block: exclusive scan of sums[0..m) in place; total -> *total_out
__global__ void __launch_bounds__(SCAN_THREADS) scan_sums_serial(int32_t* __restrict__ sums, int64_t m,
                                                                int32_t* __restrict__ total_out) {
    int carry = 0;
    for (int64_t base = 0; base < m; base += SCAN_TILE) {
        int v[SCAN_ITEMS];
        int s = 0;
        int64_t i0 = base + (int64_t)threadIdx.x * SCAN_ITEMS;
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; ++k) {
            v[k] = (i0 + k < m) ? sums[i0 + k] : 0;
            s += v[k];
        }
        int total;
        int excl = block_excl_scan(s, &total) + carry;
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; ++k) {
            if (i0 + k < m) sums[i0 + k] = excl;
            excl += v[k];
        }
        carry += total;
    }
    if (threadIdx.x == 0 && total_out) *total_out = carry;
}

// in and out may be the SAME array (the bucket table is scanned in place): no __restrict__ on them - every thread reads
// its own items before it writes them
__global__ void __launch_bounds__(SCAN_THREADS) scan_apply(const int32_t* in, int32_t* out,
                                                          int64_t n, const int32_t* __restrict__ sums) {
    int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    int v[SCAN_ITEMS];
    int s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        v[k] = (base + k < n) ? in[base + k] : 0;
        s += v[k];
    }
    int total;
    int excl = block_excl_scan(s, &total) + sums[blockIdx.x];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        if (base + k < n) out[base + k] = excl;
        excl += v[k];
    }
}

int rb_exclusive_scan_i32(rb_ctx* ctx, const int32_t* in, int32_t* out, int64_t n, int32_t* total_out,
                          cudaStream_t stream) {
    if (n <= 0) {
        if (total_out) RB_CUDA(cudaMemsetAsync(total_out, 0, sizeof(int32_t), stream));
        return RB_OK;
    }
    int64_t nb = rb_div_up(n, SCAN_TILE);
    void* sums;
    RB_TRY(rb_scratch_get(ctx, RB_S_BLOCKSUM, sizeof(int32_t) * (size_t)nb, &sums));
    RB_CUDA(rb_launch(ctx, scan_block_sums, dim3((unsigned)nb), dim3(SCAN_THREADS), 0, stream, in, n, (int32_t*)sums));
    RB_LAUNCH_CHECK(ctx);
    RB_CUDA(rb_launch(ctx, scan_sums_serial, dim3(1), dim3(SCAN_THREADS), 0, stream, (int32_t*)sums, nb, total_out));
    RB_LAUNCH_CHECK(ctx);
    RB_CUDA(rb_launch(ctx, scan_apply, dim3((unsigned)nb), dim3(SCAN_THREADS), 0, stream, in, out, n, (const int32_t*)sums));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}
