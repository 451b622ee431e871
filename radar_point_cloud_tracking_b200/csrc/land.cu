// Land / stationary persistence filter (reference 4_temporal_object_tracker.py:359-436).
//
//   rb_bounds          global min/max of x, y                       (T4:365-369)
//   rb_land_accumulate per-cell POINT counts + float64 intensity sums (T4:378-389)
//   rb_land_cells      persistence / mean-intensity predicate        (T4:394-410)
//   rb_land_filter     order-preserving removal of land points        (T4:413-436)
//
// The cell of a coordinate reproduces np.digitize on the host's float64 np.arange edges exactly:
// a first guess from the (nearly uniform) edge spacing, then a fix-up against the real edges.
#include <float.h>

#include "common.cuh"

namespace {

constexpr int LD_THREADS = 256;

// ---- bounds -------------------------------------------------------------------------------------
struct Bounds4 { float xmin, xmax, ymin, ymax; };

__device__ __forceinline__ Bounds4 merge(Bounds4 a, Bounds4 b) {
    Bounds4 r;
    r.xmin = fminf(a.xmin, b.xmin); r.xmax = fmaxf(a.xmax, b.xmax);
    r.ymin = fminf(a.ymin, b.ymin); r.ymax = fmaxf(a.ymax, b.ymax);
    return r;
}

__device__ __forceinline__ Bounds4 block_reduce_bounds(Bounds4 b) {
    __shared__ Bounds4 s[LD_THREADS / 32];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        Bounds4 o;
        o.xmin = __shfl_xor_sync(0xffffffffu, b.xmin, d); o.xmax = __shfl_xor_sync(0xffffffffu, b.xmax, d);
        o.ymin = __shfl_xor_sync(0xffffffffu, b.ymin, d); o.ymax = __shfl_xor_sync(0xffffffffu, b.ymax, d);
        b = merge(b, o);
    }
    if (rb_lane() == 0) s[threadIdx.x >> 5] = b;
    __syncthreads();
    if (threadIdx.x < 32) {
        Bounds4 r = threadIdx.x < LD_THREADS / 32 ? s[threadIdx.x] : Bounds4{FLT_MAX, -FLT_MAX, FLT_MAX, -FLT_MAX};
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            Bounds4 o;
            o.xmin = __shfl_xor_sync(0xffffffffu, r.xmin, d); o.xmax = __shfl_xor_sync(0xffffffffu, r.xmax, d);
            o.ymin = __shfl_xor_sync(0xffffffffu, r.ymin, d); o.ymax = __shfl_xor_sync(0xffffffffu, r.ymax, d);
            r = merge(r, o);
        }
        b = r;
    }
    return b;   // valid in thread 0
}

__global__ void __launch_bounds__(LD_THREADS) bounds_partial(const float* __restrict__ x, const float* __restrict__ y,
                                                            int64_t n, const int64_t* __restrict__ n_dev,
                                                            Bounds4* __restrict__ partial) {
    if (n_dev) n = *n_dev < n ? *n_dev : n;
    Bounds4 b{FLT_MAX, -FLT_MAX, FLT_MAX, -FLT_MAX};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float xv = x[i], yv = y[i];
        b.xmin = fminf(b.xmin, xv); b.xmax = fmaxf(b.xmax, xv);
        b.ymin = fminf(b.ymin, yv); b.ymax = fmaxf(b.ymax, yv);
    }
    b = block_reduce_bounds(b);
    if (threadIdx.x == 0) partial[blockIdx.x] = b;
}

__global__ void __launch_bounds__(LD_THREADS) bounds_final(const Bounds4* __restrict__ partial, int m,
                                                          float* __restrict__ out4) {
    Bounds4 b{FLT_MAX, -FLT_MAX, FLT_MAX, -FLT_MAX};
    for (int i = threadIdx.x; i < m; i += blockDim.x) b = merge(b, partial[i]);
    b = block_reduce_bounds(b);
    if (threadIdx.x == 0) { out4[0] = b.xmin; out4[1] = b.xmax; out4[2] = b.ymin; out4[3] = b.ymax; }
}

// ---- cell lookup ----------------------------------------------------------------------------------
// np.clip(np.digitize(v, edges) - 1, 0, n_cells - 1) with increasing float64 edges:
// digitize = number of edges <= v (side='right').
__device__ __forceinline__ int cell_of(double v, const double* __restrict__ edges, int n_edges, int n_cells,
                                       double e0, double inv_step) {
    if (n_cells <= 0) return 0;
    double g = floor((v - e0) * inv_step);
    int k = g < 0.0 ? 0 : (g > (double)(n_edges - 1) ? n_edges - 1 : (int)g);   // candidate: edges[k] <= v
    while (k > 0 && edges[k] > v) --k;
    while (k + 1 < n_edges && edges[k + 1] <= v) ++k;
    if (k == 0 && edges[0] > v) k = -1;          // v below the first edge: digitize = 0
    int idx = k;                                  // digitize - 1
    return idx < 0 ? 0 : (idx > n_cells - 1 ? n_cells - 1 : idx);
}

struct GridArgs {
    const double* xe; const double* ye;
    int nxe, nye, nx, ny;
};

// first edge + reciprocal spacing for the initial guess (any guess is fixed up against the edges)
struct AxisGuess { double e0, inv_step; };
__device__ __forceinline__ AxisGuess axis_guess(const double* __restrict__ edges, int n_edges) {
    AxisGuess a;
    a.e0 = edges[0];
    double step = n_edges > 1 ? edges[1] - edges[0] : 1.0;
    a.inv_step = step > 0.0 ? 1.0 / step : 0.0;
    return a;
}

// ---- accumulate -------------------------------------------------------------------------------------
// np.add.at(count, (ix, iy), 1) and np.add.at(isum, (ix, iy), intensity) (T4:388-389) add one point after the other; a
// parallel float64 sum is order dependent - unless every addend is an integer. Radar echoes ARE integers (0..255,
// PIPELINE_DOCUMENTATION.txt:47), so the fast path works in integer arithmetic, which is exact in any order, and CHECKS
// that assumption on the device: an intensity that is not an integer in [0, 65535] raises a flag (*inexact); the caller
// then repeats the accumulation with rb_land_accumulate_ordered, which adds in the reference's order for any input.
//
// Privatised histogram in shared memory (int32 count + uint32 sum per cell, 8 bytes: the whole ~93 x 93 grid of a
// 231 m sweep takes 69 KB, so two CTAs fit beside the mask kernel's ring), flushed to the global grids every 65536 points
// per block (65536 x 65535 < 2^32) with one atomic pair per touched cell. A thread takes ACC_ITEMS CONSECUTIVE points -
// neighbouring range bins of one spoke, a run of which falls into one cell - and adds each run with one pair of native
// integer shared-memory atomics (round 1 used float64 shared atomics, a compare-and-swap loop each: 0.22 ms per 1024-frame
// block; pooling the runs of a warp with __match_any_sync first was measured too and is slower, 0.46 ms).
constexpr int ACC_ITEMS = 8;
constexpr int ACC_FLUSH_POINTS = 65536;
__global__ void __launch_bounds__(LD_THREADS) land_accumulate_smem(const float* __restrict__ x, const float* __restrict__ y,
                                                                  const float* __restrict__ inten, int64_t n,
                                                                  GridArgs g, int32_t* __restrict__ count,
                                                                  double* __restrict__ isum, int32_t* __restrict__ inexact) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int cells = g.nx * g.ny;
    double* s_xe = reinterpret_cast<double*>(smem);
    double* s_ye = s_xe + g.nxe;
    int* s_cnt = reinterpret_cast<int*>(s_ye + g.nye);
    unsigned* s_sum = reinterpret_cast<unsigned*>(s_cnt + cells);
    for (int i = threadIdx.x; i < cells; i += blockDim.x) { s_sum[i] = 0u; s_cnt[i] = 0; }
    for (int i = threadIdx.x; i < g.nxe; i += blockDim.x) s_xe[i] = g.xe[i];
    for (int i = threadIdx.x; i < g.nye; i += blockDim.x) s_ye[i] = g.ye[i];
    __syncthreads();
    const AxisGuess gx = axis_guess(s_xe, g.nxe), gy = axis_guess(s_ye, g.nye);
    constexpr unsigned FULL = 0xffffffffu;
    const unsigned lane = rb_lane();
    bool bad = false;
    const int64_t step = (int64_t)blockDim.x * ACC_ITEMS;                       // points per block and iteration
    const int64_t chunk = (int64_t)gridDim.x * step;
    int since_flush = 0;
    // every thread of the block runs the same number of iterations (the flush below is a block-wide barrier)
    for (int64_t base0 = (int64_t)blockIdx.x * step; base0 < n; base0 += chunk) {
        const int64_t base = base0 + (int64_t)threadIdx.x * ACC_ITEMS;
        int cur = -1, cnt = 0;
        unsigned sum = 0;
#pragma unroll
        for (int j = 0; j < ACC_ITEMS; ++j) {
            const int64_t i = base + j;
            if (i >= n) break;
            const int ix = cell_of((double)x[i], s_xe, g.nxe, g.nx, gx.e0, gx.inv_step);
            const int iy = cell_of((double)y[i], s_ye, g.nye, g.ny, gy.e0, gy.inv_step);
            const int c = ix * g.ny + iy;
            const float f = inten[i];
            const int iv = (int)f;
            bad |= !(f == (float)iv && iv >= 0 && iv <= 65535);
            if (c != cur) {                                                     // a run ends where the cell changes
                if (cnt) { atomicAdd(&s_cnt[cur], cnt); atomicAdd(&s_sum[cur], sum); }
                cur = c; cnt = 0; sum = 0;
            }
            ++cnt;
            sum += (unsigned)iv & 0xffffu;
        }
        if (cnt) { atomicAdd(&s_cnt[cur], cnt); atomicAdd(&s_sum[cur], sum); }
        since_flush += (int)step;
        if (since_flush + (int)step > ACC_FLUSH_POINTS || base0 + chunk >= n) {   // block-uniform condition
            __syncthreads();
            for (int i = threadIdx.x; i < cells; i += blockDim.x) {
                const int c = s_cnt[i];
                if (c) { atomicAdd(&count[i], c); atomicAdd(&isum[i], (double)s_sum[i]); s_cnt[i] = 0; s_sum[i] = 0u; }
            }
            __syncthreads();
            since_flush = 0;
        }
    }
    if (__any_sync(FULL, bad) && lane == 0) atomicOr(inexact, 1);
}

// grids too large for shared memory: global atomics (float64 adds of integers are exact in any order; same check)
__global__ void __launch_bounds__(LD_THREADS) land_accumulate_global(const float* __restrict__ x, const float* __restrict__ y,
                                                                    const float* __restrict__ inten, int64_t n,
                                                                    GridArgs g, int32_t* __restrict__ count,
                                                                    double* __restrict__ isum, int32_t* __restrict__ inexact) {
    const AxisGuess gx = axis_guess(g.xe, g.nxe), gy = axis_guess(g.ye, g.nye);
    bool bad = false;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int ix = cell_of((double)x[i], g.xe, g.nxe, g.nx, gx.e0, gx.inv_step);
        int iy = cell_of((double)y[i], g.ye, g.nye, g.ny, gy.e0, gy.inv_step);
        int c = ix * g.ny + iy;
        const float f = inten[i];
        bad |= !(f == rintf(f) && fabsf(f) <= 16777216.f);
        atomicAdd(&count[c], 1);
        atomicAdd(&isum[c], (double)f);
    }
    if (bad) atomicOr(inexact, 1);
}

// ---- the ordered accumulation (any intensities): cell id per point, then the points of every cell in their original
// order (the stable partition of clusters.cu), then one thread per cell adds them one after the other in float64 -
// exactly np.add.at's order
__global__ void __launch_bounds__(LD_THREADS) land_cell_id_kernel(const float* __restrict__ x, const float* __restrict__ y, int64_t n,
                                                                 GridArgs g, int32_t* __restrict__ cell) {
    const AxisGuess gx = axis_guess(g.xe, g.nxe), gy = axis_guess(g.ye, g.nye);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        cell[i] = cell_of((double)x[i], g.xe, g.nxe, g.nx, gx.e0, gx.inv_step) * g.ny + cell_of((double)y[i], g.ye, g.nye, g.ny, gy.e0, gy.inv_step);
}

__global__ void __launch_bounds__(128) land_ordered_sum_kernel(const int32_t* __restrict__ seg_label, const int32_t* __restrict__ seg_count,
                                                              const int64_t* __restrict__ seg_start, int64_t n_seg,
                                                              const float* __restrict__ grouped, int32_t* __restrict__ count,
                                                              double* __restrict__ isum) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_seg) return;
    const int c = seg_label[k];
    if (c < 0) return;
    const int m = seg_count[k];
    const float* __restrict__ v = grouped + seg_start[k];
    double acc = isum[c];
    for (int i = 0; i < m; ++i) acc = __dadd_rn(acc, (double)v[i]);
    isum[c] = acc;
    count[c] += m;
}

__global__ void land_cells_kernel(const int32_t* __restrict__ count, const double* __restrict__ isum, int64_t n_cells,
                                  double frames, double persistence, double min_intensity,
                                  uint8_t* __restrict__ land) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_cells) return;
    int c = count[i];
    double frac = __ddiv_rn((double)c, frames);                       // T4:401
    double mean = c > 0 ? __ddiv_rn(isum[i], (double)c) : 0.0;        // T4:405
    land[i] = (frac >= persistence) && (mean >= min_intensity);      // T4:408
}

// ---- filter (order-preserving compaction) -----------------------------------------------------------
constexpr int FL_ITEMS = 4;
constexpr int FL_TILE = LD_THREADS * FL_ITEMS;     // 1024 points per block, blocked arrangement per warp

// pass 1: keep flag per point + survivors per tile
__global__ void __launch_bounds__(LD_THREADS) land_keep_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                              int64_t n, GridArgs g, const uint8_t* __restrict__ land,
                                                              uint8_t* __restrict__ keep, int32_t* __restrict__ tile_count) {
    __shared__ int s_warp[LD_THREADS / 32];
    int64_t base = (int64_t)blockIdx.x * FL_TILE;
    int local = 0;
    const AxisGuess gx = axis_guess(g.xe, g.nxe), gy = axis_guess(g.ye, g.nye);
#pragma unroll
    for (int k = 0; k < FL_ITEMS; ++k) {
        int64_t i = base + k * LD_THREADS + threadIdx.x;
        bool kp = false;
        if (i < n) {
            int ix = cell_of((double)x[i], g.xe, g.nxe, g.nx, gx.e0, gx.inv_step);
            int iy = cell_of((double)y[i], g.ye, g.nye, g.ny, gy.e0, gy.inv_step);
            kp = !land[ix * g.ny + iy];
            keep[i] = kp;
        }
        local += __popc(__ballot_sync(0xffffffffu, kp));
    }
    if (rb_lane() == 0) s_warp[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
        for (int i = 0; i < LD_THREADS / 32; ++i) s += s_warp[i];
        tile_count[blockIdx.x] = s;
    }
}

// pass 2 (after the scan of tile_count): scatter survivors in order
__global__ void __launch_bounds__(LD_THREADS) land_scatter_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                                 const float* __restrict__ inten, const int32_t* __restrict__ gain,
                                                                 int64_t n, const uint8_t* __restrict__ keep,
                                                                 const int32_t* __restrict__ tile_prefix,
                                                                 float* __restrict__ xo, float* __restrict__ yo,
                                                                 float* __restrict__ io, int32_t* __restrict__ go) {
    __shared__ int s_row[FL_ITEMS][LD_THREADS / 32];
    int64_t base = (int64_t)blockIdx.x * FL_TILE;
    const unsigned lt = rb_lanemask_lt();
    const int warp = threadIdx.x >> 5;
    bool kp[FL_ITEMS];
    int below[FL_ITEMS];
#pragma unroll
    for (int k = 0; k < FL_ITEMS; ++k) {
        int64_t i = base + k * LD_THREADS + threadIdx.x;
        kp[k] = i < n && keep[i];
        unsigned b = __ballot_sync(0xffffffffu, kp[k]);
        below[k] = __popc(b & lt);
        if (rb_lane() == 0) s_row[k][warp] = __popc(b);
    }
    __syncthreads();
    int offset = tile_prefix[blockIdx.x];
#pragma unroll
    for (int k = 0; k < FL_ITEMS; ++k) {
        // element order inside the tile: row k (256 consecutive points), then warp, then lane
        int before = 0;
        for (int kk = 0; kk < k; ++kk)
            for (int wv = 0; wv < LD_THREADS / 32; ++wv) before += s_row[kk][wv];
        for (int wv = 0; wv < warp; ++wv) before += s_row[k][wv];
        if (kp[k]) {
            int64_t i = base + k * LD_THREADS + threadIdx.x;
            int64_t pos = (int64_t)offset + before + below[k];
            xo[pos] = x[i]; yo[pos] = y[i]; io[pos] = inten[i]; go[pos] = gain[i];
        }
    }
}

// new frame offsets: survivors before frame_off[f]; one warp per frame boundary
__global__ void land_frame_offsets_kernel(const int64_t* __restrict__ frame_off, int64_t n_frames, int64_t n,
                                          const uint8_t* __restrict__ keep, const int32_t* __restrict__ tile_prefix,
                                          const int32_t* __restrict__ total, int64_t* __restrict__ frame_off_out) {
    int64_t f = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (f > n_frames) return;
    int64_t off = frame_off[f];
    if (off >= n) {
        if (rb_lane() == 0) frame_off_out[f] = *total;
        return;
    }
    int64_t tile = off / FL_TILE;
    int cnt = 0;
    for (int64_t i = tile * FL_TILE + rb_lane(); i < off; i += 32) cnt += keep[i];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
    if (rb_lane() == 0) frame_off_out[f] = (int64_t)tile_prefix[tile] + cnt;
}

GridArgs make_grid_args(const double* xe, int nxe, const double* ye, int nye) {
    GridArgs g;
    g.xe = xe; g.ye = ye; g.nxe = nxe; g.nye = nye;
    g.nx = nxe - 1; g.ny = nye - 1;
    return g;
}

}  // namespace

extern "C" int rb_bounds(rb_ctx* ctx, const float* x, const float* y, int64_t n, float* out4, void* stream_) {
    RB_REQUIRE(ctx && out4, "NULL argument");
    RB_REQUIRE(n > 0 && x && y, "rb_bounds needs at least one point");
    cudaStream_t stream = (cudaStream_t)stream_;
    int blocks = (int)(rb_div_up(n, LD_THREADS * 8) < (int64_t)ctx->sm_count * 8 ? rb_div_up(n, LD_THREADS * 8)
                                                                                 : (int64_t)ctx->sm_count * 8);
    void* partial;
    RB_TRY(rb_scratch_get(ctx, RB_S_REDUCE, sizeof(Bounds4) * (size_t)blocks, &partial));
    RB_CUDA(rb_launch(ctx, bounds_partial, dim3(blocks), dim3(LD_THREADS), 0, stream, x, y, n, nullptr, (Bounds4*)partial));
    RB_LAUNCH_CHECK(ctx);
    RB_CUDA(rb_launch(ctx, bounds_final, dim3(1), dim3(LD_THREADS), 0, stream, (const Bounds4*)partial, blocks, out4));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}

int rb_bounds_devn(rb_ctx* ctx, const float* x, const float* y, const int64_t* n_dev, int64_t n_max, float* out4, cudaStream_t stream) {
    if (n_max <= 0) return RB_OK;
    int blocks = (int)(rb_div_up(n_max, LD_THREADS * 8) < (int64_t)ctx->sm_count * 4 ? rb_div_up(n_max, LD_THREADS * 8)
                                                                                     : (int64_t)ctx->sm_count * 4);
    void* partial;
    RB_TRY(rb_scratch_get(ctx, RB_S_REDUCE, sizeof(Bounds4) * (size_t)blocks, &partial));
    RB_CUDA(rb_launch(ctx, bounds_partial, dim3(blocks), dim3(LD_THREADS), 0, stream, x, y, n_max, n_dev, (Bounds4*)partial));
    RB_LAUNCH_CHECK(ctx);
    RB_CUDA(rb_launch(ctx, bounds_final, dim3(1), dim3(LD_THREADS), 0, stream, (const Bounds4*)partial, blocks, out4));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}

extern "C" int rb_bounds_counted(rb_ctx* ctx, const float* x, const float* y, const int64_t* n_dev, int64_t n_max, float* out4,
                                 void* stream) {
    RB_REQUIRE(ctx && n_dev && out4 && n_max >= 0 && (n_max == 0 || (x && y)), "bad arguments");
    return rb_bounds_devn(ctx, x, y, n_dev, n_max, out4, (cudaStream_t)stream);
}

int rb_land_inexact_flag(rb_ctx* ctx, int32_t** flag, cudaStream_t stream) {
    rb_scratch& slot = ctx->slots[RB_S_LAND_FLAG];
    const void* before = slot.ptr;
    void* p;
    RB_TRY(rb_scratch_get(ctx, RB_S_LAND_FLAG, 64, &p));
    if (slot.ptr != before) RB_CUDA(cudaMemsetAsync(p, 0, 64, stream));
    *flag = (int32_t*)p;
    return RB_OK;
}

extern "C" int rb_land_accumulate(rb_ctx* ctx, const float* x, const float* y, const float* inten, int64_t n,
                                  const double* x_edges, int n_x_edges, const double* y_edges, int n_y_edges,
                                  int32_t* count, double* isum, void* stream_) {
    RB_REQUIRE(ctx && x_edges && y_edges && count && isum, "NULL argument");
    RB_REQUIRE(n_x_edges >= 2 && n_y_edges >= 2, "need at least two edges per axis");
    if (n <= 0) return RB_OK;
    RB_REQUIRE(x && y && inten, "NULL points");
    cudaStream_t stream = (cudaStream_t)stream_;
    GridArgs g = make_grid_args(x_edges, n_x_edges, y_edges, n_y_edges);
    int32_t* inexact;
    RB_TRY(rb_land_inexact_flag(ctx, &inexact, stream));
    int64_t cells = (int64_t)g.nx * g.ny;
    size_t smem = (size_t)cells * 8 + (size_t)(n_x_edges + n_y_edges) * 8;
    const int per_sm = smem <= 72 * 1024 ? 3 : (smem <= 110 * 1024 ? 2 : 1);
    int blocks = (int)(rb_div_up(n, LD_THREADS * ACC_ITEMS) < (int64_t)ctx->sm_count * per_sm ? rb_div_up(n, LD_THREADS * ACC_ITEMS)
                                                                                              : (int64_t)ctx->sm_count * per_sm);
    if (smem <= 220 * 1024) {
        if (!ctx->attr_land) {                          // once per context (= per device): allow the largest grid that fits
            RB_CUDA(cudaFuncSetAttribute(land_accumulate_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
            ctx->attr_land = true;
        }
        RB_CUDA(rb_launch(ctx, land_accumulate_smem, dim3(blocks), dim3(LD_THREADS), smem, stream, x, y, inten, n, g, count, isum, inexact));
        ctx->land_last_variant = 1;
    } else {
        blocks = (int)(rb_div_up(n, LD_THREADS) < (int64_t)ctx->sm_count * 8 ? rb_div_up(n, LD_THREADS)
                                                                           : (int64_t)ctx->sm_count * 8);
        RB_CUDA(rb_launch(ctx, land_accumulate_global, dim3(blocks), dim3(LD_THREADS), 0, stream, x, y, inten, n, g, count, isum, inexact));
        ctx->land_last_variant = 2;
    }
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}

extern "C" int rb_land_accumulate_status(rb_ctx* ctx, int32_t* inexact_out, void* stream_) {
    RB_REQUIRE(ctx && inexact_out, "NULL argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    int32_t* flag;
    RB_TRY(rb_land_inexact_flag(ctx, &flag, stream));
    int32_t* h = (int32_t*)ctx->pinned;
    RB_CUDA(cudaMemcpyAsync(h, flag, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    RB_CUDA(cudaMemsetAsync(flag, 0, sizeof(int32_t), stream));
    RB_CUDA(cudaStreamSynchronize(stream));
    *inexact_out = h[0];
    return RB_OK;
}

extern "C" int rb_land_accumulate_status_async(rb_ctx* ctx, int32_t* dst, void* stream_) {
    RB_REQUIRE(ctx && dst, "NULL argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    int32_t* flag;
    RB_TRY(rb_land_inexact_flag(ctx, &flag, stream));
    RB_CUDA(cudaMemcpyAsync(dst, flag, sizeof(int32_t), cudaMemcpyDefault, stream));
    RB_CUDA(cudaMemsetAsync(flag, 0, sizeof(int32_t), stream));
    return RB_OK;
}

int rb_stable_group(rb_ctx* ctx, const float* values, const int32_t* labels, int64_t n, int64_t n_labels, int32_t* seg_label,
                    int32_t* seg_count, int64_t* seg_start, int64_t cap_segments, float* grouped, int64_t* n_segments, cudaStream_t stream);

extern "C" int rb_land_accumulate_ordered(rb_ctx* ctx, const float* x, const float* y, const float* inten, int64_t n,
                                          const double* x_edges, int n_x_edges, const double* y_edges, int n_y_edges,
                                          int32_t* count, double* isum, void* stream_) {
    RB_REQUIRE(ctx && x_edges && y_edges && count && isum, "NULL argument");
    RB_REQUIRE(n_x_edges >= 2 && n_y_edges >= 2, "need at least two edges per axis");
    RB_REQUIRE(n < ((int64_t)1 << 31), "too many points");
    if (n <= 0) return RB_OK;
    RB_REQUIRE(x && y && inten, "NULL points");
    cudaStream_t stream = (cudaStream_t)stream_;
    GridArgs g = make_grid_args(x_edges, n_x_edges, y_edges, n_y_edges);
    const int64_t cells = (int64_t)g.nx * g.ny;
    // scratch: cell id per point, grouped intensities, segment table (one segment per occupied cell)
    void* raw;
    const size_t seg_cap = (size_t)cells + 1;
    RB_TRY(rb_scratch_get(ctx, RB_S_LAND_ORDERED, sizeof(int32_t) * (size_t)n + sizeof(float) * (size_t)n + seg_cap * 16 + 64, &raw));
    int64_t* seg_start = (int64_t*)raw;
    int32_t* seg_label = (int32_t*)(seg_start + seg_cap);
    int32_t* seg_count = seg_label + seg_cap;
    int32_t* cell = seg_count + seg_cap;
    float* grouped = (float*)(cell + n);
    const int blocks = (int)(rb_div_up(n, LD_THREADS) < (int64_t)ctx->sm_count * 8 ? rb_div_up(n, LD_THREADS) : (int64_t)ctx->sm_count * 8);
    RB_CUDA(rb_launch(ctx, land_cell_id_kernel, dim3(blocks), dim3(LD_THREADS), 0, stream, x, y, n, g, cell));
    RB_LAUNCH_CHECK(ctx);
    ctx->land_last_variant = 3;
    int64_t n_seg = 0;
    RB_TRY(rb_stable_group(ctx, inten, cell, n, cells, seg_label, seg_count, seg_start, (int64_t)seg_cap, grouped, &n_seg, stream));
    if (n_seg > 0) {
        RB_CUDA(rb_launch(ctx, land_ordered_sum_kernel, dim3((unsigned)rb_div_up(n_seg, 128)), dim3(128), 0, stream, (const int32_t*)seg_label,
                          (const int32_t*)seg_count, (const int64_t*)seg_start, n_seg, (const float*)grouped, count, isum));
        RB_LAUNCH_CHECK(ctx);
    }
    return RB_OK;
}

extern "C" int rb_land_cells(rb_ctx* ctx, const int32_t* count, const double* isum, int64_t n_cells,
                             int64_t num_frames, double persistence, double min_intensity, uint8_t* land,
                             void* stream_) {
    RB_REQUIRE(ctx && count && isum && land, "NULL argument");
    if (n_cells <= 0) return RB_OK;
    cudaStream_t stream = (cudaStream_t)stream_;
    double frames = (double)(num_frames > 1 ? num_frames : 1);       // max(num_frames, 1), T4:401
    RB_CUDA(rb_launch(ctx, land_cells_kernel, dim3((unsigned)rb_div_up(n_cells, 256)), dim3(256), 0, stream, count, isum, n_cells, frames,
                                                                            persistence, min_intensity, land));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}

extern "C" int rb_land_filter(rb_ctx* ctx, const float* x, const float* y, const float* inten, const int32_t* gain,
                              int64_t n, const int64_t* frame_off, int64_t n_frames, const double* x_edges,
                              int n_x_edges, const double* y_edges, int n_y_edges, const uint8_t* land,
                              float* x_out, float* y_out, float* inten_out, int32_t* gain_out,
                              int64_t* frame_off_out, uint8_t* keep_mask, void* stream_) {
    RB_REQUIRE(ctx && x_edges && y_edges && land && frame_off && frame_off_out, "NULL argument");
    RB_REQUIRE(n_x_edges >= 2 && n_y_edges >= 2, "need at least two edges per axis");
    RB_REQUIRE(n >= 0 && n < ((int64_t)1 << 31) && n_frames >= 0, "bad sizes");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n == 0) {
        RB_CUDA(cudaMemsetAsync(frame_off_out, 0, sizeof(int64_t) * (size_t)(n_frames + 1), stream));
        return RB_OK;
    }
    RB_REQUIRE(x && y && inten && gain && x_out && y_out && inten_out && gain_out, "NULL points");
    GridArgs g = make_grid_args(x_edges, n_x_edges, y_edges, n_y_edges);
    int64_t tiles = rb_div_up(n, FL_TILE);
    void* keep = keep_mask;
    if (!keep) RB_TRY(rb_scratch_get(ctx, RB_S_KEEP, (size_t)n, &keep));
    void* tile_count;
    RB_TRY(rb_scratch_get(ctx, RB_S_BLOCKSUM2, sizeof(int32_t) * (size_t)(tiles + 1), &tile_count));
    int32_t* tc = (int32_t*)tile_count;
    RB_CUDA(rb_launch(ctx, land_keep_kernel, dim3((unsigned)tiles), dim3(LD_THREADS), 0, stream, x, y, n, g, land, (uint8_t*)keep, tc));
    RB_LAUNCH_CHECK(ctx);
    RB_TRY(rb_exclusive_scan_i32(ctx, tc, tc, tiles, tc + tiles, stream));
    RB_CUDA(rb_launch(ctx, land_scatter_kernel, dim3((unsigned)tiles), dim3(LD_THREADS), 0, stream, x, y, inten, gain, n, (const uint8_t*)keep, tc,
                                                                   x_out, y_out, inten_out, gain_out));
    RB_LAUNCH_CHECK(ctx);
    unsigned warps = (unsigned)(n_frames + 1);
    RB_CUDA(rb_launch(ctx, land_frame_offsets_kernel, dim3((unsigned)rb_div_up((int64_t)warps * 32, 256)), dim3(256), 0, stream, frame_off, n_frames, n, (const uint8_t*)keep, tc, tc + tiles, frame_off_out));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}
