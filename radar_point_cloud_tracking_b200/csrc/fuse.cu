// Max fusion of gains on a grid (reference 5_gain_fusion_ply_builder.py:222-273, fuse_gains_max), for one frame
// (rb_fuse_max) or for many frames per call (rb_fuse_max_frames). One pooling rule serves both:
//   cell = trunc((v - v_min) / res) in float32 (T5:258-259), max intensity per cell starting from 0 (T5:262-263),
//   cells whose maximum is > 0 emitted in y-major order (T5:267).
// Every frame gets a dense int32 grid, y-major (iy * nx + ix), at a scanned offset of one scratch array. The frames of a
// group (consecutive frames whose grids fit the scratch bound together) are pooled with atomicMax on the float bits -
// every stored value is >= 0, so integer order is float order - and the grid is then read twice in tiles of FT cells:
// once to count the occupied cells of each tile, once, after a scan of the tile counts, to emit them in order. The
// output offset of a group is the last frame offset the previous group wrote, which stays on the device.
#include <math.h>

#include "common.cuh"

namespace {

constexpr int FT_THREADS = 256;
constexpr int FT_ITEMS = 8;
constexpr int FT = FT_THREADS * FT_ITEMS;    // cells per tile; every group's grid is padded to a multiple of it
constexpr int PT = 32 * 8;                   // points per warp tile of the bounds and pooling kernels
constexpr int64_t CELL_LIMIT = (int64_t)1 << 30;
constexpr int64_t DEFAULT_GROUP_CELLS = (int64_t)1 << 28;   // 1 GiB of int32 grid

struct FuseFrame {
    float x_min, y_min;
    int32_t nx, ny;
};

// total order of floats as unsigned keys (for atomicMin / atomicMax)
__device__ __forceinline__ unsigned fkey(float v) {
    unsigned b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float fkey_inv(unsigned k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

// largest f in [lo, hi) with off[f] <= i (off ascending, off[lo] <= i): the frame of point (or cell) i, empty frames skipped
__device__ __forceinline__ int64_t seg_of(const int64_t* __restrict__ off, int64_t lo, int64_t hi, int64_t i) {
    while (hi - lo > 1) {
        int64_t mid = (lo + hi) >> 1;
        if (off[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// Per-frame float32 min / max of x and y. A warp tile inside one frame is reduced in registers (4 atomics per tile);
// a tile across frame boundaries updates per point.
__global__ void fuse_bounds_kernel(const float* __restrict__ x, const float* __restrict__ y, int64_t n,
                                   const int64_t* __restrict__ off, int64_t F, unsigned* __restrict__ bmin,
                                   unsigned* __restrict__ bmax) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t t = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; t * PT < n; t += warps) {
        const int64_t a = t * PT, b = a + PT < n ? a + PT : n;
        int64_t f = seg_of(off, 0, F, a);
        if (off[f + 1] >= b) {
            float x0 = INFINITY, x1 = -INFINITY, y0 = INFINITY, y1 = -INFINITY;
            for (int64_t i = a + lane; i < b; i += 32) {
                float xv = x[i], yv = y[i];
                x0 = fminf(x0, xv); x1 = fmaxf(x1, xv); y0 = fminf(y0, yv); y1 = fmaxf(y1, yv);
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                x0 = fminf(x0, __shfl_xor_sync(0xffffffffu, x0, d));
                x1 = fmaxf(x1, __shfl_xor_sync(0xffffffffu, x1, d));
                y0 = fminf(y0, __shfl_xor_sync(0xffffffffu, y0, d));
                y1 = fmaxf(y1, __shfl_xor_sync(0xffffffffu, y1, d));
            }
            if (lane == 0) {
                atomicMin(bmin + 2 * f, fkey(x0)); atomicMin(bmin + 2 * f + 1, fkey(y0));
                atomicMax(bmax + 2 * f, fkey(x1)); atomicMax(bmax + 2 * f + 1, fkey(y1));
            }
        } else {
            for (int64_t i = a + lane; i < b; i += 32) {
                while (f + 1 < F && off[f + 1] <= i) ++f;
                float xv = x[i], yv = y[i];
                atomicMin(bmin + 2 * f, fkey(xv)); atomicMin(bmin + 2 * f + 1, fkey(yv));
                atomicMax(bmax + 2 * f, fkey(xv)); atomicMax(bmax + 2 * f + 1, fkey(yv));
            }
        }
    }
}

// Per frame: nx = int(ceil((x_max - x_min) / res)) + 1 in float32 (T5:251-256), likewise ny; cells = nx * ny, or
// INT64_MAX when that is not finite. A frame without points gets no grid.
__global__ void fuse_plan_kernel(const int64_t* __restrict__ off, int64_t F, const unsigned* __restrict__ bmin,
                                 const unsigned* __restrict__ bmax, float res, FuseFrame* __restrict__ fr,
                                 int64_t* __restrict__ cells) {
    int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    FuseFrame o = {0.f, 0.f, 0, 0};
    int64_t c = 0;
    if (off[f + 1] > off[f]) {
        float x0 = fkey_inv(bmin[2 * f]), y0 = fkey_inv(bmin[2 * f + 1]);
        float x1 = fkey_inv(bmax[2 * f]), y1 = fkey_inv(bmax[2 * f + 1]);
        double nx = (double)ceilf(__fdiv_rn(__fsub_rn(x1, x0), res)) + 1.0;
        double ny = (double)ceilf(__fdiv_rn(__fsub_rn(y1, y0), res)) + 1.0;
        double nc = nx * ny;
        o.x_min = x0; o.y_min = y0;
        if (nc < (double)CELL_LIMIT) {                      // false for NaN and inf too
            o.nx = (int32_t)nx; o.ny = (int32_t)ny;
            c = (int64_t)o.nx * o.ny;
        } else {
            c = nc < 9.0e18 ? (int64_t)nc : INT64_MAX;
        }
    }
    fr[f] = o;
    cells[f] = c;
}

// atomicMax of the intensity bits of every point with intensity > 0 into its frame's grid (goff = grid offsets, global)
__global__ void fuse_pool_kernel(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ inten,
                                 const int64_t* __restrict__ off, const FuseFrame* __restrict__ fr,
                                 const int64_t* __restrict__ goff, int64_t fa, int64_t fb, float res, int* __restrict__ grid) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t p0 = off[fa], p1 = off[fb], g0 = goff[fa];
    for (int64_t t = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; p0 + t * PT < p1; t += warps) {
        const int64_t a = p0 + t * PT, b = a + PT < p1 ? a + PT : p1;
        int64_t f = seg_of(off, fa, fb, a);
        for (int64_t i = a + lane; i < b; i += 32) {
            while (f + 1 < fb && off[f + 1] <= i) ++f;
            const FuseFrame F_ = fr[f];
            int ix = (int)__fdiv_rn(__fsub_rn(x[i], F_.x_min), res);
            int iy = (int)__fdiv_rn(__fsub_rn(y[i], F_.y_min), res);
            float v = inten[i];
            if (ix < 0 || ix >= F_.nx || iy < 0 || iy >= F_.ny) continue;    // only for rb_fuse_max's caller-given grid
            if (v > 0.f) atomicMax(grid + (goff[f] - g0) + (int64_t)iy * F_.nx + ix, __float_as_int(v));
        }
    }
}

__device__ __forceinline__ void load_tile(const int* __restrict__ grid, int64_t tile, int v[FT_ITEMS]) {
    const int4* p = reinterpret_cast<const int4*>(grid + tile * FT + (int64_t)threadIdx.x * FT_ITEMS);
    int4 a = p[0], b = p[1];
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// exclusive prefix of one value per thread over the block, and the block's total
__device__ __forceinline__ int block_prefix(int c, int* total) {
    __shared__ int ws[FT_THREADS / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) ws[w] = incl;
    __syncthreads();
    int before = 0, all = 0;
#pragma unroll
    for (int k = 0; k < FT_THREADS / 32; ++k) {
        before += k < w ? ws[k] : 0;
        all += ws[k];
    }
    *total = all;
    return before + incl - c;
}

__global__ void __launch_bounds__(FT_THREADS) fuse_count_kernel(const int* __restrict__ grid, int32_t* __restrict__ tile_cnt) {
    int v[FT_ITEMS];
    load_tile(grid, blockIdx.x, v);
    int c = 0;
#pragma unroll
    for (int k = 0; k < FT_ITEMS; ++k) c += v[k] != 0;
    int total;
    block_prefix(c, &total);
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = total;
}

// Occupied cells of a group in order, at base + tile_base[tile] + their rank in the tile. CENTRES: float64 centres
// x_min + ix * res + res / 2, left to right (T5:269-270); otherwise the cell indices (rb_fuse_max).
template <bool CENTRES>
__global__ void __launch_bounds__(FT_THREADS) fuse_emit_kernel(const int* __restrict__ grid, const int32_t* __restrict__ tile_base,
                                                               const FuseFrame* __restrict__ fr, const int64_t* __restrict__ goff,
                                                               int64_t fa, int64_t fb, const int64_t* __restrict__ base_at,
                                                               double res, int64_t cap, double* __restrict__ cx,
                                                               double* __restrict__ cy, int32_t* __restrict__ cix,
                                                               int32_t* __restrict__ ciy, float* __restrict__ cmax) {
    int v[FT_ITEMS];
    load_tile(grid, blockIdx.x, v);
    int c = 0;
#pragma unroll
    for (int k = 0; k < FT_ITEMS; ++k) c += v[k] != 0;
    int total;
    int64_t o = *base_at + tile_base[blockIdx.x] + block_prefix(c, &total);
    if (!c) return;
    const int64_t g0 = goff[fa];
    const int64_t k0 = (int64_t)blockIdx.x * FT + (int64_t)threadIdx.x * FT_ITEMS;
    int64_t f = seg_of(goff, fa, fb, g0 + k0);
#pragma unroll
    for (int k = 0; k < FT_ITEMS; ++k) {
        if (!v[k]) continue;
        const int64_t cell = g0 + k0 + k;
        while (f + 1 < fb && goff[f + 1] <= cell) ++f;
        const FuseFrame F_ = fr[f];
        const int64_t local = cell - goff[f];
        const int iy = (int)(local / F_.nx), ix = (int)(local - (int64_t)iy * F_.nx);
        if (o < cap) {
            if (CENTRES) {
                cx[o] = __dadd_rn(__dadd_rn((double)F_.x_min, __dmul_rn((double)ix, res)), res * 0.5);
                cy[o] = __dadd_rn(__dadd_rn((double)F_.y_min, __dmul_rn((double)iy, res)), res * 0.5);
            } else {
                cix[o] = ix;
                ciy[o] = iy;
            }
            cmax[o] = __int_as_float(v[k]);
        }
        ++o;
    }
}

// cell_off[f] for f in (fa, fb]: occupied cells of the group before frame f's grid, plus the group's base. One warp per frame.
__global__ void fuse_frame_offsets_kernel(const int* __restrict__ grid, const int32_t* __restrict__ tile_base,
                                          const int64_t* __restrict__ goff, int64_t fa, int64_t fb, int64_t* __restrict__ cell_off) {
    int64_t f = fa + 1 + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (f > fb) return;
    const int lane = threadIdx.x & 31;
    const int64_t r = goff[f] - goff[fa];
    const int64_t tile = r / FT;
    int cnt = 0;
    for (int64_t i = tile * FT + lane; i < r; i += 32) cnt += grid[i] != 0;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
    if (lane == 0) cell_off[f] = cell_off[fa] + tile_base[tile] + cnt;
}

int grow_pinned(rb_ctx* ctx, size_t need, cudaStream_t stream) {
    if (ctx->pinned_cap >= need) return RB_OK;
    RB_CUDA(cudaStreamSynchronize(stream));
    if (ctx->pinned) RB_CUDA(cudaFreeHost(ctx->pinned));
    ctx->pinned = nullptr; ctx->pinned_cap = 0;
    RB_CUDA(cudaMallocHost(&ctx->pinned, need + 4096));
    ctx->pinned_cap = need + 4096;
    return RB_OK;
}

inline int64_t pad_tiles(int64_t cells) { return rb_div_up(cells, FT) * FT; }

// Pools and emits frames [0, F) group by group (cuts[0..K]); frame offsets, frame table and grid offsets are on the
// device, goff_h / off_h their host copies. cell_off[0] must already hold the first output offset.
template <bool CENTRES>
int fuse_groups(rb_ctx* ctx, const float* x, const float* y, const float* inten, const int64_t* off, const int64_t* off_h,
                const FuseFrame* fr, const int64_t* goff, const int64_t* goff_h, const int64_t* cuts, int64_t K, float res32,
                double res, int64_t cap, double* cx, double* cy, int32_t* cix, int32_t* ciy, float* cmax, int64_t* cell_off,
                cudaStream_t stream) {
    int64_t max_cells = 0;
    for (int64_t k = 0; k < K; ++k) {
        int64_t c = pad_tiles(goff_h[cuts[k + 1]] - goff_h[cuts[k]]);
        if (c > max_cells) max_cells = c;
    }
    void *gbuf, *tbuf;
    RB_TRY(rb_scratch_get(ctx, RB_S_FUSE_GRID, sizeof(int) * (size_t)max_cells, &gbuf));
    RB_TRY(rb_scratch_get(ctx, RB_S_FUSE_TILES, sizeof(int32_t) * (size_t)(max_cells / FT + 1), &tbuf));
    int* grid = (int*)gbuf;
    int32_t* tiles = (int32_t*)tbuf;
    for (int64_t k = 0; k < K; ++k) {
        const int64_t fa = cuts[k], fb = cuts[k + 1];
        const int64_t cells = pad_tiles(goff_h[fb] - goff_h[fa]), nt = cells / FT;
        const int64_t pts = off_h[fb] - off_h[fa];
        if (cells > 0) {
            RB_CUDA(cudaMemsetAsync(grid, 0, sizeof(int) * (size_t)cells, stream));
            if (pts > 0) {
                int64_t want = rb_div_up(pts, PT * (FT_THREADS / 32));
                int blocks = (int)(want < (int64_t)ctx->sm_count * 16 ? want : (int64_t)ctx->sm_count * 16);
                RB_CUDA(rb_launch(ctx, fuse_pool_kernel, dim3(blocks), dim3(FT_THREADS), 0, stream, x, y, inten, off, fr, goff, fa, fb,
                                  res32, grid));
                RB_LAUNCH_CHECK(ctx);
            }
            RB_CUDA(rb_launch(ctx, fuse_count_kernel, dim3((unsigned)nt), dim3(FT_THREADS), 0, stream, (const int*)grid, tiles));
            RB_LAUNCH_CHECK(ctx);
        }
        RB_TRY(rb_exclusive_scan_i32(ctx, tiles, tiles, nt, tiles + nt, stream));      // tiles[nt] = the group's cells
        if (cells > 0) {
            RB_CUDA(rb_launch(ctx, fuse_emit_kernel<CENTRES>, dim3((unsigned)nt), dim3(FT_THREADS), 0, stream, (const int*)grid,
                              (const int32_t*)tiles, fr, goff, fa, fb, (const int64_t*)(cell_off + fa), res, cap, cx, cy, cix, ciy,
                              cmax));
            RB_LAUNCH_CHECK(ctx);
        }
        unsigned ob = (unsigned)rb_div_up((fb - fa) * 32, 256);
        RB_CUDA(rb_launch(ctx, fuse_frame_offsets_kernel, dim3(ob), dim3(256), 0, stream, (const int*)grid, (const int32_t*)tiles, goff,
                          fa, fb, cell_off));
        RB_LAUNCH_CHECK(ctx);
    }
    return RB_OK;
}

}  // namespace

extern "C" int64_t rb_fuse_plan_groups(const int64_t* cells, int64_t n_frames, int64_t max_cells, int64_t* cuts, int64_t cap) {
    if (n_frames < 0 || max_cells < 1 || (n_frames > 0 && !cells)) {
        rb_set_error("rb_fuse_plan_groups: bad arguments");
        return RB_ERR_ARG;
    }
    int64_t k = 0, sum = 0;
    if (cuts && cap > 0) cuts[0] = 0;
    for (int64_t f = 0; f < n_frames; ++f) {
        if (cells[f] < 0) {
            rb_set_error("rb_fuse_plan_groups: negative cell count");
            return RB_ERR_ARG;
        }
        if (cells[f] > 0 && sum > 0 && sum + cells[f] > max_cells) {    // frame f starts a new group
            ++k;
            if (cuts && k < cap) cuts[k] = f;
            sum = 0;
        }
        sum += cells[f];
    }
    if (n_frames > 0) {
        ++k;
        if (cuts && k < cap) cuts[k] = n_frames;
    }
    return k;
}

extern "C" int rb_fuse_max_frames(rb_ctx* ctx, const float* x, const float* y, const float* inten, int64_t n,
                                  const int64_t* frame_off, int64_t n_frames, double resolution, double* cell_x, double* cell_y,
                                  float* cell_max, int64_t cap_cells, int64_t* cell_off, int64_t* n_cells_out, void* stream_) {
    RB_REQUIRE(ctx && n_cells_out && frame_off && cell_off, "NULL argument");
    RB_REQUIRE(n_frames >= 0 && n_frames < ((int64_t)1 << 31) && n >= 0 && cap_cells >= 0, "bad sizes");
    RB_REQUIRE(isfinite(resolution) && resolution > 0, "resolution must be finite and > 0");
    RB_REQUIRE(n == 0 || (x && y && inten), "NULL point array");
    RB_REQUIRE(cap_cells == 0 || (cell_x && cell_y && cell_max), "NULL output array");
    cudaStream_t stream = (cudaStream_t)stream_;
    const int64_t F = n_frames;
    *n_cells_out = 0;
    RB_CUDA(cudaMemsetAsync(cell_off, 0, sizeof(int64_t), stream));
    if (F == 0) {
        if (n != 0) { rb_set_error("rb_fuse_max_frames: %lld points in no frame", (long long)n); return RB_ERR_ARG; }
        return RB_OK;
    }
    const float res32 = (float)resolution;          // numpy >= 2 takes the Python float as float32 (T5:255, T5:258)
    // frames slot: bmin[2F] | bmax[2F] (u32) | FuseFrame[F] | cells[F] | goff[F+1] (int64)
    const size_t b_bytes = sizeof(unsigned) * 2 * (size_t)F;
    const size_t fr_at = 2 * b_bytes, cells_at = (fr_at + sizeof(FuseFrame) * (size_t)F + 7) & ~size_t(7);
    const size_t goff_at = cells_at + sizeof(int64_t) * (size_t)F;
    void* buf;
    RB_TRY(rb_scratch_get(ctx, RB_S_FUSE_FRAMES, goff_at + sizeof(int64_t) * (size_t)(F + 1), &buf));
    unsigned char* base = (unsigned char*)buf;
    unsigned* bmin = (unsigned*)base;
    unsigned* bmax = (unsigned*)(base + b_bytes);
    FuseFrame* fr = (FuseFrame*)(base + fr_at);
    int64_t* cells_d = (int64_t*)(base + cells_at);
    int64_t* goff = (int64_t*)(base + goff_at);
    // pinned: frame offsets [F+1] | cells [F] (read back) | grid offsets [F+1] (uploaded)
    RB_TRY(grow_pinned(ctx, sizeof(int64_t) * (size_t)(3 * F + 2), stream));
    int64_t* h_off = (int64_t*)ctx->pinned;
    int64_t* h_cells = h_off + F + 1;
    int64_t* h_goff = h_cells + F;

    RB_CUDA(cudaMemsetAsync(bmin, 0xff, b_bytes, stream));
    RB_CUDA(cudaMemsetAsync(bmax, 0, b_bytes, stream));
    if (n > 0) {
        int64_t want = rb_div_up(n, PT * 8);
        int blocks = (int)(want < (int64_t)ctx->sm_count * 16 ? want : (int64_t)ctx->sm_count * 16);
        RB_CUDA(rb_launch(ctx, fuse_bounds_kernel, dim3(blocks), dim3(256), 0, stream, x, y, n, frame_off, F, bmin, bmax));
        RB_LAUNCH_CHECK(ctx);
    }
    RB_CUDA(rb_launch(ctx, fuse_plan_kernel, dim3((unsigned)rb_div_up(F, 256)), dim3(256), 0, stream, frame_off, F,
                      (const unsigned*)bmin, (const unsigned*)bmax, res32, fr, cells_d));
    RB_LAUNCH_CHECK(ctx);
    RB_CUDA(cudaMemcpyAsync(h_off, frame_off, sizeof(int64_t) * (size_t)(F + 1), cudaMemcpyDeviceToHost, stream));
    RB_CUDA(cudaMemcpyAsync(h_cells, cells_d, sizeof(int64_t) * (size_t)F, cudaMemcpyDeviceToHost, stream));
    RB_CUDA(cudaStreamSynchronize(stream));                                          // sync 1: offsets and grid sizes

    if (h_off[0] != 0 || h_off[F] != n) {
        rb_set_error("rb_fuse_max_frames: frame_off must run from 0 to n = %lld (got %lld .. %lld)", (long long)n,
                     (long long)h_off[0], (long long)h_off[F]);
        return RB_ERR_ARG;
    }
    h_goff[0] = 0;
    for (int64_t f = 0; f < F; ++f) {
        if (h_off[f + 1] < h_off[f]) {
            rb_set_error("rb_fuse_max_frames: frame_off decreases at frame %lld", (long long)f);
            return RB_ERR_ARG;
        }
        if (h_cells[f] >= CELL_LIMIT) {
            rb_set_error("rb_fuse_max_frames: frame %lld needs a grid of %lld cells at resolution %g; the limit is 2^30 cells "
                         "per frame", (long long)f, (long long)h_cells[f], resolution);
            return RB_ERR_ARG;
        }
        h_goff[f + 1] = h_goff[f] + h_cells[f];
    }
    const int64_t bound = ctx->opt_fuse_group_cells > 0 ? ctx->opt_fuse_group_cells : DEFAULT_GROUP_CELLS;
    int64_t K = rb_fuse_plan_groups(h_cells, F, bound, nullptr, 0);
    if (K < 0) return (int)K;
    std::vector<int64_t> cuts((size_t)K + 1);
    rb_fuse_plan_groups(h_cells, F, bound, cuts.data(), K + 1);
    RB_CUDA(cudaMemcpyAsync(goff, h_goff, sizeof(int64_t) * (size_t)(F + 1), cudaMemcpyHostToDevice, stream));
    RB_TRY(fuse_groups<true>(ctx, x, y, inten, frame_off, h_off, fr, goff, h_goff, cuts.data(), K, res32, resolution, cap_cells,
                             cell_x, cell_y, nullptr, nullptr, cell_max, cell_off, stream));
    RB_CUDA(cudaMemcpyAsync(h_cells, cell_off + F, sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
    RB_CUDA(cudaStreamSynchronize(stream));                                          // sync 2: the total
    *n_cells_out = h_cells[0];
    if (h_cells[0] > cap_cells) {
        rb_set_error("rb_fuse_max_frames: %lld cells exceed capacity %lld", (long long)h_cells[0], (long long)cap_cells);
        return RB_ERR_CAPACITY;
    }
    return RB_OK;
}

extern "C" int rb_fuse_max(rb_ctx* ctx, const float* x, const float* y, const float* inten, int64_t n, float x_min,
                           float y_min, float resolution, int nx, int ny, int32_t* cell_ix, int32_t* cell_iy,
                           float* cell_max, int64_t cap_cells, int64_t* n_cells_out, void* stream_) {
    RB_REQUIRE(ctx && n_cells_out, "NULL argument");
    RB_REQUIRE(nx > 0 && ny > 0 && (int64_t)nx * ny < CELL_LIMIT, "bad grid size");
    RB_REQUIRE(resolution > 0, "resolution must be positive");
    cudaStream_t stream = (cudaStream_t)stream_;
    *n_cells_out = 0;
    if (n <= 0) return RB_OK;
    RB_REQUIRE(x && y && inten && cell_ix && cell_iy && cell_max, "NULL argument");
    // one frame with the caller's grid: frame offsets {0, n}, grid offsets {0, nx * ny}, then the frames' kernels
    struct Staged {
        int64_t off[2], goff[2], cell_off[2];
        FuseFrame fr;
    };
    void* buf;
    RB_TRY(rb_scratch_get(ctx, RB_S_FUSE_FRAMES, sizeof(Staged), &buf));
    Staged* d = (Staged*)buf;
    RB_TRY(grow_pinned(ctx, 2 * sizeof(Staged), stream));
    Staged* h = (Staged*)ctx->pinned;
    const int64_t cells = (int64_t)nx * ny;
    *h = Staged{{0, n}, {0, cells}, {0, 0}, {x_min, y_min, nx, ny}};
    RB_CUDA(cudaMemcpyAsync(d, h, sizeof(Staged), cudaMemcpyHostToDevice, stream));
    const int64_t cuts[2] = {0, 1};
    RB_TRY(fuse_groups<false>(ctx, x, y, inten, d->off, h->off, &d->fr, d->goff, h->goff, cuts, 1, resolution, (double)resolution,
                              cap_cells, nullptr, nullptr, cell_ix, cell_iy, cell_max, d->cell_off, stream));
    int64_t* total = (int64_t*)(h + 1);
    RB_CUDA(cudaMemcpyAsync(total, &d->cell_off[1], sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
    RB_CUDA(cudaStreamSynchronize(stream));
    *n_cells_out = *total;
    if (*total > cap_cells) {
        rb_set_error("rb_fuse_max: %lld cells exceed capacity %lld", (long long)*total, (long long)cap_cells);
        return RB_ERR_CAPACITY;
    }
    return RB_OK;
}
