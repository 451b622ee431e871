// ASCII PLY body writer (SURVEY.md section 8 f, rank 4): the lines np.savetxt(fh, data, fmt="%.4f %.4f %.4f %d %d %d")
// produces in write_ply_fast (5_gain_fusion_ply_builder.py:370-403; the same bytes as the per-point f-string loop of
// write_ply, T5:345-367, and as the ASCII branch of PointCloudWorkF/stdbscan_denoising_pipeline.py:828-851), for
// float32 coordinates and uint8 colours - without building the float64 table and formatting it row by row in Python.
// The host writer (rb_ply_append_ascii) and the device formatter (rb_ply_format_ascii) share one digit routine, fixed4.
//
// "%.4f" of a float32 value, exactly, for every float32:
//  * |v| < 1e14: v * 10^4 is exact in float64 (24-bit significand times 10^4 = 625 * 2^4 needs at most 34 bits), so
//    printf's correctly rounded, ties-to-even result is nearbyint(v * 1e4) split into integer part and four fraction
//    digits; the sign comes from the sign bit (printf writes "-0.0000" for -0.0 and for negatives that round to zero);
//  * |v| >= 1e14 > 2^24: v is an integer m * 2^s (m < 2^24, s <= 104, so v < 2^128) and printf writes its exact decimal
//    expansion and ".0000": the 128-bit integer is divided by 10^9 limb by limb into at most five 9-digit groups;
//  * inf, -inf and nan print as "inf", "-inf" and "nan" (no sign on a NaN, as Python prints it).
//
// Device side (rb_ply_format_ascii, three launches, no sync): lines are taken 256 per block. Pass 1 counts each line's
// bytes and sums them per block; pass 2 scans the block sums in one block (int64 byte offsets); pass 3 counts again,
// scans the line lengths inside the block, writes every line's end offset, formats the block's lines into shared memory
// and copies the block's bytes out with consecutive threads on consecutive bytes.
// Colours (rb_ply_colors_intensity / rb_ply_colors_gain) and binary records (rb_ply_pack_binary) are element-wise,
// except the per-frame normalisation, which selects the two order statistics of numpy's 99th percentile by radix select
// with one block per frame and then colours that frame.
#include <errno.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <type_traits>
#include <vector>

#include "common.cuh"

namespace {

// three "%.4f" of up to 45 characters ("-", the 39 digits of FLT_MAX, ".0000"), three "%d" of up to 3, 5 spaces, '\n'
constexpr int PLY_LINE_MAX = 150;
constexpr int FMT_THREADS = 256;            // lines per block of the device formatter
constexpr int NORM_THREADS = 512;           // threads of a frame's normalisation block

__host__ __device__ inline int dec_digits(unsigned long long v) {
    int d = 1;
    while (v >= 10ull) { v /= 10ull; ++d; }
    return d;
}

// the d decimal digits of v (d = dec_digits(v), or more for zero padding) at p[0 .. d)
__host__ __device__ inline void put_dec(char* p, unsigned long long v, int d) {
    if (v >> 32 == 0) {
        unsigned u = (unsigned)v;
        for (int i = d - 1; i >= 0; --i) { p[i] = (char)('0' + u % 10u); u /= 10u; }
    } else {
        for (int i = d - 1; i >= 0; --i) { p[i] = (char)('0' + v % 10ull); v /= 10ull; }
    }
}

template <bool W>
__host__ __device__ inline int put_text(char* p, const char* s, int len) {
    if (W) for (int i = 0; i < len; ++i) p[i] = s[i];
    return len;
}

// "%.4f" of f: writes the characters to p when W, returns their number either way
template <bool W>
__host__ __device__ __forceinline__ int fixed4(char* p, float f) {
    if (isnan(f)) return put_text<W>(p, "nan", 3);
    if (isinf(f)) return f < 0 ? put_text<W>(p, "-inf", 4) : put_text<W>(p, "inf", 3);
    int len = 0;
    if (signbit(f)) { if (W) p[0] = '-'; len = 1; }
    if (fabsf(f) < 1e14f) {
        const double r = nearbyint((double)f * 10000.0);           // exact product, ties to even
        const unsigned long long u = (unsigned long long)fabs(r);
        const unsigned long long q = u / 10000ull;
        const int d = dec_digits(q);
        if (W) {
            put_dec(p + len, q, d);
            p[len + d] = '.';
            put_dec(p + len + d + 1, u % 10000ull, 4);
        }
        return len + d + 5;
    }
    // an integer m * 2^s below 2^128: four 32-bit limbs, then 9-digit groups, least significant first
    unsigned bits;
    memcpy(&bits, &f, 4);
    const unsigned m = (bits & 0x7fffffu) | 0x800000u;
    const int s = (int)((bits >> 23) & 0xffu) - 150;                // >= 23 here: |f| >= 1e14 > 2^46
    unsigned limb[4] = {0u, 0u, 0u, 0u};
    const unsigned long long wide = (unsigned long long)m << (s & 31);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (i == (s >> 5)) limb[i] = (unsigned)wide;
        if (i == (s >> 5) + 1) limb[i] = (unsigned)(wide >> 32);
    }
    unsigned g[5];
    int ng = 0;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        unsigned long long rem = 0;
#pragma unroll
        for (int i = 3; i >= 0; --i) {
            const unsigned long long cur = (rem << 32) | limb[i];
            limb[i] = (unsigned)(cur / 1000000000ull);
            rem = cur % 1000000000ull;
        }
        g[k] = (unsigned)rem;
        if (rem || limb[0] || limb[1] || limb[2] || limb[3]) ng = k + 1;
    }
    int at = len;
#pragma unroll
    for (int k = 4; k >= 0; --k) {
        if (k < ng) {
            const int d = k == ng - 1 ? dec_digits(g[k]) : 9;
            if (W) put_dec(p + at, g[k], d);
            at += d;
        }
    }
    return at + put_text<W>(p + at, ".0000", 5);
}

__host__ __device__ inline int put_u8(char* p, unsigned v, bool w) {
    const int d = v >= 100u ? 3 : v >= 10u ? 2 : 1;
    if (w) put_dec(p, v, d);
    return d;
}

// one vertex line "%.4f %.4f %.4f %d %d %d\n"
template <bool W>
__host__ __device__ inline int ply_line(char* p, float x, float y, float z, const uint8_t* c) {
    int at = fixed4<W>(p, x);
    if (W) p[at] = ' ';
    at += 1;
    at += fixed4<W>(p + at, y);
    if (W) p[at] = ' ';
    at += 1;
    at += fixed4<W>(p + at, z);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (W) p[at] = ' ';
        at += 1;
        at += put_u8(p + at, c[k], W);
    }
    if (W) p[at] = '\n';
    return at + 1;
}

// ---- device formatter --------------------------------------------------------------------------------------------
// inclusive block-wide sum scan of v (blockDim.x = T, a multiple of 32); *total = the block's sum
template <int T, typename V>
__device__ inline V block_scan_incl(V v, V* warp_sums, V* total) {
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const V t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= (unsigned)o) v += t;
    }
    if (lane == 31) warp_sums[warp] = v;
    __syncthreads();
    if (warp == 0) {
        V w = lane < T / 32 ? warp_sums[lane] : V(0);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const V t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= (unsigned)o) w += t;
        }
        if (lane < T / 32) warp_sums[lane] = w;
    }
    __syncthreads();
    if (warp) v += warp_sums[warp - 1];
    *total = warp_sums[T / 32 - 1];
    __syncthreads();                                                 // warp_sums may be reused by the caller
    return v;
}

__global__ void __launch_bounds__(FMT_THREADS) ply_tile_bytes_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                                     const float* __restrict__ z, const uint8_t* __restrict__ rgb,
                                                                     int64_t n, int64_t* __restrict__ tile_bytes) {
    __shared__ int sums[FMT_THREADS / 32];
    const int64_t i = (int64_t)blockIdx.x * FMT_THREADS + threadIdx.x;
    const int len = i < n ? ply_line<false>(nullptr, x[i], y[i], z[i], rgb + 3 * i) : 0;
    int total;
    block_scan_incl<FMT_THREADS>(len, sums, &total);
    if (threadIdx.x == 0) tile_bytes[blockIdx.x] = total;
}

// exclusive scan of the per-block byte counts in place, in one block; *total = all bytes
__global__ void __launch_bounds__(1024) ply_scan_tiles_kernel(int64_t* __restrict__ tile, int64_t n_tiles, int64_t* __restrict__ total) {
    __shared__ long long sums[32];
    long long carry = 0;
    for (int64_t base = 0; base < n_tiles; base += 1024) {
        const int64_t i = base + threadIdx.x;
        const long long v = i < n_tiles ? tile[i] : 0;
        long long all;
        const long long incl = block_scan_incl<1024>(v, sums, &all);
        if (i < n_tiles) tile[i] = carry + incl - v;
        carry += all;
    }
    if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(FMT_THREADS) ply_write_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                                const float* __restrict__ z, const uint8_t* __restrict__ rgb,
                                                                int64_t n, const int64_t* __restrict__ tile_base,
                                                                const int64_t* __restrict__ total, int64_t cap,
                                                                char* __restrict__ text, int64_t* __restrict__ line_end) {
    __shared__ char buf[FMT_THREADS * PLY_LINE_MAX];
    __shared__ int sums[FMT_THREADS / 32];
    const int64_t i = (int64_t)blockIdx.x * FMT_THREADS + threadIdx.x;
    float vx = 0.f, vy = 0.f, vz = 0.f;
    uint8_t c[3] = {0, 0, 0};
    int len = 0;
    if (i < n) {
        vx = x[i], vy = y[i], vz = z[i];
        c[0] = rgb[3 * i], c[1] = rgb[3 * i + 1], c[2] = rgb[3 * i + 2];
        len = ply_line<false>(nullptr, vx, vy, vz, c);
    }
    int bytes;
    const int incl = block_scan_incl<FMT_THREADS>(len, sums, &bytes);
    const int64_t base = tile_base[blockIdx.x];
    if (i < n) line_end[i] = base + incl;
    if (*total > cap) return;                                        // too small a buffer: offsets only, no text
    if (i < n) ply_line<true>(buf + (incl - len), vx, vy, vz, c);
    __syncthreads();
    char* out = text + base;
    for (int k = threadIdx.x; k < bytes; k += FMT_THREADS) out[k] = buf[k];
}

__global__ void ply_pack_binary_kernel(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ z,
                                       const uint8_t* __restrict__ rgb, int64_t n, uint8_t* __restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float v[3] = {x[i], y[i], z[i]};
        uint8_t* r = out + 15 * i;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const unsigned b = __float_as_uint(v[k]);
            r[4 * k] = (uint8_t)b, r[4 * k + 1] = (uint8_t)(b >> 8), r[4 * k + 2] = (uint8_t)(b >> 16), r[4 * k + 3] = (uint8_t)(b >> 24);
        }
        r[12] = rgb[3 * i], r[13] = rgb[3 * i + 1], r[14] = rgb[3 * i + 2];
    }
}

// ---- colours -----------------------------------------------------------------------------------------------------
// intensity_to_rgb (T5:292-327) of one value in [0, 255] with numpy >= 2's dtype rules: T = the input's dtype throughout
// (v / 255.0 stays float32 for float32), each ramp evaluated left to right as written, truncated to uint8
template <typename T>
__device__ inline void intensity_rgb_of(T v, uint8_t* c) {
    const T u = v / T(255);
    uint8_t r = 0, g = 0, b = 0;
    if (u < T(0.25)) {
        g = (uint8_t)(unsigned)(u * T(4) * T(255)); b = 255;
    } else if (u < T(0.5)) {
        g = 255; b = (uint8_t)(unsigned)((T(1) - (u - T(0.25)) * T(4)) * T(255));
    } else if (u < T(0.75)) {
        r = (uint8_t)(unsigned)((u - T(0.5)) * T(4) * T(255)); g = 255;
    } else {
        r = 255; g = (uint8_t)(unsigned)((T(1) - (u - T(0.75)) * T(4)) * T(255));
    }
    c[0] = r, c[1] = g, c[2] = b;
}

// a value outside [0, 255] (or NaN) has no defined uint8 in the reference: flag it, colour it black
template <typename T>
__device__ inline void colour_checked(T v, uint8_t* c, int32_t* status) {
    if (!(v >= T(0) && v <= T(255))) {
        atomicOr(status, 1);
        c[0] = c[1] = c[2] = 0;
        return;
    }
    intensity_rgb_of(v, c);
}

template <typename T>
__global__ void colors_intensity_kernel(const T* __restrict__ v, int64_t n, uint8_t* __restrict__ rgb, int32_t* status) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        colour_checked(v[i], rgb + 3 * i, status);
}

__device__ inline uint32_t order_key(float v) {
    const uint32_t b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ inline uint64_t order_key(double v) {
    const uint64_t b = (uint64_t)__double_as_longlong(v);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ inline float key_value(uint32_t k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }
__device__ inline double key_value(uint64_t k) {
    return __longlong_as_double((long long)((k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k));
}

// the k-th smallest key (0-based) of v[0, n) by radix select, 8 bits per pass; *below = keys smaller than it, *equal =
// keys equal to it. Every thread of the block calls it and gets the same results.
template <typename T, typename K>
__device__ __forceinline__ K block_select(const T* __restrict__ v, int64_t n, int64_t k, int* hist, K* shared_key, long long* shared_cnt,
                          long long* below, long long* equal) {
    K prefix = 0, mask = 0;
    long long lt = 0, eq = 0;
    for (int shift = (int)sizeof(K) * 8 - 8; shift >= 0; shift -= 8) {
        for (int b = threadIdx.x; b < 256; b += blockDim.x) hist[b] = 0;
        __syncthreads();
        for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
            const K key = order_key(v[i]);
            if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 0xff], 1);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            long long acc = 0;
            int b = 0;
            for (; b < 255 && acc + hist[b] <= k - lt; ++b) acc += hist[b];
            *shared_key = (K)b;
            shared_cnt[0] = lt + acc;
            shared_cnt[1] = hist[b];
        }
        __syncthreads();
        prefix |= *shared_key << shift;
        mask |= (K)0xff << shift;
        lt = shared_cnt[0];
        eq = shared_cnt[1];
        __syncthreads();
    }
    *below = lt;
    *equal = eq;
    return prefix;
}

// normalize_intensity (T5:276-289) of each frame, then its colours: top = numpy's linear 99th percentile (q = 99 / 100 and
// the virtual index (n - 1) * q in T, gamma = its fraction, _lerp's two formulas), low = the minimum; top <= low gives
// zeros, otherwise clip((v - low) / (top - low) * 255, 0, 255), all in T. One block per frame; a NaN in the frame makes
// every normalised value NaN in the reference, so it is flagged.
template <typename T>
__global__ void __launch_bounds__(NORM_THREADS, 1) colors_normalized_kernel(const T* __restrict__ values, const int64_t* __restrict__ frame_off,
                                                                         uint8_t* __restrict__ rgb, int32_t* status) {
    using K = typename std::conditional<sizeof(T) == 4, uint32_t, uint64_t>::type;
    __shared__ int hist[256];
    __shared__ K skey;
    __shared__ long long scnt[2];
    __shared__ K red[NORM_THREADS / 32];
    __shared__ int nan_seen;
    const int64_t a = frame_off[blockIdx.x], n = frame_off[blockIdx.x + 1] - a;
    if (n <= 0) return;
    const T* v = values + a;
    uint8_t* c = rgb + 3 * a;
    if (threadIdx.x == 0) nan_seen = 0;
    __syncthreads();
    K kmin = ~K(0);
    for (int64_t i = threadIdx.x; i < n; i += NORM_THREADS) {
        if (isnan(v[i])) nan_seen = 1;
        const K key = order_key(v[i]);
        kmin = key < kmin ? key : kmin;
    }
    for (int o = 16; o; o >>= 1) {
        const K t = __shfl_xor_sync(0xffffffffu, kmin, o);
        kmin = t < kmin ? t : kmin;
    }
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = kmin;
    __syncthreads();
    if (nan_seen) {
        if (threadIdx.x == 0) atomicOr(status, 1);
        for (int64_t i = threadIdx.x; i < 3 * n; i += NORM_THREADS) c[i] = 0;
        return;
    }
    kmin = red[0];
    for (int w = 1; w < NORM_THREADS / 32; ++w) kmin = red[w] < kmin ? red[w] : kmin;
    const T low = key_value(kmin);

    const T q = T(99) / T(100);
    const T vi = T(n - 1) * q;
    const T prev = floor(vi);
    const bool above = vi >= T(n - 1);
    const int64_t i0 = above ? n - 1 : (int64_t)prev, i1 = above ? n - 1 : i0 + 1;
    const T gamma = vi - prev;
    long long lt, eq;
    const K k0 = block_select(v, n, i0, hist, &skey, scnt, &lt, &eq);
    K k1 = k0;
    if (i1 >= lt + eq) {                                             // the next order statistic: the smallest key above k0
        K m = ~K(0);
        for (int64_t i = threadIdx.x; i < n; i += NORM_THREADS) {
            const K key = order_key(v[i]);
            if (key > k0 && key < m) m = key;
        }
        for (int o = 16; o; o >>= 1) {
            const K t = __shfl_xor_sync(0xffffffffu, m, o);
            m = t < m ? t : m;
        }
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
        __syncthreads();
        m = red[0];
        for (int w = 1; w < NORM_THREADS / 32; ++w) m = red[w] < m ? red[w] : m;
        k1 = m;
    }
    const T lo_v = key_value(k0), hi_v = key_value(k1);
    const T diff = hi_v - lo_v;
    const T top = gamma >= T(0.5) ? hi_v - diff * (T(1) - gamma) : lo_v + diff * gamma;
    const bool flat = top <= low;
    const T span = top - low;
    for (int64_t i = threadIdx.x; i < n; i += NORM_THREADS) {
        T w = T(0);
        if (!flat) {
            w = (v[i] - low) / span * T(255);
            w = w < T(0) ? T(0) : (w > T(255) ? T(255) : w);
        }
        colour_checked(w, c + 3 * i, status);
    }
}

__global__ void colors_gain_kernel(const int32_t* __restrict__ gains, int64_t n, uint8_t* __restrict__ rgb) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        uint8_t r = 0, g = 0, b = 0;                                 // GAIN_COLORS (T5:45-50), black otherwise
        switch (gains[i]) {
            case 40: r = 0, g = 114, b = 255; break;
            case 50: r = 0, g = 200, b = 83; break;
            case 70: r = 255, g = 165, b = 0; break;
            case 75: r = 255, g = 87, b = 34; break;
            default: break;
        }
        rgb[3 * i] = r, rgb[3 * i + 1] = g, rgb[3 * i + 2] = b;
    }
}

inline unsigned elementwise_blocks(rb_ctx* ctx, int64_t n) {
    const int64_t want = rb_div_up(n, 256), most = (int64_t)ctx->sm_count * 32;
    return (unsigned)(want < most ? want : most);
}

}  // namespace

extern "C" int rb_ply_append_ascii(const char* path, const float* x, const float* y, const float* z, const uint8_t* rgb,
                                   int64_t n) {
    if (!path || n < 0 || (n && (!x || !y || !z || !rgb))) {
        rb_set_error("rb_ply_append_ascii: bad arguments");
        return RB_ERR_ARG;
    }
    FILE* fh = fopen(path, "ab");
    if (!fh) {
        rb_set_error("rb_ply_append_ascii: cannot open %s: %s", path, strerror(errno));
        return RB_ERR_ARG;
    }
    constexpr int64_t CHUNK = 4096;                                 // lines per write
    std::vector<char> buf((size_t)(CHUNK * PLY_LINE_MAX));
    int rc = RB_OK;
    for (int64_t i0 = 0; i0 < n && rc == RB_OK; i0 += CHUNK) {
        const int64_t i1 = i0 + CHUNK < n ? i0 + CHUNK : n;
        char* p = buf.data();
        for (int64_t i = i0; i < i1; ++i) p += ply_line<true>(p, x[i], y[i], z[i], rgb + 3 * i);
        const size_t len = (size_t)(p - buf.data());
        if (fwrite(buf.data(), 1, len, fh) != len) {
            rb_set_error("rb_ply_append_ascii: write to %s failed: %s", path, strerror(errno));
            rc = RB_ERR_ARG;
        }
    }
    if (fclose(fh) != 0 && rc == RB_OK) {
        rb_set_error("rb_ply_append_ascii: closing %s failed: %s", path, strerror(errno));
        rc = RB_ERR_ARG;
    }
    return rc;
}

extern "C" int rb_ply_format_ascii(rb_ctx* ctx, const float* x, const float* y, const float* z, const uint8_t* rgb, int64_t n,
                                   char* text, int64_t cap, int64_t* line_end, int64_t* total, void* stream_) {
    RB_REQUIRE(ctx && total && n >= 0 && cap >= 0, "rb_ply_format_ascii: bad arguments");
    RB_REQUIRE(n == 0 || (x && y && z && rgb && line_end && (text || cap == 0)), "rb_ply_format_ascii: NULL argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n == 0) {
        RB_CUDA(cudaMemsetAsync(total, 0, sizeof(int64_t), stream));
        return RB_OK;
    }
    const int64_t tiles = rb_div_up(n, FMT_THREADS);
    RB_REQUIRE(tiles < (1ll << 31), "rb_ply_format_ascii: too many lines for one call");
    void* buf;
    RB_TRY(rb_scratch_get(ctx, RB_S_PLY_TILES, sizeof(int64_t) * (size_t)tiles, &buf));
    int64_t* tile = (int64_t*)buf;
    RB_CUDA(rb_launch(ctx, ply_tile_bytes_kernel, dim3((unsigned)tiles), dim3(FMT_THREADS), 0, stream, x, y, z, rgb, n, tile));
    RB_LAUNCH_CHECK(ctx);
    RB_CUDA(rb_launch(ctx, ply_scan_tiles_kernel, dim3(1), dim3(1024), 0, stream, tile, tiles, total));
    RB_LAUNCH_CHECK(ctx);
    RB_CUDA(rb_launch(ctx, ply_write_kernel, dim3((unsigned)tiles), dim3(FMT_THREADS), 0, stream, x, y, z, rgb, n,
                      (const int64_t*)tile, (const int64_t*)total, cap, text, line_end));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}

extern "C" int rb_ply_pack_binary(rb_ctx* ctx, const float* x, const float* y, const float* z, const uint8_t* rgb, int64_t n,
                                  uint8_t* out, void* stream_) {
    RB_REQUIRE(ctx && n >= 0, "rb_ply_pack_binary: bad arguments");
    if (n == 0) return RB_OK;
    RB_REQUIRE(x && y && z && rgb && out, "rb_ply_pack_binary: NULL argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    RB_CUDA(rb_launch(ctx, ply_pack_binary_kernel, dim3(elementwise_blocks(ctx, n)), dim3(256), 0, stream, x, y, z, rgb, n, out));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}

extern "C" int rb_ply_colors_intensity(rb_ctx* ctx, const void* values, int is_f64, int64_t n, const int64_t* frame_off,
                                       int64_t n_frames, int normalize, uint8_t* rgb, int32_t* status, void* stream_) {
    RB_REQUIRE(ctx && status && n >= 0 && (is_f64 == 0 || is_f64 == 1), "rb_ply_colors_intensity: bad arguments");
    RB_REQUIRE(n == 0 || (values && rgb), "rb_ply_colors_intensity: NULL argument");
    RB_REQUIRE(!normalize || (frame_off && n_frames >= 0 && n_frames < (1ll << 31)), "rb_ply_colors_intensity: bad frame offsets");
    cudaStream_t stream = (cudaStream_t)stream_;
    RB_CUDA(cudaMemsetAsync(status, 0, sizeof(int32_t), stream));
    if (normalize) {
        if (n_frames == 0) return RB_OK;
        if (is_f64)
            RB_CUDA(rb_launch(ctx, colors_normalized_kernel<double>, dim3((unsigned)n_frames), dim3(NORM_THREADS), 0, stream,
                              (const double*)values, frame_off, rgb, status));
        else
            RB_CUDA(rb_launch(ctx, colors_normalized_kernel<float>, dim3((unsigned)n_frames), dim3(NORM_THREADS), 0, stream,
                              (const float*)values, frame_off, rgb, status));
    } else {
        if (n == 0) return RB_OK;
        const dim3 grid(elementwise_blocks(ctx, n));
        if (is_f64)
            RB_CUDA(rb_launch(ctx, colors_intensity_kernel<double>, grid, dim3(256), 0, stream, (const double*)values, n, rgb, status));
        else
            RB_CUDA(rb_launch(ctx, colors_intensity_kernel<float>, grid, dim3(256), 0, stream, (const float*)values, n, rgb, status));
    }
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}

extern "C" int rb_ply_colors_gain(rb_ctx* ctx, const int32_t* gains, int64_t n, uint8_t* rgb, void* stream_) {
    RB_REQUIRE(ctx && n >= 0, "rb_ply_colors_gain: bad arguments");
    if (n == 0) return RB_OK;
    RB_REQUIRE(gains && rgb, "rb_ply_colors_gain: NULL argument");
    RB_CUDA(rb_launch(ctx, colors_gain_kernel, dim3(elementwise_blocks(ctx, n)), dim3(256), 0, (cudaStream_t)stream_, gains, n, rgb));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}
