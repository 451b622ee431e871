// Ingest: one radar sweep CSV parsed on the GPU (SURVEY.md section 8 f, rank 2; reference 4_temporal_object_tracker.py:
// 184-209 - pd.read_csv(path, header=None, names=[Status, Scale, Range, Gain, Angle, Echo_0..Echo_{E-1}], skiprows=1) is
// ~70 % of the reference's per-sweep load time [SURVEY, probed]).
//
// What the device does: finds the lines, and turns the E echo columns of every data line - 99.5 % of the bytes - into
// uint8, which is what rb_spoke_to_points_u8 consumes (the parsed echoes never exist as float32 on the host and never
// cross PCIe a second time). What stays on the host: the five leading fields of each line (Scale may be a decimal; the
// caller runs the reference's own parser on just those few bytes per line, from the offsets this call returns), file
// discovery and the error message.
//
// The grammar accepted here is deliberately narrow: every echo field is empty (pandas: NaN -> fillna(0) -> 0, T4:206)
// or 1..3 decimal digits with a value <= 255; every data line has exactly E + 5 fields; no blank lines. Anything else
// only sets a status bit - the caller then parses that file with the reference's parser, so exotic input keeps the
// reference's exact behaviour (including its quirks) instead of an imitation of it.
//
// Batches of files (rb_csv_sweeps_lines + rb_csv_parse_sweeps): the text of W files in one buffer, each file at a
// CSV_CHUNK-aligned offset, so a chunk of the newline passes never holds bytes of two files and the padding between files
// is never looked at. The same row parser runs per row; the leading fields Scale and Angle of every row (and Gain of
// row 0) are decoded on the device too, under a grammar on which pandas' C parser is exact (csv_lead_number).
#include "common.cuh"

namespace {

constexpr int CSV_THREADS = 256;
constexpr int CSV_CHUNK = CSV_THREADS * 16;          // bytes per block in the newline passes

// exclusive prefix of a per-thread count over the block; returns the block total through *total
__device__ __forceinline__ int block_exclusive(int v, int* s_warp, int* total) {
    const unsigned lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, incl, d);
        if ((int)lane >= d) incl += o;
    }
    if (lane == 31) s_warp[wid] = incl;
    __syncthreads();
    int base = 0, sum = 0;
#pragma unroll
    for (int w = 0; w < CSV_THREADS / 32; ++w) {
        const int t = s_warp[w];
        if (w < (int)wid) base += t;
        sum += t;
    }
    __syncthreads();
    *total = sum;
    return base + incl - v;
}

// pass 1 (FILL = false): newlines per chunk. pass 2 (FILL = true): their byte offsets, in order.
// file_off == nullptr: one file of n_bytes, status bits go to status[0]. Otherwise the chunk belongs to the last file w
// with file_off[w] <= its first byte; only bytes before file_off[w] + file_len[w] count, status bits go to status[w], and
// pass 1 also flags blank lines (a line after the header that is empty or only "\r").
template <bool FILL>
__global__ void __launch_bounds__(CSV_THREADS) csv_newline_kernel(const uint8_t* __restrict__ text, int64_t n_bytes,
                                                                 const int64_t* __restrict__ file_off, const int64_t* __restrict__ file_len,
                                                                 int n_files, int32_t* __restrict__ chunk_count,
                                                                 const int32_t* __restrict__ chunk_base, int32_t* __restrict__ nl,
                                                                 int64_t nl_cap, int32_t* __restrict__ status) {
    __shared__ int s_warp[CSV_THREADS / 32];
    __shared__ int s_file;
    const int64_t chunk0 = (int64_t)blockIdx.x * CSV_CHUNK;
    const int64_t first = chunk0 + (int64_t)threadIdx.x * 16;
    int64_t lo = 0, hi = n_bytes;
    int32_t* st = status;
    if (file_off) {
        if (threadIdx.x == 0) {
            int a = 0, b = n_files;                                  // first w with file_off[w] > chunk0
            while (a < b) { const int m = (a + b) >> 1; if (file_off[m] <= chunk0) a = m + 1; else b = m; }
            s_file = a - 1;
        }
        __syncthreads();
        const int w = s_file;
        if (w < 0) hi = 0;
        else { lo = file_off[w]; hi = lo + file_len[w]; st = status + w; }
    }
    unsigned hits = 0;
    bool lone_cr = false, blank = false;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        if (first + j >= hi) break;
        const uint8_t ch = text[first + j];
        if (ch == '\n') hits |= 1u << j;
        // a carriage return that is not part of "\r\n": the reference's parser ends a line there, this grammar does not
        if (!FILL && ch == '\r' && (first + j + 1 >= hi || text[first + j + 1] != '\n')) lone_cr = true;
        if (!FILL && file_off && ch == '\n' && first + j - 1 >= lo &&
            (text[first + j - 1] == '\n' || (text[first + j - 1] == '\r' && first + j - 2 >= lo && text[first + j - 2] == '\n')))
            blank = true;
    }
    if (!FILL && lone_cr) atomicOr(st, RB_CSV_NOT_INTEGER);
    if (!FILL && blank) atomicOr(st, RB_CSV_BLANK_LINE);
    int total;
    const int rank = block_exclusive(__popc(hits), s_warp, &total);
    if (!FILL) {
        if (threadIdx.x == 0) chunk_count[blockIdx.x] = total;
        return;
    }
    int64_t slot = (int64_t)chunk_base[blockIdx.x] + rank;
#pragma unroll
    for (int j = 0; j < 16; ++j)
        if (hits >> j & 1) { if (slot < nl_cap) nl[slot] = (int32_t)(first + j); ++slot; }
}

// The echo columns of one data row [start, end) into out[0..n_echo) (zeroed by the caller: an empty field stays 0); the
// fifth comma's offset minus `rel` goes to *prefix_end. Called by every thread of the block; returns RB_CSV_* bits (those
// the calling thread saw; the blank-line and field-count bits are seen by all).
__device__ __forceinline__ unsigned csv_parse_row(const uint8_t* __restrict__ text, int start, int end, int n_echo,
                                                  uint8_t* __restrict__ out, int32_t* __restrict__ prefix_end, int rel,
                                                  int* s_warp) {
    if (end <= start) return RB_CSV_BLANK_LINE;
    int commas_before = 0;                                           // in the chunks already done
    unsigned bad = 0;
    for (int c0 = start; c0 < end; c0 += CSV_THREADS) {
        const int i = c0 + (int)threadIdx.x;
        const bool in = i < end;
        const uint8_t ch = in ? text[i] : 0;
        const bool comma = in && ch == ',';
        if (in && ch == '"') bad |= RB_CSV_NOT_INTEGER;              // quoted fields: leave the file to the reference's parser
        int total;
        const int before = commas_before + block_exclusive(comma ? 1 : 0, s_warp, &total);     // commas left of char i
        if (comma && before == 4) *prefix_end = i - rel;             // the fifth comma ends the leading fields
        const bool field_start = in && (i == start || text[i - 1] == ',');
        if (field_start && before >= 5) {
            const int col = before - 5;
            // the field: [i, first comma or end of line)
            int v = 0, len = 0;
            bool ok = true;
            for (int k = i; k < end; ++k) {
                const uint8_t d = text[k];
                if (d == ',') break;
                if (d < '0' || d > '9' || len == 3) { ok = false; break; }
                v = v * 10 + (d - '0');
                ++len;
            }
            if (!ok) bad |= RB_CSV_NOT_INTEGER;
            else if (v > 255) bad |= RB_CSV_OUT_OF_RANGE;
            else if (col >= n_echo) bad |= RB_CSV_RAGGED;
            else out[col] = (uint8_t)v;                              // empty field: 0 (NaN -> fillna(0))
        }
        commas_before += total;
    }
    if (commas_before != n_echo + 4) bad |= RB_CSV_RAGGED;           // exactly 5 + E fields per line
    return bad;
}

// One block per data row (row r = line r + 1 of the file).
__global__ void __launch_bounds__(CSV_THREADS) csv_parse_rows_kernel(const uint8_t* __restrict__ text, int64_t n_bytes,
                                                                    const int32_t* __restrict__ nl, const int32_t* __restrict__ n_nl_dev,
                                                                    int n_echo, int64_t max_rows, uint8_t* __restrict__ echo,
                                                                    int32_t* __restrict__ row_start, int32_t* __restrict__ prefix_end,
                                                                    int32_t* __restrict__ info) {
    __shared__ int s_warp[CSV_THREADS / 32];
    const int n_nl = *n_nl_dev;
    // lines = newline-terminated pieces, plus an unterminated last one
    const bool open_tail = n_bytes > 0 && text[n_bytes - 1] != '\n';
    const int n_lines = n_nl + (open_tail ? 1 : 0);
    const int64_t r = blockIdx.x;
    if (r == 0 && threadIdx.x == 0) info[0] = n_lines;
    if (n_nl == 0 || r + 1 >= n_lines) return;                       // (no header line, or) no such row
    if (r >= max_rows) { if (threadIdx.x == 0) atomicOr(info + 1, RB_CSV_CAPACITY); return; }
    const int start = nl[r] + 1;
    int end = (r + 1 < n_nl) ? nl[r + 1] : (int)n_bytes;
    if (end > start && text[end - 1] == '\r') --end;                 // \r\n line ends
    if (threadIdx.x == 0) { row_start[r] = start; prefix_end[r] = end; }
    const unsigned bad = csv_parse_row(text, start, end, n_echo, echo + r * (int64_t)n_echo, prefix_end + r, 0, s_warp);
    if (bad) atomicOr(info + 1, (int)bad);
}


// 10^k for k <= 15: every one is exact in double
__constant__ double c_pow10[16] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15};

// A leading field [a, b) under the device grammar: -?D+ (integer_only) or -?D+ / -?D+.D+, at most 15 digits in all, and
// not a negative zero. The value is the digits as an exact double divided once by the exact 10^k (k = fraction digits):
// what pandas' C parser (precise_xstrtod: digits accumulated in a double, one division by a power of ten) gives for such a
// token, and, for an integer column, exactly the int64 it stores (below 2^53). pandas gives -0.0 for "-0" in a float
// column and +0.0 in an integer one, so a negative zero depends on the other rows: it is left to pandas.
__device__ bool csv_lead_number(const uint8_t* __restrict__ t, int a, int b, bool integer_only, double* v) {
    int i = a;
    const bool neg = i < b && t[i] == '-';
    if (neg) ++i;
    double m = 0.0;
    int digits = 0, frac = -1;                                       // frac: digits after the point, -1 = no point
    for (; i < b; ++i) {
        const uint8_t c = t[i];
        if (c >= '0' && c <= '9') {
            if (++digits > 15) return false;
            m = m * 10.0 + (double)(c - '0');                        // exact: below 10^15 < 2^53 (no FMA: --fmad=false)
            if (frac >= 0) ++frac;
        } else if (c == '.' && !integer_only && frac < 0 && digits > 0) {
            frac = 0;
        } else {
            return false;
        }
    }
    if (digits == 0 || frac == 0 || (neg && m == 0.0)) return false;
    if (frac > 0) m = m / c_pow10[frac];
    *v = neg ? -m : m;
    return true;
}

// Batch, pass 1 tail: rows per file from the scanned chunk counts (the file's chunks hold its newlines and nothing else).
__global__ void csv_file_rows_kernel(const uint8_t* __restrict__ text, const int64_t* __restrict__ file_off,
                                     const int64_t* __restrict__ file_len, int n_files, int n_echo,
                                     const int32_t* __restrict__ chunk_base, int32_t* __restrict__ rows, int32_t* __restrict__ status) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_files) return;
    const int64_t lo = file_off[w], len = file_len[w];
    const int n_nl = chunk_base[(lo + len + CSV_CHUNK - 1) / CSV_CHUNK] - chunk_base[lo / CSV_CHUNK];
    const int n_lines = n_nl + ((len > 0 && text[lo + len - 1] != '\n') ? 1 : 0);
    int r = n_nl == 0 ? 0 : n_lines - 1;                             // no header line: no rows
    // a row holds E + 4 commas: more lines than that allows can only be a ragged file, whose rows are not allocated
    if (r > len / (n_echo + 5) + 1) { atomicOr(status + w, RB_CSV_CAPACITY); r = 0; }
    rows[w] = r;
}

// Batch, pass 2: one block per data row of all files. Row r belongs to the last file w with row_base[w] <= r.
__global__ void __launch_bounds__(CSV_THREADS) csv_parse_batch_rows_kernel(
        const uint8_t* __restrict__ text, const int64_t* __restrict__ file_off, const int64_t* __restrict__ file_len, int n_files,
        const int32_t* __restrict__ chunk_base, const int32_t* __restrict__ nl, const int64_t* __restrict__ row_base, int n_echo,
        uint8_t* __restrict__ echo, int32_t* __restrict__ row_start, int32_t* __restrict__ prefix_end, float* __restrict__ angle,
        float* __restrict__ scale, int32_t* __restrict__ gain, int32_t* __restrict__ status) {
    __shared__ int s_warp[CSV_THREADS / 32];
    __shared__ int s_file;
    const int64_t r = blockIdx.x;
    if (threadIdx.x == 0) {
        int a = 0, b = n_files + 1;                                  // first index with row_base > r
        while (a < b) { const int m = (a + b) >> 1; if (row_base[m] <= r) a = m + 1; else b = m; }
        s_file = a - 1;
    }
    __syncthreads();
    const int w = s_file;
    const int64_t lr = r - row_base[w];
    const int64_t lo = file_off[w], hi = lo + file_len[w];
    const int nl0 = chunk_base[lo / CSV_CHUNK];
    const int n_nl = chunk_base[(hi + CSV_CHUNK - 1) / CSV_CHUNK] - nl0;
    const int start = nl[nl0 + lr] + 1;
    int end = (lr + 1 < n_nl) ? nl[nl0 + lr + 1] : (int)hi;
    if (end > start && text[end - 1] == '\r') --end;                 // \r\n line ends
    if (threadIdx.x == 0) { row_start[r] = start - (int)lo; prefix_end[r] = end - (int)lo; }
    unsigned bad = csv_parse_row(text, start, end, n_echo, echo + r * (int64_t)n_echo, prefix_end + r, (int)lo, s_warp);
    if (threadIdx.x == 0 && bad == 0) {
        // Status, Scale, Range, Gain, Angle: the row has E + 4 commas, so all five fields end at one
        int c[5], k = 0;
        for (int i = start; k < 5; ++i)
            if (text[i] == ',') c[k++] = i;
        double s, a, g;
        if (csv_lead_number(text, c[0] + 1, c[1], false, &s) && csv_lead_number(text, c[3] + 1, c[4], false, &a)) {
            scale[r] = __double2float_rn(s);
            angle[r] = __double2float_rn(a);
        } else {
            bad = RB_CSV_LEAD_FIELDS;
        }
        if (lr == 0) {
            if (csv_lead_number(text, c[2] + 1, c[3], true, &g) && g >= -2147483648.0 && g <= 2147483647.0) gain[w] = (int32_t)g;
            else bad = RB_CSV_LEAD_FIELDS;
        }
    }
    if (bad) atomicOr(status + w, (int)bad);
}

}  // namespace

extern "C" int rb_csv_parse_sweep(rb_ctx* ctx, const uint8_t* text, int64_t n_bytes, int n_echo_columns, int64_t max_rows,
                                  uint8_t* echo, int32_t* row_start, int32_t* prefix_end, int32_t* info, void* stream_) {
    RB_REQUIRE(ctx && info, "NULL argument");
    RB_REQUIRE(n_bytes >= 0 && n_bytes < ((int64_t)1 << 31) && n_echo_columns > 0 && max_rows >= 0, "bad sizes");
    cudaStream_t stream = (cudaStream_t)stream_;
    RB_CUDA(cudaMemsetAsync(info, 0, sizeof(int32_t) * 2, stream));
    if (n_bytes == 0) return RB_OK;
    RB_REQUIRE(text && (max_rows == 0 || (echo && row_start && prefix_end)), "NULL buffers");
    const int64_t chunks = rb_div_up(n_bytes, CSV_CHUNK);
    const int64_t nl_cap = max_rows + 2;                             // header + rows (+ one to notice an overflow)
    void* scratch;
    RB_TRY(rb_scratch_get(ctx, RB_S_CSV, sizeof(int32_t) * (size_t)(2 * (chunks + 1) + nl_cap + 1), &scratch));
    int32_t* chunk_count = (int32_t*)scratch;
    int32_t* chunk_base = chunk_count + chunks + 1;
    int32_t* nl = chunk_base + chunks + 1;
    RB_CUDA(rb_launch(ctx, csv_newline_kernel<false>, dim3((unsigned)chunks), dim3(CSV_THREADS), 0, stream, text, n_bytes, nullptr, nullptr, 0, chunk_count, nullptr, nullptr, 0, info + 1));
    RB_LAUNCH_CHECK(ctx);
    RB_TRY(rb_exclusive_scan_i32(ctx, chunk_count, chunk_base, chunks, chunk_base + chunks, stream));      // [chunks] = total
    RB_CUDA(rb_launch(ctx, csv_newline_kernel<true>, dim3((unsigned)chunks), dim3(CSV_THREADS), 0, stream, text, n_bytes, nullptr, nullptr, 0, nullptr, chunk_base, nl, nl_cap, info + 1));
    RB_LAUNCH_CHECK(ctx);
    if (max_rows > 0) RB_CUDA(cudaMemsetAsync(echo, 0, (size_t)max_rows * (size_t)n_echo_columns, stream));
    // one block per possible row; a file with more lines than max_rows + 1 reports RB_CSV_CAPACITY
    RB_CUDA(rb_launch(ctx, csv_parse_rows_kernel, dim3((unsigned)(max_rows + 1)), dim3(CSV_THREADS), 0, stream, text, n_bytes, nl, chunk_base + chunks, n_echo_columns,
                                                                              max_rows, echo, row_start, prefix_end, info));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}

static int csv_batch_check(const uint8_t* text, int64_t n_bytes, const int64_t* file_off, const int64_t* file_len, int n_files,
                           int n_echo_columns) {
    RB_REQUIRE(n_bytes >= 0 && n_bytes < ((int64_t)1 << 31) && n_files >= 0 && n_echo_columns > 0, "bad sizes");
    RB_REQUIRE(n_files == 0 || ((text || n_bytes == 0) && file_off && file_len), "NULL buffers");     // empty files only: no text
    return RB_OK;
}

extern "C" int rb_csv_sweeps_lines(rb_ctx* ctx, const uint8_t* text, int64_t n_bytes, const int64_t* file_off, const int64_t* file_len,
                                   int n_files, int n_echo_columns, int32_t* chunk_base, int32_t* rows, int32_t* status, void* stream_) {
    RB_REQUIRE(ctx, "NULL argument");
    RB_TRY(csv_batch_check(text, n_bytes, file_off, file_len, n_files, n_echo_columns));
    cudaStream_t stream = (cudaStream_t)stream_;
    const int64_t chunks = rb_div_up(n_bytes, CSV_CHUNK);
    RB_REQUIRE(chunk_base, "NULL chunk_base");
    if (n_files == 0 || chunks == 0) {
        RB_CUDA(cudaMemsetAsync(chunk_base, 0, sizeof(int32_t) * (size_t)(chunks + 1), stream));
        if (n_files > 0) {
            RB_CUDA(cudaMemsetAsync(rows, 0, sizeof(int32_t) * (size_t)n_files, stream));
            RB_CUDA(cudaMemsetAsync(status, 0, sizeof(int32_t) * (size_t)n_files, stream));
        }
        return RB_OK;
    }
    RB_REQUIRE(rows && status, "NULL buffers");
    RB_CUDA(cudaMemsetAsync(status, 0, sizeof(int32_t) * (size_t)n_files, stream));
    void* scratch;
    RB_TRY(rb_scratch_get(ctx, RB_S_CSV, sizeof(int32_t) * (size_t)(chunks + 1), &scratch));
    int32_t* chunk_count = (int32_t*)scratch;
    RB_CUDA(rb_launch(ctx, csv_newline_kernel<false>, dim3((unsigned)chunks), dim3(CSV_THREADS), 0, stream, text, n_bytes, file_off, file_len,
                      n_files, chunk_count, nullptr, nullptr, 0, status));
    RB_LAUNCH_CHECK(ctx);
    RB_TRY(rb_exclusive_scan_i32(ctx, chunk_count, chunk_base, chunks, chunk_base + chunks, stream));      // [chunks] = total
    RB_CUDA(rb_launch(ctx, csv_file_rows_kernel, dim3((unsigned)rb_div_up(n_files, 128)), dim3(128), 0, stream, text, file_off, file_len,
                      n_files, n_echo_columns, chunk_base, rows, status));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}

extern "C" int rb_csv_parse_sweeps(rb_ctx* ctx, const uint8_t* text, int64_t n_bytes, const int64_t* file_off, const int64_t* file_len,
                                   int n_files, int n_echo_columns, const int32_t* chunk_base, int64_t n_newlines, const int64_t* row_base,
                                   int64_t n_rows, uint8_t* echo, int32_t* row_start, int32_t* prefix_end, float* angle, float* scale,
                                   int32_t* gain, int32_t* status, void* stream_) {
    RB_REQUIRE(ctx, "NULL argument");
    RB_TRY(csv_batch_check(text, n_bytes, file_off, file_len, n_files, n_echo_columns));
    RB_REQUIRE(n_newlines >= 0 && n_newlines <= n_bytes && n_rows >= 0 && n_rows <= n_newlines, "bad row or newline count");
    if (n_rows == 0) return RB_OK;
    RB_REQUIRE(chunk_base && row_base && echo && row_start && prefix_end && angle && scale && gain && status, "NULL buffers");
    cudaStream_t stream = (cudaStream_t)stream_;
    const int64_t chunks = rb_div_up(n_bytes, CSV_CHUNK);
    void* scratch;
    RB_TRY(rb_scratch_get(ctx, RB_S_CSV, sizeof(int32_t) * (size_t)n_newlines, &scratch));
    int32_t* nl = (int32_t*)scratch;
    RB_CUDA(rb_launch(ctx, csv_newline_kernel<true>, dim3((unsigned)chunks), dim3(CSV_THREADS), 0, stream, text, n_bytes, file_off, file_len,
                      n_files, nullptr, chunk_base, nl, n_newlines, status));
    RB_LAUNCH_CHECK(ctx);
    RB_CUDA(cudaMemsetAsync(echo, 0, (size_t)n_rows * (size_t)n_echo_columns, stream));
    RB_CUDA(rb_launch(ctx, csv_parse_batch_rows_kernel, dim3((unsigned)n_rows), dim3(CSV_THREADS), 0, stream, text, file_off, file_len,
                      n_files, chunk_base, nl, row_base, n_echo_columns, echo, row_start, prefix_end, angle, scale, gain, status));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}
