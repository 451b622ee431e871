// ST-DBSCAN over a whole recording in time windows on one device (rb_stdbscan_windowed; DESIGN.md section 3.8).
//
// The time-sharded protocol of DESIGN.md section 6, run window after window on one context: window k owns frames
// [a, b) and clusters them together with a floor(eps_time)-frame halo on each side. Because the points are frame
// contiguous, a window's local problem is a zero-copy slice of the caller's arrays. Three passes over the windows:
//   1. plan + cores: the core flags of the OWNED points are exact -> one recording-wide core array
//   2. plan + set_cores (now every halo flag is exact too) + components keyed by the recording-wide point index; the
//      keys of the four boundary zones are run-length encoded on the device (rb_shard_pack_keys) and read back
//   3. plan + set_cores + components + rb_relabel with the stitched key -> id table + assign; the owned labels are copied
// Between passes 2 and 3 the host ties the zones of neighbouring windows together (rb_pair_zone_runs) and numbers the
// components (rb_stitch_components). One window is rb_stdbscan itself: one plan, no stitch.
// rb_stdbscan_windowed_wf runs the same passes with the PointCloudWorkF rules (rb_stdbscan_wf): every plan is switched to
// the min_frames core test, and pass 3 assigns border points with recording-wide indices and each cluster's recording-wide
// start, taken from the stitched table.
//
// Each pass is also a C-ABI entry of its own (rb_stdbscan_windowed_pass_cores / _keys / _labels) over a LOCAL problem
// whose windows cover only some of its frames (the owned frames [own_fa, own_fb)) and whose point i has the global
// index index_base + i: the multi-GPU recording (sharded.ShardedRecording) runs the three passes on every rank, with
// the halo exchanges and the stitch of all ranks' windows between them.
#include <math.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

namespace {

constexpr int RC_THREADS = 256;

// times[i] = ids[f] and gidx[i] = index_base + base + i for the points i of the window's local problem; off = the frame
// offsets of the caller's points, frames [fa, fb) make up the window's local problem, base = off[fa]
__global__ void __launch_bounds__(RC_THREADS) rec_local_index_kernel(const int64_t* __restrict__ off, const float* __restrict__ ids, int64_t fa,
                                                                    int64_t fb, int64_t base, int64_t index_base, int64_t n_loc,
                                                                    float* __restrict__ times, int64_t* __restrict__ gidx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_loc) return;
    const int64_t g = base + i;
    int64_t lo = fa, hi = fb - 1;                        // last frame f with off[f] <= g
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (off[mid] <= g) lo = mid; else hi = mid - 1;
    }
    times[i] = ids[lo];
    gidx[i] = index_base + g;
}

__global__ void rec_flag_or_kernel(const unsigned long long* __restrict__ src, unsigned long long* __restrict__ dst) {
    if (*src) *dst = 1ull;
}

struct Window {
    int64_t fa, fb;          // owned frames
    int64_t la, lb;          // frames of the local problem
    int64_t L, A, B, R;      // points: local problem [L, R), owned [A, B)
    int64_t A1, B0;          // end of the owned first-h-frames zone, start of the owned last-h-frames zone
};

template <typename T>
int scratch_as(rb_ctx* ctx, rb_slot slot, size_t count, T** out) {
    void* p;
    RB_TRY(rb_scratch_get(ctx, slot, sizeof(T) * (count ? count : 1), &p));
    *out = (T*)p;
    return RB_OK;
}

}  // namespace

extern "C" int64_t rb_pair_zone_runs(const int64_t* keys_a, const int64_t* starts_a, int64_t n_a, const int64_t* keys_b,
                                     const int64_t* starts_b, int64_t n_b, int64_t* pair_a, int64_t* pair_b, int64_t cap) {
    if (n_a < 0 || n_b < 0 || cap < 0 || (n_a && (!keys_a || !starts_a)) || (n_b && (!keys_b || !starts_b)) || (cap && (!pair_a || !pair_b))) {
        rb_set_error("rb_pair_zone_runs: bad arguments");
        return RB_ERR_ARG;
    }
    if (n_a == 0 || n_b == 0) {
        if (n_a != n_b) { rb_set_error("rb_pair_zone_runs: one zone is empty, the other is not"); return RB_ERR_ARG; }
        return 0;
    }
    if (starts_a[0] != 0 || starts_b[0] != 0) { rb_set_error("rb_pair_zone_runs: a zone's first run must start at 0"); return RB_ERR_ARG; }
    std::vector<std::pair<int64_t, int64_t>> pairs;
    int64_t i = 0, j = 0;
    while (true) {                                       // walk the union of both run starts
        const int64_t ka = keys_a[i], kb = keys_b[j];
        if ((ka >= 0) != (kb >= 0)) {
            rb_set_error("rb_pair_zone_runs: the two encodings disagree on the core points of the zone");
            return RB_ERR_ARG;
        }
        if (ka >= 0) pairs.emplace_back(ka, kb);
        const int64_t na = i + 1 < n_a ? starts_a[i + 1] : INT64_MAX, nb = j + 1 < n_b ? starts_b[j + 1] : INT64_MAX;
        if (na == INT64_MAX && nb == INT64_MAX) break;
        const int64_t next = na < nb ? na : nb;
        if ((na == next && na <= starts_a[i]) || (nb == next && nb <= starts_b[j])) {
            rb_set_error("rb_pair_zone_runs: run starts must increase");
            return RB_ERR_ARG;
        }
        if (na == next) ++i;
        if (nb == next) ++j;
    }
    std::sort(pairs.begin(), pairs.end());
    pairs.erase(std::unique(pairs.begin(), pairs.end()), pairs.end());
    const int64_t m = (int64_t)pairs.size();
    for (int64_t k = 0; k < m && k < cap; ++k) { pair_a[k] = pairs[(size_t)k].first; pair_b[k] = pairs[(size_t)k].second; }
    return m;
}

namespace {

// The windows of one call over a local problem and what its passes share: the host frame table, its device copy, the
// hint-violation flag and the buffers of one window's local problem.
struct Windows {
    rb_ctx* ctx = nullptr;
    const float *x = nullptr, *y = nullptr, *z = nullptr;
    int64_t stride = 1;
    const int64_t* off = nullptr;                 // host: frame offsets of the local problem [n_frames + 1]
    const float* ids = nullptr;                   // host: frame ids [n_frames]
    int64_t n_frames = 0, own_fa = 0, own_fb = 0, index_base = 0, h = 0, max_loc = 0;
    double eps_space = 0.0;
    float eps_time = 0.f;
    int min_samples = 0, min_frames = 0;
    const rb_stdbscan_hint* hint = nullptr;
    void* stream_ = nullptr;
    cudaStream_t stream = nullptr;
    std::vector<Window> win;
    int64_t* d_off = nullptr;
    float* d_ids = nullptr;
    unsigned long long* d_bad = nullptr;
    float* t_loc = nullptr;
    int64_t *g_loc = nullptr, *k_loc = nullptr;
    int32_t *cl_loc = nullptr, *lab_loc = nullptr;
    uint8_t* c_loc = nullptr;
};

// input checks (host arrays only: nothing is enqueued for a call that fails them) and the window list
int windows_check(Windows& W, rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride, const int64_t* frame_off_host,
                  const float* frame_ids_host, int64_t n_frames, int64_t own_fa, int64_t own_fb, const int64_t* cuts_host, int64_t n_windows,
                  int64_t index_base, double eps_space, float eps_time, int min_samples, int min_frames, const rb_stdbscan_hint* hint,
                  void* stream_) {
    RB_REQUIRE(n_frames >= 1 && frame_off_host && frame_ids_host, "need at least one frame, its offsets and ids");
    RB_REQUIRE(n_windows >= 1 && cuts_host, "need at least one window");
    RB_REQUIRE(frame_off_host[0] == 0, "frame offsets must start at 0");
    for (int64_t f = 0; f < n_frames; ++f) {
        RB_REQUIRE(frame_off_host[f + 1] >= frame_off_host[f], "frame offsets must not decrease");
        const float v = frame_ids_host[f];
        RB_REQUIRE(v == rintf(v) && fabsf(v) < 16777216.f, "frame ids must be integers of magnitude below 2^24");
        RB_REQUIRE(f == 0 || v > frame_ids_host[f - 1], "frame ids must increase strictly");
    }
    RB_REQUIRE(0 <= own_fa && own_fa < own_fb && own_fb <= n_frames, "the owned frames must be a non-empty range of the frames");
    RB_REQUIRE(cuts_host[0] == own_fa && cuts_host[n_windows] == own_fb,
               "cuts must run from 0 to the number of frames (from the first owned frame to the end of the owned frames)");
    const int64_t h = eps_time >= 0.f ? (int64_t)floorf(eps_time) : 0;
    for (int64_t k = 0; k < n_windows; ++k) {
        RB_REQUIRE(cuts_host[k + 1] > cuts_host[k], "cuts must increase strictly");
        RB_REQUIRE(n_windows == 1 || cuts_host[k + 1] - cuts_host[k] >= h, "with several windows, each must be at least floor(eps_time) frames long");
    }
    RB_REQUIRE(index_base >= 0, "index_base must be >= 0");
    RB_REQUIRE(ctx, "ctx is NULL");
    RB_REQUIRE(x && stride >= 1 && !(z && !y), "bad coordinates");
    W.ctx = ctx; W.x = x; W.y = y; W.z = z; W.stride = stride;
    W.off = frame_off_host; W.ids = frame_ids_host; W.n_frames = n_frames; W.own_fa = own_fa; W.own_fb = own_fb;
    W.index_base = index_base; W.h = h; W.eps_space = eps_space; W.eps_time = eps_time; W.min_samples = min_samples;
    W.min_frames = min_frames; W.hint = hint; W.stream_ = stream_; W.stream = (cudaStream_t)stream_;
    W.win.resize((size_t)n_windows);
    W.max_loc = 0;
    for (int64_t k = 0; k < n_windows; ++k) {
        Window& w = W.win[(size_t)k];
        w.fa = cuts_host[k]; w.fb = cuts_host[k + 1];
        w.la = std::max<int64_t>(w.fa - h, 0); w.lb = std::min<int64_t>(w.fb + h, n_frames);
        const int64_t* off = frame_off_host;
        w.L = off[w.la]; w.A = off[w.fa]; w.B = off[w.fb]; w.R = off[w.lb];
        w.A1 = off[std::min(w.fa + h, w.fb)];
        w.B0 = off[std::max(w.fb - h, w.fa)];
        RB_REQUIRE(w.R - w.L < ((int64_t)1 << 31) - 1, "a window's local problem has 2^31-1 points or more: use shorter windows");
        W.max_loc = std::max(W.max_loc, w.R - w.L);
    }
    return RB_OK;
}

int check_min_frames(int min_frames, float eps_time) {
    RB_REQUIRE(min_frames >= 0, "min_frames must be 0 (the T4 rules) or >= 1");
    RB_REQUIRE(min_frames == 0 || eps_time <= 30.f, "min_frames needs eps_time <= 30 (the frame set of a neighbourhood is a 64-bit mask)");
    return RB_OK;
}

// device copies of the frame table; the hint-violation flag lives in a slot of its own so that it survives between the
// passes (pass 1 clears it)
int windows_upload(Windows& W, bool clear_flag) {
    rb_ctx* ctx = W.ctx;
    const int64_t n_frames = W.n_frames;
    void* fr_v;
    RB_TRY(rb_scratch_get(ctx, RB_S_REC_FRAMES, sizeof(int64_t) * (size_t)(n_frames + 1) + sizeof(float) * (size_t)n_frames + 64, &fr_v));
    W.d_off = (int64_t*)fr_v;
    W.d_ids = (float*)(W.d_off + n_frames + 1);
    void* fl;
    RB_TRY(rb_scratch_get(ctx, RB_S_REC_FLAG, sizeof(unsigned long long), &fl));
    W.d_bad = (unsigned long long*)fl;
    RB_CUDA(cudaMemcpyAsync(W.d_off, W.off, sizeof(int64_t) * (size_t)(n_frames + 1), cudaMemcpyHostToDevice, W.stream));
    RB_CUDA(cudaMemcpyAsync(W.d_ids, W.ids, sizeof(float) * (size_t)n_frames, cudaMemcpyHostToDevice, W.stream));
    if (clear_flag) RB_CUDA(cudaMemsetAsync(W.d_bad, 0, sizeof(unsigned long long), W.stream));
    return RB_OK;
}

// local problem buffers, sized once for the largest window
int windows_buffers(Windows& W) {
    const size_t n = (size_t)W.max_loc;
    void* p;
    RB_TRY(rb_scratch_get(W.ctx, RB_S_REC_LOCAL, n * (4 + 8 + 8 + 4 + 4 + 1) + 256, &p));
    W.g_loc = (int64_t*)p;
    W.k_loc = W.g_loc + n;
    W.t_loc = (float*)(W.k_loc + n);
    W.cl_loc = (int32_t*)(W.t_loc + n);
    W.lab_loc = W.cl_loc + n;
    W.c_loc = (uint8_t*)(W.lab_loc + n);
    return RB_OK;
}

// the hint of a window = the caller's box + the window's frame ids
const rb_stdbscan_hint* window_hint(const Windows& W, const Window& w, rb_stdbscan_hint* out) {
    if (!W.hint) return nullptr;
    *out = *W.hint;
    out->lo[3] = W.ids[w.la];
    out->hi[3] = W.ids[w.lb - 1];
    out->times_integer = 1;
    return out;
}

int local_index(Windows& W, const Window& w) {
    const int64_t n_loc = w.R - w.L;
    RB_CUDA(rb_launch(W.ctx, rec_local_index_kernel, dim3((unsigned)rb_div_up(n_loc, RC_THREADS)), dim3(RC_THREADS), 0, W.stream,
                      (const int64_t*)W.d_off, (const float*)W.d_ids, w.la, w.lb, w.L, W.index_base, n_loc, W.t_loc, W.g_loc));
    RB_LAUNCH_CHECK(W.ctx);
    return RB_OK;
}

int plan(Windows& W, const Window& w) {
    rb_ctx* ctx = W.ctx;
    rb_stdbscan_hint hw;
    const int64_t s = w.L * W.stride;
    RB_TRY(rb_stdbscan_plan_hinted(ctx, W.x + s, W.y ? W.y + s : nullptr, W.z ? W.z + s : nullptr, W.stride, W.t_loc, w.R - w.L, W.eps_space,
                                   W.eps_time, W.min_samples, window_hint(W, w, &hw), W.stream_));
    if (W.min_frames > 0) RB_TRY(rb_stdbscan_set_min_frames(ctx, W.min_frames));
    const unsigned long long* bad;
    RB_TRY(rb_stdbscan_hint_flag(ctx, &bad));
    RB_CUDA(rb_launch(ctx, rec_flag_or_kernel, dim3(1), dim3(1), 0, W.stream, bad, W.d_bad));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}

// ---- pass 1: exact core flags of the owned points ---------------------------------------------------------------
// a window without points (a stretch of empty frames) has nothing to plan: its zones are empty and stay unpaired
int pass_cores(Windows& W, uint8_t* core_all) {
    for (const Window& w : W.win) {
        if (w.R == w.L) continue;
        RB_TRY(local_index(W, w));
        RB_TRY(plan(W, w));
        RB_TRY(rb_stdbscan_cores(W.ctx, W.c_loc, W.stream_));
        RB_CUDA(cudaMemcpyAsync(core_all + w.A, W.c_loc + (w.A - w.L), (size_t)(w.B - w.A), cudaMemcpyDeviceToDevice, W.stream));
    }
    return RB_OK;
}

// ---- pass 2: components of every local problem, boundary zones run-length encoded -------------------------------
// zones (local positions): 0 left halo, 1 owned first h frames, 2 owned last h frames, 3 right halo; the zones without
// a neighbour to pair with (no window before / after, neither here nor on a neighbouring rank) are left empty.
// Window k's encoding: [5 running entry counts | 4 zone lengths | keys[cap] | starts[cap]] at vec + (k - k0) (9 + 2 cap).
int pass_keys(Windows& W, bool left_nb, bool right_nb, const uint8_t* core_all, int64_t k0, int64_t n_enc, int64_t cap, int64_t* vec) {
    const int64_t n_windows = (int64_t)W.win.size();
    for (int64_t k = k0; k < k0 + n_enc; ++k) {
        const Window& w = W.win[(size_t)k];
        const bool left = k > 0 || left_nb, right = k + 1 < n_windows || right_nb;
        const int64_t A = w.A - w.L, A1 = w.A1 - w.L, B0 = w.B0 - w.L, B = w.B - w.L, R = w.R - w.L;
        int64_t z8[8];
        z8[0] = 0;                 z8[1] = left ? A : 0;
        z8[2] = left ? A : 0;      z8[3] = left ? A1 : 0;
        z8[4] = right ? B0 : 0;    z8[5] = right ? B : 0;
        z8[6] = right ? B : 0;     z8[7] = right ? R : 0;
        if (w.R > w.L) {
            RB_TRY(local_index(W, w));
            RB_TRY(plan(W, w));
            RB_TRY(rb_stdbscan_set_cores_planned(W.ctx, core_all + w.L, W.stream_));
            RB_TRY(rb_stdbscan_components(W.ctx, W.g_loc, W.k_loc, W.stream_));
        }
        // n_loc 0: an all-zero encoding
        RB_TRY(rb_shard_pack_keys(W.ctx, W.k_loc, W.g_loc, w.R - w.L, z8, cap, vec + (k - k0) * (9 + 2 * cap), W.stream_));
    }
    return RB_OK;
}

// ---- pass 3: final labels of the owned points (labels[0] = the first owned point) ---------------------------------
int pass_labels(Windows& W, const uint8_t* core_all, const int64_t* tkeys, const int32_t* tids, int64_t m, const int64_t* start_of,
                int64_t n_start, int32_t* labels, const char* who) {
    rb_ctx* ctx = W.ctx;
    cudaStream_t stream = W.stream;
    int64_t* d_tkeys;
    RB_TRY(scratch_as(ctx, RB_S_REC_TABLE, (size_t)(m + m / 2 + 1 + n_start), &d_tkeys));
    int32_t* d_tids = (int32_t*)(d_tkeys + m);
    int64_t* d_start = d_tkeys + m + m / 2 + 1;
    if (m) {
        RB_CUDA(cudaMemcpyAsync(d_tkeys, tkeys, sizeof(int64_t) * (size_t)m, cudaMemcpyHostToDevice, stream));
        RB_CUDA(cudaMemcpyAsync(d_tids, tids, sizeof(int32_t) * (size_t)m, cudaMemcpyHostToDevice, stream));
    }
    if (n_start) RB_CUDA(cudaMemcpyAsync(d_start, start_of, sizeof(int64_t) * (size_t)n_start, cudaMemcpyHostToDevice, stream));
    const int64_t own0 = W.off[W.own_fa];
    for (const Window& w : W.win) {
        const int64_t n_loc = w.R - w.L;
        if (n_loc == 0) continue;
        RB_TRY(local_index(W, w));
        RB_TRY(plan(W, w));
        RB_TRY(rb_stdbscan_set_cores_planned(ctx, core_all + w.L, W.stream_));
        RB_TRY(rb_stdbscan_components(ctx, W.g_loc, W.k_loc, W.stream_));
        RB_TRY(rb_relabel(ctx, W.k_loc, n_loc, d_tkeys, d_tids, m, W.cl_loc, W.stream_));
        if (W.min_frames > 0) RB_TRY(rb_stdbscan_assign_global(ctx, W.cl_loc, W.lab_loc, W.g_loc, d_start, W.stream_));
        else RB_TRY(rb_stdbscan_assign(ctx, W.cl_loc, W.lab_loc, W.stream_));
        RB_CUDA(cudaMemcpyAsync(labels + (w.A - own0), W.lab_loc + (w.A - w.L), sizeof(int32_t) * (size_t)(w.B - w.A), cudaMemcpyDeviceToDevice,
                                stream));
    }
    unsigned long long bad = 0;
    RB_CUDA(cudaMemcpyAsync(&bad, W.d_bad, sizeof bad, cudaMemcpyDeviceToHost, stream));
    RB_CUDA(cudaStreamSynchronize(stream));
    if (bad) {
        rb_set_error("%s: the hinted box does not contain every point; the result is invalid", who);
        return RB_ERR_ARG;
    }
    return RB_OK;
}

// rb_stdbscan_windowed (min_frames = 0) and rb_stdbscan_windowed_wf (min_frames >= 1, checked by the caller): the three
// passes over all frames of the recording, with the stitch of the windows on the host between passes 2 and 3
int windowed(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride, const int64_t* frame_off_host,
             const float* frame_ids_host, int64_t n_frames, const int64_t* cuts_host, int64_t n_windows, double eps_space, float eps_time,
             int min_samples, int min_frames, const rb_stdbscan_hint* hint, int32_t* labels, uint8_t* core, int64_t* n_clusters,
             void* stream_) {
    Windows W;
    RB_TRY(windows_check(W, ctx, x, y, z, stride, frame_off_host, frame_ids_host, n_frames, 0, n_frames, cuts_host,
                         n_windows, 0, eps_space, eps_time, min_samples, min_frames, hint, stream_));
    const int64_t N = frame_off_host[n_frames];
    if (N == 0) return RB_OK;
    RB_REQUIRE(labels, "labels is NULL");
    cudaStream_t stream = (cudaStream_t)stream_;
    RB_TRY(windows_upload(W, true));

    // ---- one window: rb_stdbscan on the recording's own arrays, with 4 bytes per point of times as the only extra scratch --
    if (n_windows == 1) {
        float* times;
        RB_TRY(scratch_as(ctx, RB_S_REC_LOCAL, (size_t)N, &times));
        RB_TRY(rb_expand_frame_times(ctx, W.d_off, W.d_ids, n_frames, N, times, stream_));
        rb_stdbscan_hint hw;
        RB_TRY(rb_stdbscan_enqueue(ctx, x, y, z, stride, times, N, eps_space, eps_time, min_samples, labels, core, window_hint(W, W.win[0], &hw),
                                   stream_, min_frames));
        int64_t ncl = 0;
        RB_TRY(rb_stdbscan_fetch_stats(ctx, &ncl, stream_));         // syncs; fails if the caller's box missed a point
        if (n_clusters) *n_clusters = ncl;
        if (!ctx->retired.empty()) rb_trim(ctx);
        return RB_OK;
    }

    RB_TRY(windows_buffers(W));
    uint8_t* core_all = core;
    if (!core_all) RB_TRY(scratch_as(ctx, RB_S_REC_CORE, (size_t)N, &core_all));
    RB_TRY(pass_cores(W, core_all));

    // the capacity guess of the zone encodings is the largest encoding this context has seen; a window that outgrows
    // it is encoded again on its own
    const int64_t cap0 = std::max<int64_t>(ctx->rec_key_cap, 1 << 15);
    std::vector<int64_t*> vec((size_t)n_windows);
    std::vector<int64_t> cap((size_t)n_windows, cap0);
    {
        int64_t* d_vec;
        RB_TRY(scratch_as(ctx, RB_S_REC_KEYS, (size_t)((9 + 2 * cap0) * n_windows), &d_vec));
        for (int64_t k = 0; k < n_windows; ++k) vec[(size_t)k] = d_vec + k * (9 + 2 * cap0);
        RB_TRY(pass_keys(W, false, false, core_all, 0, n_windows, cap0, d_vec));
    }
    std::vector<int64_t> head((size_t)(9 * n_windows));
    RB_CUDA(cudaMemcpy2DAsync(head.data(), sizeof(int64_t) * 9, vec[0], sizeof(int64_t) * (size_t)(9 + 2 * cap0), sizeof(int64_t) * 9,
                              (size_t)n_windows, cudaMemcpyDeviceToHost, stream));
    RB_CUDA(cudaStreamSynchronize(stream));
    {
        std::vector<int64_t> big;
        int64_t big_len = 0, need_max = 0;
        for (int64_t k = 0; k < n_windows; ++k) {
            const int64_t need = head[(size_t)(9 * k + 4)];
            need_max = std::max(need_max, need);
            if (need > cap0) { big.push_back(k); big_len += 9 + 2 * need; }
        }
        ctx->rec_key_cap = std::min<int64_t>(std::max(ctx->rec_key_cap, need_max + need_max / 4), (int64_t)1 << 22);
        if (!big.empty()) {
            int64_t* d_big;
            RB_TRY(scratch_as(ctx, RB_S_REC_KEYS_BIG, (size_t)big_len, &d_big));
            for (int64_t k : big) {
                const int64_t need = head[(size_t)(9 * k + 4)];
                vec[(size_t)k] = d_big;
                cap[(size_t)k] = need;
                RB_TRY(pass_keys(W, false, false, core_all, k, 1, need, d_big));
                d_big += 9 + 2 * need;
            }
        }
    }
    std::vector<std::vector<int64_t>> ent((size_t)n_windows);
    for (int64_t k = 0; k < n_windows; ++k) {
        const int64_t tot = head[(size_t)(9 * k + 4)];
        auto& e = ent[(size_t)k];
        e.resize((size_t)(2 * tot + 1));
        if (tot == 0) continue;
        RB_CUDA(cudaMemcpyAsync(e.data(), vec[(size_t)k] + 9, sizeof(int64_t) * (size_t)tot, cudaMemcpyDeviceToHost, stream));
        RB_CUDA(cudaMemcpyAsync(e.data() + tot, vec[(size_t)k] + 9 + cap[(size_t)k], sizeof(int64_t) * (size_t)tot, cudaMemcpyDeviceToHost,
                                stream));
    }
    RB_CUDA(cudaStreamSynchronize(stream));

    // ---- stitch (host): the same boundary points under two windows' keys tie their components together ---------------
    std::vector<int64_t> all_keys, pa, pb;
    auto zone = [&](int64_t k, int z, const int64_t** keys, const int64_t** starts, int64_t* n) {
        const int64_t* hd = &head[(size_t)(9 * k)];
        const int64_t tot = hd[4];
        const int64_t a = z ? hd[z - 1] : 0;
        *keys = ent[(size_t)k].data() + a;
        *starts = ent[(size_t)k].data() + tot + a;
        *n = hd[z] - a;
    };
    for (int64_t k = 0; k < n_windows; ++k) {
        const int64_t* hd = &head[(size_t)(9 * k)];
        all_keys.insert(all_keys.end(), ent[(size_t)k].data() + hd[3], ent[(size_t)k].data() + hd[4]);
        if (k + 1 == n_windows) break;
        const int64_t* hn = &head[(size_t)(9 * (k + 1))];
        for (int pz = 0; pz < 2; ++pz) {                 // (own last | next's left halo), (right halo | next's own first)
            const int za = 2 + pz, zb = pz;
            RB_REQUIRE(hd[5 + za] == hn[5 + zb], "boundary zones of neighbouring windows do not match");
            const int64_t *ka, *sa, *kb, *sb;
            int64_t na, nb;
            zone(k, za, &ka, &sa, &na);
            zone(k + 1, zb, &kb, &sb, &nb);
            const int64_t m = rb_pair_zone_runs(ka, sa, na, kb, sb, nb, nullptr, nullptr, 0);
            if (m < 0) return (int)m;
            const size_t at = pa.size();
            pa.resize(at + (size_t)m); pb.resize(at + (size_t)m);
            if (m) rb_pair_zone_runs(ka, sa, na, kb, sb, nb, pa.data() + at, pb.data() + at, m);
        }
    }
    const int64_t n_keys = (int64_t)all_keys.size();
    std::vector<int64_t> tkeys((size_t)std::max<int64_t>(n_keys, 1));
    std::vector<int32_t> tids((size_t)std::max<int64_t>(n_keys, 1));
    int64_t ncl = 0;
    const int64_t m = rb_stitch_components(all_keys.data(), n_keys, pa.data(), pb.data(), (int64_t)pa.size(), tkeys.data(), tids.data(),
                                           (int64_t)tkeys.size(), &ncl);
    if (m < 0) return (int)m;
    // min_frames: the start of every cluster (its smallest core index over the whole recording) for the WF border rule.
    // A window's component key is the smallest core index of the part of the cluster inside its local problem; the
    // cluster's start can lie outside it. The start is a core point, so it is its own key in the window that owns it;
    // every other key of the cluster is larger, and the table is sorted by key: the first entry of each id.
    const int64_t n_start = min_frames > 0 ? ncl : 0;
    std::vector<int64_t> start_of((size_t)std::max<int64_t>(n_start, 1), -1);
    for (int64_t i = 0; i < m && n_start; ++i)
        if (start_of[(size_t)tids[(size_t)i]] < 0) start_of[(size_t)tids[(size_t)i]] = tkeys[(size_t)i];

    RB_TRY(pass_labels(W, core_all, tkeys.data(), tids.data(), m, start_of.data(), n_start, labels, "rb_stdbscan_windowed"));
    if (n_clusters) *n_clusters = ncl;
    if (!ctx->retired.empty()) rb_trim(ctx);
    return RB_OK;
}

}  // namespace

extern "C" int rb_stdbscan_windowed(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                                    const int64_t* frame_off_host, const float* frame_ids_host, int64_t n_frames,
                                    const int64_t* cuts_host, int64_t n_windows, double eps_space, float eps_time, int min_samples,
                                    const rb_stdbscan_hint* hint, int32_t* labels, uint8_t* core, int64_t* n_clusters, void* stream_) {
    if (n_clusters) *n_clusters = 0;
    return windowed(ctx, x, y, z, stride, frame_off_host, frame_ids_host, n_frames, cuts_host, n_windows, eps_space, eps_time, min_samples,
                    0, hint, labels, core, n_clusters, stream_);
}

extern "C" int rb_stdbscan_windowed_wf(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                                       const int64_t* frame_off_host, const float* frame_ids_host, int64_t n_frames,
                                       const int64_t* cuts_host, int64_t n_windows, double eps_space, float eps_time, int min_samples,
                                       int min_frames, const rb_stdbscan_hint* hint, int32_t* labels, uint8_t* core, int64_t* n_clusters,
                                       void* stream_) {
    if (n_clusters) *n_clusters = 0;
    RB_REQUIRE(min_frames >= 1, "min_frames must be >= 1");
    RB_REQUIRE(eps_time <= 30.f, "rb_stdbscan_windowed_wf needs eps_time <= 30 (the frame set of a neighbourhood is a 64-bit mask)");
    return windowed(ctx, x, y, z, stride, frame_off_host, frame_ids_host, n_frames, cuts_host, n_windows, eps_space, eps_time, min_samples,
                    min_frames, hint, labels, core, n_clusters, stream_);
}

// ---- the passes one by one, over a local problem whose windows cover the owned frames [own_fa, own_fb) -------------
extern "C" int rb_stdbscan_windowed_pass_cores(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                                               const int64_t* frame_off_host, const float* frame_ids_host, int64_t n_frames, int64_t own_fa,
                                               int64_t own_fb, const int64_t* cuts_host, int64_t n_windows, int64_t index_base,
                                               double eps_space, float eps_time, int min_samples, int min_frames,
                                               const rb_stdbscan_hint* hint, uint8_t* core, void* stream_) {
    RB_TRY(check_min_frames(min_frames, eps_time));
    Windows W;
    RB_TRY(windows_check(W, ctx, x, y, z, stride, frame_off_host, frame_ids_host, n_frames, own_fa, own_fb, cuts_host, n_windows, index_base,
                         eps_space, eps_time, min_samples, min_frames, hint, stream_));
    RB_TRY(windows_upload(W, true));
    if (frame_off_host[n_frames] == 0) return RB_OK;
    RB_REQUIRE(core, "core is NULL");
    RB_TRY(windows_buffers(W));
    return pass_cores(W, core);
}

extern "C" int rb_stdbscan_windowed_pass_keys(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                                              const int64_t* frame_off_host, const float* frame_ids_host, int64_t n_frames, int64_t own_fa,
                                              int64_t own_fb, const int64_t* cuts_host, int64_t n_windows, int64_t index_base,
                                              double eps_space, float eps_time, int min_samples, int min_frames,
                                              const rb_stdbscan_hint* hint, int left_neighbour, int right_neighbour, const uint8_t* core,
                                              int64_t first_window, int64_t n_encode, int64_t cap_keys, int64_t* vec,
                                              unsigned long long* hint_outside, void* stream_) {
    RB_TRY(check_min_frames(min_frames, eps_time));
    const int64_t h = eps_time >= 0.f ? (int64_t)floorf(eps_time) : 0;
    RB_REQUIRE(first_window >= 0 && n_encode >= 1 && first_window + n_encode <= n_windows && cap_keys >= 0 && vec, "bad window range or key buffer");
    RB_REQUIRE(!(left_neighbour || right_neighbour) || own_fb - own_fa >= h,
               "next to a neighbour's frames the owned frames must be at least floor(eps_time) frames long");
    RB_REQUIRE(!left_neighbour || own_fa >= h, "the left halo must hold floor(eps_time) frames");
    RB_REQUIRE(!right_neighbour || n_frames - own_fb >= h, "the right halo must hold floor(eps_time) frames");
    Windows W;
    RB_TRY(windows_check(W, ctx, x, y, z, stride, frame_off_host, frame_ids_host, n_frames, own_fa, own_fb, cuts_host, n_windows, index_base,
                         eps_space, eps_time, min_samples, min_frames, hint, stream_));
    RB_TRY(windows_upload(W, false));
    if (frame_off_host[n_frames] > 0) {
        RB_REQUIRE(core, "core is NULL");
        RB_TRY(windows_buffers(W));
    }
    RB_TRY(pass_keys(W, left_neighbour != 0, right_neighbour != 0, core, first_window, n_encode, cap_keys, vec));
    if (hint_outside) {
        RB_CUDA(rb_launch(ctx, rec_flag_or_kernel, dim3(1), dim3(1), 0, W.stream, (const unsigned long long*)W.d_bad, hint_outside));
        RB_LAUNCH_CHECK(ctx);
    }
    return RB_OK;
}

extern "C" int rb_stdbscan_windowed_pass_labels(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                                                const int64_t* frame_off_host, const float* frame_ids_host, int64_t n_frames, int64_t own_fa,
                                                int64_t own_fb, const int64_t* cuts_host, int64_t n_windows, int64_t index_base,
                                                double eps_space, float eps_time, int min_samples, int min_frames,
                                                const rb_stdbscan_hint* hint, const uint8_t* core, const int64_t* table_keys_host,
                                                const int32_t* table_ids_host, int64_t n_table, const int64_t* start_of_host, int64_t n_start,
                                                int32_t* labels, void* stream_) {
    RB_TRY(check_min_frames(min_frames, eps_time));
    Windows W;
    RB_TRY(windows_check(W, ctx, x, y, z, stride, frame_off_host, frame_ids_host, n_frames, own_fa, own_fb, cuts_host, n_windows, index_base,
                         eps_space, eps_time, min_samples, min_frames, hint, stream_));
    RB_REQUIRE(n_table >= 0 && (n_table == 0 || (table_keys_host && table_ids_host)), "bad key table");
    RB_REQUIRE(n_start >= 0 && (n_start == 0 || start_of_host), "bad cluster starts");
    RB_REQUIRE(min_frames == 0 || n_table == 0 || n_start >= 1, "min_frames needs the start of every cluster");
    if (frame_off_host[n_frames] == 0) return RB_OK;
    RB_REQUIRE(core && labels, "core or labels is NULL");
    RB_TRY(windows_upload(W, false));
    RB_TRY(windows_buffers(W));
    return pass_labels(W, core, table_keys_host, table_ids_host, n_table, start_of_host, n_start, labels, "rb_stdbscan_windowed_pass_labels");
}
