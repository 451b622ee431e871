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
#include <math.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

namespace {

constexpr int RC_THREADS = 256;

// times[i] = ids[f] and gidx[i] = base + i for the points i of the window's local problem; off = the recording's frame
// offsets, frames [fa, fb) make up the local problem, base = off[fa]
__global__ void __launch_bounds__(RC_THREADS) rec_local_index_kernel(const int64_t* __restrict__ off, const float* __restrict__ ids, int64_t fa,
                                                                    int64_t fb, int64_t base, int64_t n_loc, float* __restrict__ times,
                                                                    int64_t* __restrict__ gidx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_loc) return;
    const int64_t g = base + i;
    int64_t lo = fa, hi = fb - 1;                        // last frame f with off[f] <= g
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (off[mid] <= g) lo = mid; else hi = mid - 1;
    }
    times[i] = ids[lo];
    gidx[i] = g;
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

extern "C" int rb_stdbscan_windowed(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                                    const int64_t* frame_off_host, const float* frame_ids_host, int64_t n_frames,
                                    const int64_t* cuts_host, int64_t n_windows, double eps_space, float eps_time, int min_samples,
                                    const rb_stdbscan_hint* hint, int32_t* labels, uint8_t* core, int64_t* n_clusters, void* stream_) {
    // ---- input checks first (host arrays only): nothing is enqueued for a call that fails them ---------------------
    if (n_clusters) *n_clusters = 0;
    RB_REQUIRE(n_frames >= 1 && frame_off_host && frame_ids_host, "need at least one frame, its offsets and ids");
    RB_REQUIRE(n_windows >= 1 && cuts_host, "need at least one window");
    RB_REQUIRE(frame_off_host[0] == 0, "frame offsets must start at 0");
    for (int64_t f = 0; f < n_frames; ++f) {
        RB_REQUIRE(frame_off_host[f + 1] >= frame_off_host[f], "frame offsets must not decrease");
        const float v = frame_ids_host[f];
        RB_REQUIRE(v == rintf(v) && fabsf(v) < 16777216.f, "frame ids must be integers of magnitude below 2^24");
        RB_REQUIRE(f == 0 || v > frame_ids_host[f - 1], "frame ids must increase strictly");
    }
    RB_REQUIRE(cuts_host[0] == 0 && cuts_host[n_windows] == n_frames, "cuts must run from 0 to the number of frames");
    const int64_t h = eps_time >= 0.f ? (int64_t)floorf(eps_time) : 0;
    for (int64_t k = 0; k < n_windows; ++k) {
        RB_REQUIRE(cuts_host[k + 1] > cuts_host[k], "cuts must increase strictly");
        RB_REQUIRE(n_windows == 1 || cuts_host[k + 1] - cuts_host[k] >= h, "with several windows, each must be at least floor(eps_time) frames long");
    }
    RB_REQUIRE(ctx, "ctx is NULL");
    RB_REQUIRE(x && stride >= 1 && !(z && !y), "bad coordinates");
    const int64_t N = frame_off_host[n_frames];
    if (N == 0) return RB_OK;
    RB_REQUIRE(labels, "labels is NULL");
    cudaStream_t stream = (cudaStream_t)stream_;

    std::vector<Window> win((size_t)n_windows);
    int64_t max_loc = 0;
    for (int64_t k = 0; k < n_windows; ++k) {
        Window& w = win[(size_t)k];
        w.fa = cuts_host[k]; w.fb = cuts_host[k + 1];
        w.la = std::max<int64_t>(w.fa - h, 0); w.lb = std::min<int64_t>(w.fb + h, n_frames);
        w.L = frame_off_host[w.la]; w.A = frame_off_host[w.fa]; w.B = frame_off_host[w.fb]; w.R = frame_off_host[w.lb];
        w.A1 = frame_off_host[std::min(w.fa + h, w.fb)];
        w.B0 = frame_off_host[std::max(w.fb - h, w.fa)];
        RB_REQUIRE(w.R - w.L < ((int64_t)1 << 31) - 1, "a window's local problem has 2^31-1 points or more: use shorter windows");
        max_loc = std::max(max_loc, w.R - w.L);
    }

    // ---- device copies of the frame table; the hint of a window = the caller's box + the window's frame ids ---------
    void* fr_v;
    RB_TRY(rb_scratch_get(ctx, RB_S_REC_FRAMES, sizeof(int64_t) * (size_t)(n_frames + 1) + sizeof(float) * (size_t)n_frames + 64, &fr_v));
    int64_t* d_off = (int64_t*)fr_v;
    float* d_ids = (float*)(d_off + n_frames + 1);
    unsigned long long* d_bad = (unsigned long long*)(((uintptr_t)(d_ids + n_frames) + 15) & ~(uintptr_t)15);
    RB_CUDA(cudaMemcpyAsync(d_off, frame_off_host, sizeof(int64_t) * (size_t)(n_frames + 1), cudaMemcpyHostToDevice, stream));
    RB_CUDA(cudaMemcpyAsync(d_ids, frame_ids_host, sizeof(float) * (size_t)n_frames, cudaMemcpyHostToDevice, stream));
    RB_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(unsigned long long), stream));
    auto window_hint = [&](const Window& w, rb_stdbscan_hint* out) -> const rb_stdbscan_hint* {
        if (!hint) return nullptr;
        *out = *hint;
        out->lo[3] = frame_ids_host[w.la];
        out->hi[3] = frame_ids_host[w.lb - 1];
        out->times_integer = 1;
        return out;
    };

    // ---- one window: rb_stdbscan on the recording's own arrays, with 4 bytes per point of times as the only extra scratch --
    if (n_windows == 1) {
        float* times;
        RB_TRY(scratch_as(ctx, RB_S_REC_LOCAL, (size_t)N, &times));
        RB_TRY(rb_expand_frame_times(ctx, d_off, d_ids, n_frames, N, times, stream_));
        rb_stdbscan_hint hw;
        RB_TRY(rb_stdbscan_enqueue(ctx, x, y, z, stride, times, N, eps_space, eps_time, min_samples, labels, core, window_hint(win[0], &hw),
                                   stream_));
        int64_t ncl = 0;
        RB_TRY(rb_stdbscan_fetch_stats(ctx, &ncl, stream_));         // syncs; fails if the caller's box missed a point
        if (n_clusters) *n_clusters = ncl;
        if (!ctx->retired.empty()) rb_trim(ctx);
        return RB_OK;
    }

    // local problem buffers, sized once for the largest window
    float* t_loc;
    int64_t *g_loc, *k_loc;
    int32_t *cl_loc, *lab_loc;
    uint8_t* c_loc;
    {
        const size_t n = (size_t)max_loc;
        void* p;
        RB_TRY(rb_scratch_get(ctx, RB_S_REC_LOCAL, n * (4 + 8 + 8 + 4 + 4 + 1) + 256, &p));
        g_loc = (int64_t*)p;
        k_loc = g_loc + n;
        t_loc = (float*)(k_loc + n);
        cl_loc = (int32_t*)(t_loc + n);
        lab_loc = cl_loc + n;
        c_loc = (uint8_t*)(lab_loc + n);
    }
    auto local_index = [&](const Window& w) -> int {
        const int64_t n_loc = w.R - w.L;
        RB_CUDA(rb_launch(ctx, rec_local_index_kernel, dim3((unsigned)rb_div_up(n_loc, RC_THREADS)), dim3(RC_THREADS), 0, stream,
                          (const int64_t*)d_off, (const float*)d_ids, w.la, w.lb, w.L, n_loc, t_loc, g_loc));
        RB_LAUNCH_CHECK(ctx);
        return RB_OK;
    };
    auto plan = [&](const Window& w) -> int {
        rb_stdbscan_hint hw;
        const int64_t s = w.L * stride;
        RB_TRY(rb_stdbscan_plan_hinted(ctx, x + s, y ? y + s : nullptr, z ? z + s : nullptr, stride, t_loc, w.R - w.L, eps_space, eps_time,
                                       min_samples, window_hint(w, &hw), stream_));
        const unsigned long long* bad;
        RB_TRY(rb_stdbscan_hint_flag(ctx, &bad));
        RB_CUDA(rb_launch(ctx, rec_flag_or_kernel, dim3(1), dim3(1), 0, stream, bad, d_bad));
        RB_LAUNCH_CHECK(ctx);
        return RB_OK;
    };

    uint8_t* core_all = core;
    if (!core_all) RB_TRY(scratch_as(ctx, RB_S_REC_CORE, (size_t)N, &core_all));

    // ---- pass 1: exact core flags of the owned points ---------------------------------------------------------------
    // a window without points (a stretch of empty frames) has nothing to plan: its zones are empty and stay unpaired
    for (const Window& w : win) {
        if (w.R == w.L) continue;
        RB_TRY(local_index(w));
        RB_TRY(plan(w));
        RB_TRY(rb_stdbscan_cores(ctx, c_loc, stream_));
        RB_CUDA(cudaMemcpyAsync(core_all + w.A, c_loc + (w.A - w.L), (size_t)(w.B - w.A), cudaMemcpyDeviceToDevice, stream));
    }

    // ---- pass 2: components of every local problem, boundary zones run-length encoded -------------------------------
    // zones (local positions): 0 left halo, 1 owned first h frames, 2 owned last h frames, 3 right halo; the zones
    // without a neighbour to pair with are left empty
    auto zones_of = [&](int64_t k, int64_t z8[8]) {
        const Window& w = win[(size_t)k];
        const bool left = k > 0, right = k + 1 < n_windows;
        const int64_t A = w.A - w.L, A1 = w.A1 - w.L, B0 = w.B0 - w.L, B = w.B - w.L, R = w.R - w.L;
        z8[0] = 0;                 z8[1] = left ? A : 0;
        z8[2] = left ? A : 0;      z8[3] = left ? A1 : 0;
        z8[4] = right ? B0 : 0;    z8[5] = right ? B : 0;
        z8[6] = right ? B : 0;     z8[7] = right ? R : 0;
    };
    // window k's encoding: vec[k] = [5 running entry counts | 4 zone lengths | keys[cap[k]] | starts[cap[k]]]. The capacity
    // guess is the largest encoding this context has seen; a window that outgrows it is encoded again on its own.
    auto pass2 = [&](int64_t k, int64_t cap, int64_t* vec) -> int {
        const Window& w = win[(size_t)k];
        int64_t z8[8];
        zones_of(k, z8);
        if (w.R > w.L) {
            RB_TRY(local_index(w));
            RB_TRY(plan(w));
            RB_TRY(rb_stdbscan_set_cores_planned(ctx, core_all + w.L, stream_));
            RB_TRY(rb_stdbscan_components(ctx, g_loc, k_loc, stream_));
        }
        return rb_shard_pack_keys(ctx, k_loc, g_loc, w.R - w.L, z8, cap, vec, stream_);   // n_loc 0: an all-zero encoding
    };
    const int64_t cap0 = std::max<int64_t>(ctx->rec_key_cap, 1 << 15);
    std::vector<int64_t*> vec((size_t)n_windows);
    std::vector<int64_t> cap((size_t)n_windows, cap0);
    {
        int64_t* d_vec;
        RB_TRY(scratch_as(ctx, RB_S_REC_KEYS, (size_t)((9 + 2 * cap0) * n_windows), &d_vec));
        for (int64_t k = 0; k < n_windows; ++k) {
            vec[(size_t)k] = d_vec + k * (9 + 2 * cap0);
            RB_TRY(pass2(k, cap0, vec[(size_t)k]));
        }
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
                RB_TRY(pass2(k, need, d_big));
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
    int64_t* d_tkeys;
    RB_TRY(scratch_as(ctx, RB_S_REC_TABLE, (size_t)(m + m / 2 + 1), &d_tkeys));
    int32_t* d_tids = (int32_t*)(d_tkeys + m);
    if (m) {
        RB_CUDA(cudaMemcpyAsync(d_tkeys, tkeys.data(), sizeof(int64_t) * (size_t)m, cudaMemcpyHostToDevice, stream));
        RB_CUDA(cudaMemcpyAsync(d_tids, tids.data(), sizeof(int32_t) * (size_t)m, cudaMemcpyHostToDevice, stream));
    }

    // ---- pass 3: final labels of the owned points ---------------------------------------------------------------------
    for (const Window& w : win) {
        const int64_t n_loc = w.R - w.L;
        if (n_loc == 0) continue;
        RB_TRY(local_index(w));
        RB_TRY(plan(w));
        RB_TRY(rb_stdbscan_set_cores_planned(ctx, core_all + w.L, stream_));
        RB_TRY(rb_stdbscan_components(ctx, g_loc, k_loc, stream_));
        RB_TRY(rb_relabel(ctx, k_loc, n_loc, d_tkeys, d_tids, m, cl_loc, stream_));
        RB_TRY(rb_stdbscan_assign(ctx, cl_loc, lab_loc, stream_));
        RB_CUDA(cudaMemcpyAsync(labels + w.A, lab_loc + (w.A - w.L), sizeof(int32_t) * (size_t)(w.B - w.A), cudaMemcpyDeviceToDevice, stream));
    }
    unsigned long long bad = 0;
    RB_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof bad, cudaMemcpyDeviceToHost, stream));
    RB_CUDA(cudaStreamSynchronize(stream));
    if (bad) {
        rb_set_error("rb_stdbscan_windowed: the hinted box does not contain every point; the result is invalid");
        return RB_ERR_ARG;
    }
    if (n_clusters) *n_clusters = ncl;
    if (!ctx->retired.empty()) rb_trim(ctx);
    return RB_OK;
}
