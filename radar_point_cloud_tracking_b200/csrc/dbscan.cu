// Temporal ST-DBSCAN (reference 4_temporal_object_tracker.py:443-506, twins 3_stdbscan_point_clouds.py:
// 101-136 and radar_pipeline/processors/clustering.py:49-115; native precedent
// radar-pipeline-rs/src/processors/clustering.rs:209-325).
//
// Result contract (SURVEY.md section 8 N4 - the reference's labels are canonical):
//   neighbour(p,q) <=> fl64 sum_d (double(p_d)-double(q_d))^2 <= eps^2  and  |t_p-t_q| <= eps_t (fl32)
//   core(p) <=> |N(p)| >= min_samples (self included)
//   cluster id = rank of the component's smallest core index; border = smallest id among its core
//   neighbours; noise = -1.
//
// Phases (each an entry point, so the time-sharded multi-GPU driver can exchange data in between;
// rb_stdbscan runs them back to back):
//   plan        bounds -> [host picks the grid] -> counting sort into a dense (t, z, y, x) bucket table
//   cores       neighbour count with early exit -> core flags
//   components  connected components of the core points -> per point the KEY of its component
//               (smallest key among the component's core points; key = caller's global index)
//   assign      given the final id of every core point: ids of border points (smallest id among core
//               neighbours), noise = -1
//
// Two algorithms behind the same phases:
//   TIGHT (integer times, grid fits the budget): spatial cells with a diagonal just under eps and unit
//     time bins. Points of one spatial cell whose bins differ by <= floor(eps_t) are neighbours WITHOUT a
//     distance test; core points of one bucket (cell, bin) are mutually connected, so the union-find runs
//     over buckets: same-cell buckets inside the time window are merged directly, two buckets of
//     different cells need ONE core-core pair within eps (searched by a warp, skipped when the buckets
//     already share a root); border points read per-bucket labels and test only buckets that can lower
//     their id. Dense regions cost almost no distance tests.
//   GENERAL (non-integer times, eps 0, or a grid coarsened to fit memory): cells at least eps wide,
//     exact predicates for every candidate pair, lock-free min-root union-find over core points.
// The exact float64/float32 predicates of the reference decide every pair that is tested; the shortcuts
// only skip tests whose outcome is implied.
#include <float.h>
#include <math.h>

#include "common.cuh"

namespace {

constexpr int DB_THREADS = 256;
constexpr long long KEY_NONE = 0x7fffffffffffffffLL;

struct DbGrid {
    double lo[3];
    double inv_cell;
    double tmin;
    double inv_wt;
    int n[3];          // nx, ny, nz
    int nt;
    int tr;            // time-bin search radius
    int dim;
    int R;             // spatial search radius in cells: 1 (cells >= eps wide) or 2 (tight cells)
    int tight;
};

struct DbPoints {      // strided view of the caller's coordinates
    const float* x; const float* y; const float* z;
    int64_t stride;
    const float* t;
};

// ---- bounds: order-preserving int encoding of floats, block reduce, then atomics ------------------
__device__ __forceinline__ int f2ord(float f) {
    int b = __float_as_int(f);
    return b ^ ((b >> 31) & 0x7fffffff);
}
__host__ __device__ __forceinline__ float ord2f(int o) {
    int b = o ^ ((o >> 31) & 0x7fffffff);
#ifdef __CUDA_ARCH__
    return __int_as_float(b);
#else
    float f; memcpy(&f, &b, 4); return f;
#endif
}

// out[0..3] = min x,y,z,t ; out[4..7] = max ; out[8] = 1 if some time is not an integer
__global__ void __launch_bounds__(DB_THREADS) db_bounds_kernel(DbPoints p, int dim, int64_t n, int* __restrict__ out) {
    int mn[4] = {INT_MAX, INT_MAX, INT_MAX, INT_MAX};
    int mx[4] = {INT_MIN, INT_MIN, INT_MIN, INT_MIN};
    int nonint = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float v[4];
        v[0] = p.x[i * p.stride];
        v[1] = dim > 1 ? p.y[i * p.stride] : 0.f;
        v[2] = dim > 2 ? p.z[i * p.stride] : 0.f;
        v[3] = p.t[i];
        nonint |= !(v[3] == rintf(v[3]) && fabsf(v[3]) < 8388608.f);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            int o = f2ord(v[k]);
            mn[k] = min(mn[k], o);
            mx[k] = max(mx[k], o);
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        mn[k] = __reduce_min_sync(0xffffffffu, mn[k]);
        mx[k] = __reduce_max_sync(0xffffffffu, mx[k]);
    }
    nonint = __any_sync(0xffffffffu, nonint);
    __shared__ int s_mn[4], s_mx[4], s_non;
    if (threadIdx.x < 4) { s_mn[threadIdx.x] = INT_MAX; s_mx[threadIdx.x] = INT_MIN; }
    if (threadIdx.x == 0) s_non = 0;
    __syncthreads();
    if (rb_lane() == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) { atomicMin(s_mn + k, mn[k]); atomicMax(s_mx + k, mx[k]); }
        if (nonint) atomicOr(&s_non, 1);
    }
    __syncthreads();
    if (threadIdx.x < 4) { atomicMin(out + threadIdx.x, s_mn[threadIdx.x]); atomicMax(out + 4 + threadIdx.x, s_mx[threadIdx.x]); }
    if (threadIdx.x == 0 && s_non) atomicOr(out + 8, 1);
}

__global__ void db_bounds_init(int* out) {
    if (threadIdx.x < 4) out[threadIdx.x] = INT_MAX;
    else if (threadIdx.x < 8) out[threadIdx.x] = INT_MIN;
    else if (threadIdx.x < 16) out[threadIdx.x] = 0;
}

// ---- grid cell of a point ---------------------------------------------------------------------------
__device__ __forceinline__ int axis_cell(float v, double lo, double inv, int n) {
    int c = (int)floor(((double)v - lo) * inv);
    return c < 0 ? 0 : (c >= n ? n - 1 : c);
}

// a coordinate outside the grid's box (only possible when the caller's HINT was wrong): clamping it into an edge cell
// would make "same tight cell => neighbour" silently false, so the plan records it and the final read-back fails
__device__ __forceinline__ bool axis_outside(float v, double lo, double inv, int n) {
    const double c = floor(((double)v - lo) * inv);
    return !(c >= 0.0 && c < (double)n);
}

__device__ __forceinline__ int cell_index(const DbGrid& g, float x, float y, float z, float t) {
    int cx = axis_cell(x, g.lo[0], g.inv_cell, g.n[0]);
    int cy = g.dim > 1 ? axis_cell(y, g.lo[1], g.inv_cell, g.n[1]) : 0;
    int cz = g.dim > 2 ? axis_cell(z, g.lo[2], g.inv_cell, g.n[2]) : 0;
    int tb = axis_cell(t, g.tmin, g.inv_wt, g.nt);
    return ((tb * g.n[2] + cz) * g.n[1] + cy) * g.n[0] + cx;
}

// cell id per point + slot of the point inside its cell (the atomic's return value)
// (The slot reservation is pooled per warp: in dense data the 32 consecutive points of a warp fall into a handful of
// buckets and one atomic per point on the same few counters serialises - 7 ms for the 140 M points of a config-4 block.)
__global__ void __launch_bounds__(DB_THREADS) db_cell_kernel(DbPoints p, DbGrid g, int64_t n, int* __restrict__ cell_id,
                                                            int* __restrict__ slot, int* __restrict__ cell_count,
                                                            int* __restrict__ outside /* NULL: bounds were measured */) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned live = __ballot_sync(0xffffffffu, i < n);
    if (i >= n) return;
    float x = p.x[i * p.stride];
    float y = g.dim > 1 ? p.y[i * p.stride] : 0.f;
    float z = g.dim > 2 ? p.z[i * p.stride] : 0.f;
    const float t = p.t[i];
    if (outside) {
        const bool bad = axis_outside(x, g.lo[0], g.inv_cell, g.n[0]) || (g.dim > 1 && axis_outside(y, g.lo[1], g.inv_cell, g.n[1])) ||
                         (g.dim > 2 && axis_outside(z, g.lo[2], g.inv_cell, g.n[2])) || axis_outside(t, g.tmin, g.inv_wt, g.nt);
        if (bad) atomicOr(outside, 1);
    }
    int c = cell_index(g, x, y, z, t);
    cell_id[i] = c;
    const unsigned same = __match_any_sync(live, c);
    const int leader = __ffs(same) - 1;
    int base = 0;
    if ((int)rb_lane() == leader) base = atomicAdd(cell_count + c, __popc(same));
    base = __shfl_sync(same, base, leader);
    slot[i] = base + __popc(same & rb_lanemask_lt());
}

__global__ void __launch_bounds__(DB_THREADS) db_scatter_kernel(DbPoints p, int dim, int64_t n, const int* __restrict__ cell_id,
                                                               const int* __restrict__ slot, const int* __restrict__ cell_start,
                                                               int* __restrict__ sidx, int* __restrict__ scell,
                                                               float* __restrict__ sx, float* __restrict__ sy,
                                                               float* __restrict__ sz, float* __restrict__ st) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int c = cell_id[i];
    int pos = cell_start[c] + slot[i];
    sidx[pos] = (int)i;
    scell[pos] = c;
    sx[pos] = p.x[i * p.stride];
    if (dim > 1) sy[pos] = p.y[i * p.stride];
    if (dim > 2) sz[pos] = p.z[i * p.stride];
    st[pos] = p.t[i];
}

// ---- shared device helpers -----------------------------------------------------------------------------
struct Sorted {
    const float* x; const float* y; const float* z; const float* t;
    const int* cell; const int* cell_start;
};

template <int DIM>
struct Pt { float x, y, z, t; };

template <int DIM>
__device__ __forceinline__ Pt<DIM> load_pt(const Sorted& s, int i) {
    Pt<DIM> p;
    p.x = s.x[i];
    p.y = DIM > 1 ? s.y[i] : 0.f;
    p.z = DIM > 2 ? s.z[i] : 0.f;
    p.t = s.t[i];
    return p;
}

// (A float32 pre-test that decides all pairs outside a 4e-6 band around eps^2 was measured in round 1: the kernels
// are bound by divergence and loads, not by the float64 arithmetic - it made dbt_count_kernel 5 % slower. Not kept.)
template <int DIM>
__device__ __forceinline__ bool near_enough(const Pt<DIM>& a, const Pt<DIM>& b, double eps2) {
    double d = (double)a.x - (double)b.x;                 // sklearn rdist: d += tmp*tmp, float64, no FMA
    double acc = __dmul_rn(d, d);
    if (DIM > 1) { d = (double)a.y - (double)b.y; acc = __dadd_rn(acc, __dmul_rn(d, d)); }
    if (DIM > 2) { d = (double)a.z - (double)b.z; acc = __dadd_rn(acc, __dmul_rn(d, d)); }
    return acc <= eps2;
}

template <int DIM>
__device__ __forceinline__ bool is_neighbour(const Pt<DIM>& a, const Pt<DIM>& b, double eps2, float eps_t) {
    float dt = __fsub_rn(b.t, a.t);                       // T4:486, float32
    if (!(fabsf(dt) <= eps_t)) return false;
    return near_enough<DIM>(a, b, eps2);
}

struct CellPos { int cx, cy, cz, tb; };
__device__ __forceinline__ CellPos decode_cell(const DbGrid& g, int cell) {
    CellPos c;
    c.cx = cell % g.n[0];
    int rest = cell / g.n[0];
    c.cy = rest % g.n[1];
    rest /= g.n[1];
    c.cz = rest % g.n[2];
    c.tb = rest / g.n[2];
    return c;
}

__device__ __forceinline__ void add_counter(unsigned long long* ctr, unsigned long long v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    if (rb_lane() == 0 && v) atomicAdd(ctr, v);
}

__device__ __forceinline__ int uf_find(int* parent, int a) {
    int cur = a;
    while (true) {
        int p = rb_ld_relaxed_s32(parent + cur);
        if (p == cur) return cur;
        int gp = rb_ld_relaxed_s32(parent + p);
        if (gp != p) parent[cur] = gp;                    // path halving; any ancestor is a valid parent
        cur = p;
    }
}

// read-only find for the finalising kernels: while they flatten (parent[x] = root) nothing else may write
// parents, or a late path-halving store could replace a root by a stale ancestor
__device__ __forceinline__ int uf_find_ro(const int* parent, int a) {
    int cur = a;
    while (true) {
        int p = rb_ld_relaxed_s32(parent + cur);
        if (p == cur) return cur;
        cur = p;
    }
}

// roots only ever move to SMALLER indices, so the structure stays acyclic under races
__device__ __forceinline__ void uf_union(int* parent, int a, int b) {
    while (true) {
        a = uf_find(parent, a);
        b = uf_find(parent, b);
        if (a == b) return;
        if (a < b) { int t = a; a = b; b = t; }
        if (atomicCAS(parent + a, a, b) == a) return;
    }
}

// Union of the sets of two nodes, given (possibly stale) roots of theirs: hook the larger index under the smaller with
// ONE atomic when it is still a root. The smaller one need not be a root: parents only point to smaller indices, so a
// node below a root cannot belong to that root's set, and any member of the other set will do as parent. When the CAS
// loses, the value it returns is the parent somebody else gave that node - a member of the same set with a smaller
// index - and the loop goes on from there: no separate find, one atomic per step, the larger index falls every step.
// (Many neighbouring buckets try the same hook at once; with a find-based retry those losers cost half the kernel.)
__device__ __forceinline__ void uf_union_roots(int* parent, int ra, int rb) {
    while (ra != rb) {
        const int hi = max(ra, rb), lo = min(ra, rb);
        const int old = atomicCAS(parent + hi, hi, lo);
        if (old == hi || old == lo) return;
        ra = old; rb = lo;
    }
}

__device__ __forceinline__ long long point_key(const long long* __restrict__ gidx, int orig) {
    return gidx ? gidx[orig] : (long long)orig;
}

// ======================================================================================================
// GENERAL algorithm: exact predicates for every candidate, union-find over core points
// ======================================================================================================
// Calls f(q) for every sorted index q in the cells around `cell`; f returns false to stop.
template <int DIM, typename F>
__device__ __forceinline__ void for_each_candidate(const DbGrid& g, const int* __restrict__ cell_start, int cell, F&& f) {
    const CellPos c = decode_cell(g, cell);
    const int x0 = max(c.cx - 1, 0), x1 = min(c.cx + 1, g.n[0] - 1);
    const int y0 = DIM > 1 ? max(c.cy - 1, 0) : 0, y1 = DIM > 1 ? min(c.cy + 1, g.n[1] - 1) : 0;
    const int z0 = DIM > 2 ? max(c.cz - 1, 0) : 0, z1 = DIM > 2 ? min(c.cz + 1, g.n[2] - 1) : 0;
    const int t0 = max(c.tb - g.tr, 0), t1 = min(c.tb + g.tr, g.nt - 1);
    for (int tt = t0; tt <= t1; ++tt)
        for (int zz = z0; zz <= z1; ++zz)
            for (int yy = y0; yy <= y1; ++yy) {
                int row = ((tt * g.n[2] + zz) * g.n[1] + yy) * g.n[0];
                int b = cell_start[row + x0], e = cell_start[row + x1 + 1];
                for (int q = b; q < e; ++q)
                    if (!f(q)) return;
            }
}

// core[p]: 1 = core, 0 = not core, 2 = not core and alone (no neighbour but itself)
// WF = the PointCloudWorkF variant (stdbscan_denoising_pipeline.py:308-315): the neighbours must also span at least
// min_frames distinct int32(times). |t_q - t_p| <= eps_t <= 30 keeps int(t_q) - int(t_p) + 31 inside a 64-bit mask.
template <int DIM, bool WF>
__global__ void __launch_bounds__(DB_THREADS) dbg_count_kernel(Sorted s, DbGrid g, int n, double eps2, float eps_t,
                                                              int min_samples, int min_frames, uint8_t* __restrict__ core,
                                                              unsigned long long* __restrict__ ctr) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long tests = 0;
    if (p < n) {
        Pt<DIM> a = load_pt<DIM>(s, p);
        int cnt = 0;
        unsigned long long frames = 0;
        const int ta = (int)a.t;
        for_each_candidate<DIM>(g, s.cell_start, s.cell[p], [&](int q) {
            ++tests;
            const Pt<DIM> b = load_pt<DIM>(s, q);
            if (is_neighbour<DIM>(a, b, eps2, eps_t)) {
                ++cnt;
                if (WF) frames |= 1ull << ((int)b.t - ta + 31);
            }
            return cnt < min_samples || cnt < 2 || (WF && __popcll(frames) < min_frames);   // until core is certain
        });
        const bool is_core = cnt >= min_samples && (!WF || __popcll(frames) >= min_frames);
        core[p] = is_core ? 1 : (cnt <= 1 ? 2 : 0);
    }
    add_counter(ctr, tests);
}

__global__ void __launch_bounds__(DB_THREADS) dbg_init_kernel(int n, int* __restrict__ parent, long long* __restrict__ minkey) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) { parent[p] = p; minkey[p] = KEY_NONE; }
}

template <int DIM>
__global__ void __launch_bounds__(DB_THREADS) dbg_union_kernel(Sorted s, DbGrid g, int n, double eps2, float eps_t,
                                                              const uint8_t* __restrict__ core, int* __restrict__ parent,
                                                              unsigned long long* __restrict__ ctr) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long tests = 0;
    if (p < n && core[p] == 1) {
        Pt<DIM> a = load_pt<DIM>(s, p);
        int my_root = p;                                  // a recent root of p: same root => nothing to do
        for_each_candidate<DIM>(g, s.cell_start, s.cell[p], [&](int q) {
            if (q < p && core[q] == 1) {                  // each core-core edge once
                if (rb_ld_relaxed_s32(parent + q) == my_root) return true;
                ++tests;
                if (is_neighbour<DIM>(a, load_pt<DIM>(s, q), eps2, eps_t)) {
                    uf_union(parent, p, q);
                    my_root = uf_find(parent, p);
                }
            }
            return true;
        });
    }
    add_counter(ctr, tests);
}

__global__ void __launch_bounds__(DB_THREADS) dbg_minkey_kernel(int n, const uint8_t* __restrict__ core, int* __restrict__ parent,
                                                               const int* __restrict__ sidx, const long long* __restrict__ gidx,
                                                               long long* __restrict__ minkey) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n || core[p] != 1) return;
    int r = uf_find_ro(parent, p);
    parent[p] = r;
    const long long k = point_key(gidx, sidx[p]);
    if (k < *(volatile long long*)(minkey + r)) atomicMin(minkey + r, k);
}

__global__ void __launch_bounds__(DB_THREADS) dbg_keyout_kernel(int n, const uint8_t* __restrict__ core, const int* __restrict__ parent,
                                                               const int* __restrict__ sidx, const long long* __restrict__ minkey,
                                                               long long* __restrict__ comp_key) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    comp_key[sidx[p]] = core[p] == 1 ? minkey[parent[p]] : -1;
}

// WF border rule (FIFO expansion of stdbscan_denoising_pipeline.py:337-366, see oracle st_dbscan_wf_canonical): the
// cluster of a core neighbour q may be joined only if it started before the border point was looked at (its start
// point = smallest core index = comp_key < the border point's index) or q IS the start point.
template <int DIM, bool WF>
__global__ void __launch_bounds__(DB_THREADS) dbg_border_kernel(Sorted s, DbGrid g, double eps2, float eps_t,
                                                               const uint8_t* __restrict__ core, const int* __restrict__ slabel,
                                                               const int* __restrict__ sidx, const long long* __restrict__ comp_key,
                                                               const int* __restrict__ open_list, const int* __restrict__ n_open,
                                                               int32_t* __restrict__ labels, unsigned long long* __restrict__ ctr) {
    // one thread per LISTED point (core == 0: not core, not alone); everything else got its label from the gather kernel
    const int total = *n_open;
    unsigned long long tests = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int p = open_list[i];
        Pt<DIM> a = load_pt<DIM>(s, p);
        int best = INT_MAX;
        for_each_candidate<DIM>(g, s.cell_start, s.cell[p], [&](int q) {
            if (core[q] == 1) {
                int lq = slabel[q];
                if (lq < best) {                          // only a smaller id can change the answer
                    if (WF) {
                        const int oq = sidx[q];
                        const long long start = comp_key[oq];
                        if (!(start < (long long)sidx[p] || start == (long long)oq)) return true;
                    }
                    ++tests;
                    if (is_neighbour<DIM>(a, load_pt<DIM>(s, q), eps2, eps_t)) best = lq;
                }
            }
            return best != 0;                             // id 0 cannot be beaten
        });
        if (best != INT_MAX) labels[sidx[p]] = best;
    }
    add_counter(ctr, tests);
}

// ======================================================================================================
// TIGHT algorithm: buckets = (time bin, spatial cell), cell diagonal < eps, unit time bins
// ======================================================================================================
struct Window {                    // cells to visit around a point / bucket
    int x0, x1, y0, y1, z0, z1, t0, t1;
};
template <int DIM>
__device__ __forceinline__ Window window_of(const DbGrid& g, const CellPos& c) {
    Window w;
    w.x0 = max(c.cx - g.R, 0); w.x1 = min(c.cx + g.R, g.n[0] - 1);
    w.y0 = DIM > 1 ? max(c.cy - g.R, 0) : 0; w.y1 = DIM > 1 ? min(c.cy + g.R, g.n[1] - 1) : 0;
    w.z0 = DIM > 2 ? max(c.cz - g.R, 0) : 0; w.z1 = DIM > 2 ? min(c.cz + g.R, g.n[2] - 1) : 0;
    w.t0 = max(c.tb - g.tr, 0); w.t1 = min(c.tb + g.tr, g.nt - 1);
    return w;
}

template <int DIM, bool WF>
__global__ void __launch_bounds__(DB_THREADS) dbt_count_kernel(Sorted s, DbGrid g, int n, double eps2, int min_samples, int min_frames,
                                                              uint8_t* __restrict__ core, unsigned long long* __restrict__ ctr) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long tests = 0;
    if (p < n) {
        const int cell = s.cell[p];
        const CellPos c = decode_cell(g, cell);
        const Window w = window_of<DIM>(g, c);
        const int per_t = g.n[0] * g.n[1] * g.n[2];
        const int sp = cell - c.tb * per_t;
        int cnt = 0;
        unsigned long long frames = 0;                    // WF: time bins (= integer times) seen among the neighbours
        // own spatial cell over the time window: neighbours by construction
        for (int tt = w.t0; tt <= w.t1; ++tt) {
            const int k = s.cell_start[tt * per_t + sp + 1] - s.cell_start[tt * per_t + sp];
            cnt += k;
            if (WF && k > 0) frames |= 1ull << (tt - w.t0);
        }
        auto open = [&]() { return cnt < min_samples || (WF && __popcll(frames) < min_frames); };
        if (open()) {
            const Pt<DIM> a = load_pt<DIM>(s, p);
            for (int tt = w.t0; tt <= w.t1 && open(); ++tt)
                for (int zz = w.z0; zz <= w.z1 && open(); ++zz)
                    for (int yy = w.y0; yy <= w.y1 && open(); ++yy) {
                        const int row = ((tt * g.n[2] + zz) * g.n[1] + yy) * g.n[0];
                        const bool own_row = zz == c.cz && yy == c.cy;
                        // the row's cells x0..x1 are one contiguous range of sorted points; skip the own cell
                        const int b = s.cell_start[row + w.x0], e = s.cell_start[row + w.x1 + 1];
                        int hb = e, he = e;                                   // hole = the own cell's points (already counted)
                        if (own_row) { hb = s.cell_start[row + c.cx]; he = s.cell_start[row + c.cx + 1]; }
                        for (int q = b; q < hb && open(); ++q) {
                            ++tests;
                            if (near_enough<DIM>(a, load_pt<DIM>(s, q), eps2)) { ++cnt; if (WF) frames |= 1ull << (tt - w.t0); }
                        }
                        for (int q = he; q < e && open(); ++q) {
                            ++tests;
                            if (near_enough<DIM>(a, load_pt<DIM>(s, q), eps2)) { ++cnt; if (WF) frames |= 1ull << (tt - w.t0); }
                        }
                    }
        }
        core[p] = !open() ? 1 : (cnt <= 1 ? 2 : 0);
    }
    add_counter(ctr, tests);
}

// (Round 2 tried the count in two passes - bucket sizes first, the undecided points compacted and then counted by EIGHT
// lanes per point with a group reduction after every row: 0.94 ms instead of 0.48 ms per 1024-frame block. The kernel is
// bound by the number of instructions per point, not by idle lanes: spreading a point over lanes adds index arithmetic and
// shuffles and loses part of the early exit (151 M instead of 124 M tests). Not kept; profiles/r02_tail_kernels.txt.)
__global__ void __launch_bounds__(DB_THREADS) dbt_bucket_init_kernel(int64_t n_cells, int* __restrict__ b_ncore, int* __restrict__ b_parent,
                                                                    long long* __restrict__ b_minkey, int* __restrict__ n_cb) {
    int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b == 0) *n_cb = 0;
    if (b < n_cells) { b_ncore[b] = 0; b_minkey[b] = KEY_NONE; }            // parents: dbt_bucket_list_kernel
    if (b == n_cells) b_ncore[b] = 0;                                        // scan sentinel
}

// The points are SORTED by bucket, so the lanes of a warp that share a bucket are contiguous: a segmented reduction by
// shuffles leaves every run's result in its first lane, and only that lane touches the bucket's words. One atomic per
// core point on the same bucket serialises in dense data (thousands of points per bucket in config 4: 23 + 26 ms of a
// 70 ms block went into the two kernels below before this).
template <typename T, typename Op>
__device__ __forceinline__ T seg_reduce_sorted(T v, int key, Op op) {
    const unsigned lane = rb_lane();
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const T ov = __shfl_down_sync(0xffffffffu, v, d);
        const int ok = __shfl_down_sync(0xffffffffu, key, d);
        if (lane + d < 32 && ok == key) v = op(v, ov);
    }
    return v;                                              // valid in the first lane of every run of equal keys
}
__device__ __forceinline__ bool seg_head(int key) {
    const int prev = __shfl_up_sync(0xffffffffu, key, 1);
    return rb_lane() == 0 || prev != key;
}

__global__ void __launch_bounds__(DB_THREADS) dbt_bucket_stats_kernel(int n, const uint8_t* __restrict__ core, const int* __restrict__ scell,
                                                                     const int* __restrict__ sidx, const long long* __restrict__ gidx,
                                                                     int* __restrict__ b_ncore, long long* __restrict__ b_minkey) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const bool is_core = p < n && core[p] == 1;
    const int b = p < n ? scell[p] : -1;
    const int cnt = seg_reduce_sorted<int>(is_core ? 1 : 0, b, [](int a, int c) { return a + c; });
    const long long key = seg_reduce_sorted<long long>(is_core ? point_key(gidx, sidx[p]) : KEY_NONE, b,
                                                       [](long long a, long long c) { return a < c ? a : c; });
    if (seg_head(b) && cnt > 0) {
        atomicAdd(b_ncore + b, cnt);
        atomicMin(b_minkey + b, key);
    }
}

// list of the buckets that hold core points; b_label[b] temporarily holds the bucket's slot in the list.
// A block takes LIST_PER_THREAD consecutive buckets per thread, ranks its core buckets with a block scan and reserves
// its part of the list with ONE atomic (one atomic per bucket - even warp aggregated - serialises on the counter's
// address at ~3.4 ns each: 88 us for the 1.1 M core buckets of a 512-frame block). The list comes out sorted inside
// each block's range, so neighbouring list entries are neighbouring buckets - what dbt_union_kernel's lanes want.
// Also: parent = own index for core buckets, -1 for the others (see dbt_union_kernel).
constexpr int LIST_PER_THREAD = 8;
__global__ void __launch_bounds__(DB_THREADS) dbt_bucket_list_kernel(int64_t n_cells, const int* __restrict__ b_ncore,
                                                                    int* __restrict__ cb_list, int* __restrict__ n_cb,
                                                                    int* __restrict__ cb_slot, int* __restrict__ cb_bbox,
                                                                    int* __restrict__ b_parent) {
    __shared__ int warp_tot[DB_THREADS / 32];
    __shared__ int block_base;
    const int64_t first = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * LIST_PER_THREAD;
    unsigned has = 0;
#pragma unroll
    for (int j = 0; j < LIST_PER_THREAD; ++j)
        if (first + j < n_cells && b_ncore[first + j] > 0) has |= 1u << j;
    const int mine = __popc(has);
    // exclusive rank inside the block: warp scan, then the warp totals
    const unsigned lane = rb_lane(), wid = threadIdx.x >> 5;
    int incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, d);
        if ((int)lane >= d) incl += v;
    }
    if (lane == 31) warp_tot[wid] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
#pragma unroll
        for (int w = 0; w < DB_THREADS / 32; ++w) { const int t = warp_tot[w]; warp_tot[w] = run; run += t; }
        block_base = run ? atomicAdd(n_cb, run) : 0;
    }
    __syncthreads();
    int slot = block_base + warp_tot[wid] + incl - mine;
#pragma unroll
    for (int j = 0; j < LIST_PER_THREAD; ++j) {
        const int64_t bkt = first + j;
        if (bkt >= n_cells) break;
        if (has >> j & 1) {
            cb_list[slot] = (int)bkt;
            cb_slot[bkt] = slot;
            b_parent[bkt] = (int)bkt;
#pragma unroll
            for (int k = 0; k < 3; ++k) { cb_bbox[slot * 6 + k] = INT_MAX; cb_bbox[slot * 6 + 3 + k] = INT_MIN; }
            ++slot;
        } else {
            cb_slot[bkt] = -1;
            b_parent[bkt] = -1;                          // "no core points here": the window walk of dbt_union_kernel reads
                                                         // ONE word per bucket (empty / same root as mine / look closer)
        }
    }
}

// bounding box of the core points of every listed bucket (order-preserving int encoding of the floats)
template <int DIM>
__global__ void __launch_bounds__(DB_THREADS) dbt_bucket_bbox_kernel(Sorted s, int n, const uint8_t* __restrict__ core,
                                                                    const int* __restrict__ cb_slot, int* __restrict__ cb_bbox) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const bool is_core = p < n && core[p] == 1;
    const int b = p < n ? s.cell[p] : -1;
    int lo[3] = {INT_MAX, INT_MAX, INT_MAX}, hi[3] = {INT_MIN, INT_MIN, INT_MIN};
    if (is_core) {
        lo[0] = hi[0] = f2ord(s.x[p]);
        if (DIM > 1) lo[1] = hi[1] = f2ord(s.y[p]);
        if (DIM > 2) lo[2] = hi[2] = f2ord(s.z[p]);
    }
    const int any = seg_reduce_sorted<int>(is_core ? 1 : 0, b, [](int a, int c) { return a | c; });
#pragma unroll
    for (int k = 0; k < DIM; ++k) {
        lo[k] = seg_reduce_sorted<int>(lo[k], b, [](int a, int c) { return a < c ? a : c; });
        hi[k] = seg_reduce_sorted<int>(hi[k], b, [](int a, int c) { return a > c ? a : c; });
    }
    if (seg_head(b) && any) {                             // the first lane of the bucket's run in this warp
        int* bb = cb_bbox + (size_t)cb_slot[b] * 6;
#pragma unroll
        for (int k = 0; k < DIM; ++k) { atomicMin(bb + k, lo[k]); atomicMax(bb + 3 + k, hi[k]); }
    }
}

struct BBox { float lo[3], hi[3]; };
template <int DIM>
__device__ __forceinline__ BBox load_bbox(const int* __restrict__ cb_bbox, int slot) {
    BBox b;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        b.lo[k] = k < DIM ? ord2f(__ldg(cb_bbox + (size_t)slot * 6 + k)) : 0.f;
        b.hi[k] = k < DIM ? ord2f(__ldg(cb_bbox + (size_t)slot * 6 + 3 + k)) : 0.f;
    }
    return b;
}
// all core points of the bucket share one position (always so with a single core point): box_gap2 against another such
// box IS the exact squared distance of every core pair, in near_enough's own arithmetic (0 + d*d == d*d)
template <int DIM>
__device__ __forceinline__ bool box_is_point(const BBox& b) {
    bool same = b.lo[0] == b.hi[0];
    if (DIM > 1) same = same && b.lo[1] == b.hi[1];
    if (DIM > 2) same = same && b.lo[2] == b.hi[2];
    return same;
}
// squared gap between two boxes / a point and a box, in the arithmetic of near_enough (float64, no FMA): a lower
// bound of every pair distance it covers, so "gap > eps^2" proves that no pair can pass the exact test
template <int DIM>
__device__ __forceinline__ double box_gap2(const BBox& a, const BBox& b) {
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < DIM; ++k) {
        double d = fmax(fmax((double)a.lo[k] - (double)b.hi[k], (double)b.lo[k] - (double)a.hi[k]), 0.0);
        acc = __dadd_rn(acc, __dmul_rn(d, d));
    }
    return acc;
}
template <int DIM>
__device__ __forceinline__ double point_gap2(const Pt<DIM>& p, const BBox& b) {
    const float v[3] = {p.x, p.y, p.z};
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < DIM; ++k) {
        double d = fmax(fmax((double)b.lo[k] - (double)v[k], (double)v[k] - (double)b.hi[k]), 0.0);
        acc = __dadd_rn(acc, __dmul_rn(d, d));
    }
    return acc;
}

// Same spatial cell, other time bins: all cores are neighbours; linking a bucket to the NEAREST earlier bin
// (inside the time window) that holds cores is enough - that bucket links further back itself. The links form
// chains along time, so no union-find is needed here: parent = that bucket; dbt_flatten_kernel then points
// every bucket at the head of its chain.
__global__ void __launch_bounds__(DB_THREADS) dbt_link_time_kernel(DbGrid g, const int* __restrict__ cb_list, const int* __restrict__ n_cb,
                                                                  const int* __restrict__ b_ncore, int* __restrict__ b_parent) {
    const int total = *n_cb;
    const int per_t = g.n[0] * g.n[1] * g.n[2];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int A = cb_list[i];
        const int tb = A / per_t;
        const int t0 = max(tb - g.tr, 0);
        for (int tt = tb - 1; tt >= t0; --tt) {
            const int b = A - (tb - tt) * per_t;
            if (b_ncore[b] > 0) { b_parent[A] = b; break; }
        }
    }
}

__global__ void __launch_bounds__(DB_THREADS) dbt_flatten_kernel(const int* __restrict__ cb_list, const int* __restrict__ n_cb,
                                                                int* __restrict__ b_parent) {
    const int total = *n_cb;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int b = cb_list[i];
        const int r = uf_find_ro(b_parent, b);
        if (r != b) b_parent[b] = r;                  // only roots are written: concurrent read-only finds stay valid
    }
}

// root lookup through the L1-cached path, for FILTERING only: a cached parent may be stale, but sets only ever
// merge, so "same root" read from stale data is still true; "different" is re-checked by the union itself.
// The walk ends by pointing its start at the root it found. (Compressing every node of the path was measured too: the
// chains are short, the extra loads and stores made the kernel 30 % slower.) Why the store is safe: parents only ever
// point to SMALLER indices of the SAME set, and only non-roots are written (roots change by CAS alone).
__device__ __forceinline__ int uf_find_cached(int* __restrict__ parent, int a) {
    const int p = __ldca(parent + a);
    if (p == a) return a;
    int root = p;
    while (true) {
        const int q = __ldca(parent + root);
        if (q == root) break;
        root = q;
    }
    if (root != p) parent[a] = root;
    return root;
}

// One LANE per bucket A that holds core points (a warp = 32 consecutive entries of the core-bucket list, i.e. mostly
// neighbouring cells): connect A to the earlier buckets (B < A) in the OTHER cells of its window. The warp walks the
// half window row by row (a row = the SIDE buckets with the same dt, dz, dy - consecutive bucket indices): every lane
// loads the parents of its row together (independent loads in flight, and neighbouring lanes
// read neighbouring words), drops the buckets that already share A's root - the common case once the big components
// have formed - and only then looks for ONE core-core pair within eps in what is left: small pairs alone, 32 lanes at
// a time; big pairs with the whole warp. Cells at Chebyshev distance 1 come in a first pass, the far ones in a
// second, when they are usually connected through a near one already.
// (Round-1 history: the first version gave every bucket a warp with one window cell per lane; 20 % of its instructions
// were the per-bucket cell decode and its scattered window loads kept it latency bound - 953 us per 512-frame block.)
template <int DIM>
__global__ void __launch_bounds__(DB_THREADS, DIM == 2 ? 3 : 2) dbt_union_kernel(Sorted s, DbGrid g, const int* __restrict__ cb_list,
                                                              const int* __restrict__ n_cb, const uint8_t* __restrict__ core,
                                                              const int* __restrict__ b_ncore, int* __restrict__ b_parent,
                                                              const int* __restrict__ cb_slot, const int* __restrict__ cb_bbox,
                                                              double eps2, unsigned long long* __restrict__ ctr) {
    constexpr int SIDE = 5;                                         // tight grids search (2R+1)^DIM cells, R = 2
    constexpr int R = SIDE / 2;
    constexpr int RY = DIM > 1 ? R : 0, RZ = DIM > 2 ? R : 0;
    constexpr int SMALL_PAIR = 96;                                  // |A| * |B| up to which ONE lane searches the pair
    constexpr unsigned FULL = 0xffffffffu;
    const unsigned lane = rb_lane();
    const int total = *n_cb;
    const int nxy = g.n[0] * g.n[1];
    const int per_t = nxy * g.n[2];
    const int n_threads = gridDim.x * blockDim.x;
    unsigned long long tests = 0;
    for (int wbase = (blockIdx.x * blockDim.x + threadIdx.x) & ~31; wbase < total; wbase += n_threads) {
        const int i = wbase + (int)lane;
        const bool live = i < total;
        int A = -1, a0 = 0, a1 = 0, root_a = -1;
        CellPos c = {0, 0, 0, 0};
        BBox box_a = {};
        if (live) {
            A = cb_list[i];
            c = decode_cell(g, A);
            a0 = s.cell_start[A]; a1 = s.cell_start[A + 1];
            root_a = uf_find_cached(b_parent, A);
            box_a = load_bbox<DIM>(cb_bbox, i);
        }
        const bool a_point = box_is_point<DIM>(box_a);
        for (int pass = 0; pass < 2; ++pass) {
            for (int dt = -g.tr; dt <= 0; ++dt) {
                const bool t_ok = live && c.tb + dt >= 0;
                for (int dz = -RZ; dz <= RZ; ++dz) {
                    for (int dy = -RY; dy <= RY; ++dy) {
                        // rows after the centre belong to the other half of the window (their buckets look back at A)
                        if (dt == 0 && (dz > 0 || (dz == 0 && dy > 0))) continue;
                        const bool row_far = max(abs(dy), abs(dz)) > 1;
                        if (pass == 0 && row_far) continue;
                        const bool centre_row = dt == 0 && dz == 0 && dy == 0;       // only dx < 0 there
                        const bool same_cell_row = dz == 0 && dy == 0;               // dx = 0 is A's own cell: the time chain
                        const int yy = c.cy + dy, zz = c.cz + dz;
                        const bool row_ok = t_ok && yy >= 0 && yy < g.n[1] && zz >= 0 && zz < g.n[2];
                        const int row = A + dt * per_t + dz * nxy + dy * g.n[0];     // the bucket at dx = 0
                        // ---- parents of the row: -1 = no core points there, A's root = same set already ----
                        unsigned m = 0;
                        int par[SIDE];
#pragma unroll
                        for (int k = 0; k < SIDE; ++k) {
                            const int dx = k - R;
                            const bool far = row_far || abs(dx) > 1;
                            const bool use = row_ok && (int)far == pass && !(centre_row && dx >= 0) && !(same_cell_row && dx == 0) &&
                                             c.cx + dx >= 0 && c.cx + dx < g.n[0];
                            par[k] = use ? __ldca(b_parent + row + dx) : -1;
                            if (par[k] >= 0 && par[k] != root_a) m |= 1u << k;
                        }
                        if (!__any_sync(FULL, m != 0)) continue;
                        // a different parent: bring A's root up to date (it may have been hooked since), finish the walk of
                        // the other bucket (and compress); par[k] = its root
                        if (m) root_a = uf_find_cached(b_parent, root_a);
#pragma unroll
                        for (int k = 0; k < SIDE; ++k) {
                            if (!(m >> k & 1)) continue;
                            if (par[k] != root_a) par[k] = uf_find_cached(b_parent, row + (k - R));
                            if (par[k] == root_a) m &= ~(1u << k);
                        }
                        if (!__any_sync(FULL, m != 0)) continue;
                        // ---- what is left: one bucket of the row at a time ----
                        for (int k = 0; k < SIDE; ++k) {
                            int B = (m >> k & 1) ? row + (k - R) : -1;
                            if (!__any_sync(FULL, B >= 0)) continue;
                            BBox box_b = {};
                            int b0 = 0, b1 = 0, rb = root_a;
                            if (B >= 0) {
#pragma unroll
                                for (int q = 0; q < SIDE; ++q) rb = q == k ? par[q] : rb;          // par[k] without register indexing
                                box_b = load_bbox<DIM>(cb_bbox, __ldg(cb_slot + B));
                                const double gap2 = box_gap2<DIM>(box_a, box_b);
                                ++tests;
                                if (gap2 > eps2) {
                                    B = -1;                        // boxes of the core points more than eps apart: no pair can exist
                                } else if (a_point && box_is_point<DIM>(box_b)) {
                                    uf_union_roots(b_parent, root_a, rb);          // the gap is the exact distance of every core pair
                                    root_a = min(root_a, rb);                      // a member of the merged set, most likely its root
                                    B = -1;
                                } else {
                                    b0 = s.cell_start[B]; b1 = s.cell_start[B + 1];
                                }
                            }
                            // small pairs: the lane searches its pair alone
                            if (B >= 0 && (a1 - a0) * (b1 - b0) <= SMALL_PAIR) {
                                bool found = false;
                                for (int ia = a0; ia < a1 && !found; ++ia) {
                                    if (core[ia] != 1) continue;
                                    const Pt<DIM> pa = load_pt<DIM>(s, ia);
                                    if (point_gap2<DIM>(pa, box_b) > eps2) continue;
                                    for (int jb = b0; jb < b1; ++jb) {
                                        if (core[jb] != 1) continue;
                                        ++tests;
                                        if (near_enough<DIM>(pa, load_pt<DIM>(s, jb), eps2)) { found = true; break; }
                                    }
                                }
                                if (found) {
                                    uf_union_roots(b_parent, root_a, rb);
                                    root_a = min(root_a, rb);
                                }
                                B = -1;
                            }
                            // big pairs: the whole warp, 32 x 32 points in registers at a time
                            unsigned todo = __ballot_sync(FULL, B >= 0);
                            while (todo) {
                                const int src = __ffs(todo) - 1;
                                todo &= todo - 1;
                                const int Aw = __shfl_sync(FULL, A, src), Bw = __shfl_sync(FULL, B, src);
                                int same = 0;
                                if (lane == 0) same = uf_find(b_parent, Aw) == uf_find(b_parent, Bw);
                                if (__shfl_sync(FULL, same, 0)) continue;
                                const int u0 = __shfl_sync(FULL, a0, src), u1 = __shfl_sync(FULL, a1, src);
                                const int w0 = __shfl_sync(FULL, b0, src), w1 = __shfl_sync(FULL, b1, src);
                                BBox ba, bb;
#pragma unroll
                                for (int q = 0; q < 3; ++q) {
                                    ba.lo[q] = __shfl_sync(FULL, box_a.lo[q], src); ba.hi[q] = __shfl_sync(FULL, box_a.hi[q], src);
                                    bb.lo[q] = __shfl_sync(FULL, box_b.lo[q], src); bb.hi[q] = __shfl_sync(FULL, box_b.hi[q], src);
                                }
                                bool found = false;
                                for (int ia0 = u0; ia0 < u1 && !found; ia0 += 32) {
                                    const int ia_l = ia0 + (int)lane;
                                    Pt<DIM> mine_a = {};
                                    bool use_a = false;
                                    if (ia_l < u1 && core[ia_l] == 1) { mine_a = load_pt<DIM>(s, ia_l); use_a = point_gap2<DIM>(mine_a, bb) <= eps2; }
                                    const unsigned act_a = __ballot_sync(FULL, use_a);
                                    if (!act_a) continue;
                                    for (int jb0 = w0; jb0 < w1 && !found; jb0 += 32) {
                                        const int jb_l = jb0 + (int)lane;
                                        Pt<DIM> mine_b = {};
                                        bool use_b = false;
                                        if (jb_l < w1 && core[jb_l] == 1) { mine_b = load_pt<DIM>(s, jb_l); use_b = point_gap2<DIM>(mine_b, ba) <= eps2; }
                                        if (!__any_sync(FULL, use_b)) continue;
                                        unsigned act = act_a;
                                        while (act) {
                                            const int la = __ffs(act) - 1;
                                            act &= act - 1;
                                            Pt<DIM> pa;
                                            pa.x = __shfl_sync(FULL, mine_a.x, la);
                                            pa.y = DIM > 1 ? __shfl_sync(FULL, mine_a.y, la) : 0.f;
                                            pa.z = DIM > 2 ? __shfl_sync(FULL, mine_a.z, la) : 0.f;
                                            pa.t = 0.f;
                                            bool ok = false;
                                            if (use_b) { ++tests; ok = near_enough<DIM>(pa, mine_b, eps2); }
                                            if (__any_sync(FULL, ok)) { found = true; break; }
                                        }
                                    }
                                }
                                if (found && lane == 0) uf_union(b_parent, Aw, Bw);
                                if (found && (int)lane == src) root_a = uf_find_cached(b_parent, A);
                            }
                        }
                    }
                }
            }
        }
    }
    add_counter(ctr, tests);
}

__global__ void __launch_bounds__(DB_THREADS) dbt_compmin_kernel(const int* __restrict__ cb_list, const int* __restrict__ n_cb,
                                                                int* __restrict__ b_parent, long long* __restrict__ b_minkey) {
    const int total = *n_cb;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int b = cb_list[i];
        const int r = uf_find_ro(b_parent, b);
        if (r != b) {
            b_parent[b] = r;
            const long long k = b_minkey[b];
            // most buckets do not hold their component's smallest key: look before paying for a contended atomic
            if (k < *(volatile long long*)(b_minkey + r)) atomicMin(b_minkey + r, k);
        }
    }
}

__global__ void __launch_bounds__(DB_THREADS) dbt_keyout_kernel(int n, const uint8_t* __restrict__ core, const int* __restrict__ scell,
                                                               const int* __restrict__ sidx, const int* __restrict__ b_parent,
                                                               const long long* __restrict__ b_minkey, long long* __restrict__ comp_key) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    long long k = -1;
    if (core[p] == 1) { const int b = scell[p]; k = b_minkey[b_parent[b]]; }   // parents were flattened by dbt_compmin_kernel
    comp_key[sidx[p]] = k;
}

// sorted copy of the core labels + the label of every bucket that holds cores (all its cores share it); final label of
// every core point (its id) and of every point that is certainly noise (-1); the points that may be border points
// (core == 0: not core, but not alone) are LISTED - one warp-aggregated atomic per warp - so that the border search runs
// over a dense list instead of one busy lane in a hundred.
__global__ void __launch_bounds__(DB_THREADS) db_gather_labels_kernel(int n, const uint8_t* __restrict__ core, const int* __restrict__ sidx,
                                                                     const int* __restrict__ scell, const int32_t* core_label,
                                                                     int* __restrict__ slabel, int* __restrict__ b_label, int32_t* labels,
                                                                     int* __restrict__ open_list, int* __restrict__ n_open) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    bool open = false;
    if (p < n) {
        const int orig = sidx[p];
        int lab = -1;
        if (core[p] == 1) { lab = core_label[orig]; if (b_label) b_label[scell[p]] = lab; }     // (core_label may alias labels:
        slabel[p] = lab;                                                                         //  element orig belongs to this thread)
        labels[orig] = lab;
        open = core[p] == 0;
    }
    const unsigned m = __ballot_sync(0xffffffffu, open);
    if (m) {
        int base = 0;
        if (rb_lane() == (unsigned)(__ffs(m) - 1)) base = atomicAdd(n_open, __popc(m));
        base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
        if (open) open_list[base + __popc(m & rb_lanemask_lt())] = p;
    }
}

// One THREAD per listed point (core == 0: not core, not alone), the list being dense. Step 1: cores of the own spatial
// cell inside the time window are neighbours by construction, their bucket labels count without a test. Step 2: the
// other buckets of the window, row by row; only a bucket whose label can lower the best id so far is searched for ONE
// core point within eps, and id 0 ends the search.
// (Round 1 ran the same search with one thread per point over ALL points: the ~10 % that are border candidates sat
// nearly alone in their warps, 3.3 active lanes per warp. Round 2 first gave every listed point a WARP with the lanes
// over the window's rows: no faster (0.31 ms per 1024-frame block) - 25 lanes search at once where the serial walk stops
// at the first bucket of cluster 0, 4.9 M instead of 1.2 M tests. The dense list with the serial early-exit walk keeps
// both: full warps and few tests.)
template <int DIM, bool WF>
__global__ void __launch_bounds__(DB_THREADS) dbt_border_kernel(Sorted s, DbGrid g, double eps2, const uint8_t* __restrict__ core,
                                                               const int* __restrict__ sidx, const int* __restrict__ open_list,
                                                               const int* __restrict__ n_open, const int* __restrict__ b_ncore,
                                                               const int* __restrict__ core_start, const int* __restrict__ b_label,
                                                               const int* __restrict__ b_parent, const long long* __restrict__ b_minkey,
                                                               int32_t* __restrict__ labels, unsigned long long* __restrict__ ctr) {
    const int total = *n_open;
    const int per_t = g.n[0] * g.n[1] * g.n[2];
    unsigned long long tests = 0;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < total; k += gridDim.x * blockDim.x) {
        const int p = open_list[k];
        const int cell = s.cell[p];
        const CellPos c = decode_cell(g, cell);
        const Window w = window_of<DIM>(g, c);
        const int sp = cell - c.tb * per_t;
        const long long me = sidx[p];
        int best = INT_MAX;
        for (int tt = w.t0; tt <= w.t1; ++tt) {
            const int b = tt * per_t + sp;
            if (b_ncore[b] <= 0) continue;
            if (WF) {
                // WF border rule: the bucket's cluster must have started before this point was looked at, or its start
                // point itself (the core whose index is the component key) must be among the neighbours
                const long long start = b_minkey[b_parent[b]];
                bool ok = start < me;
                for (int q = s.cell_start[b]; !ok && q < s.cell_start[b + 1]; ++q) ok = core[q] == 1 && (long long)sidx[q] == start;
                if (!ok) continue;
            }
            best = min(best, b_label[b]);
        }
        if (best != 0) {
            const Pt<DIM> a = load_pt<DIM>(s, p);
            for (int tt = w.t0; tt <= w.t1 && best != 0; ++tt)
                for (int zz = w.z0; zz <= w.z1 && best != 0; ++zz)
                    for (int yy = w.y0; yy <= w.y1 && best != 0; ++yy) {
                        const int row = ((tt * g.n[2] + zz) * g.n[1] + yy) * g.n[0];
                        if (core_start[row + w.x1 + 1] == core_start[row + w.x0]) continue;      // no core in this row
                        for (int xx = w.x0; xx <= w.x1; ++xx) {
                            const int b = row + xx;
                            if (b_ncore[b] == 0 || (xx == c.cx && yy == c.cy && zz == c.cz)) continue;
                            const int lb = b_label[b];
                            if (lb >= best) continue;                 // only a smaller id can change the answer
                            const long long start = WF ? b_minkey[b_parent[b]] : 0;
                            const bool any_core = !WF || start < me;   // WF: else only the start point itself counts
                            for (int q = s.cell_start[b]; q < s.cell_start[b + 1]; ++q) {
                                if (core[q] != 1 || (!any_core && (long long)sidx[q] != start)) continue;
                                ++tests;
                                if (near_enough<DIM>(a, load_pt<DIM>(s, q), eps2)) { best = lb; break; }
                            }
                        }
                    }
        }
        if (best != INT_MAX) labels[me] = best;
    }
    add_counter(ctr, tests);
}

// ======================================================================================================
// shared phase kernels
// ======================================================================================================
__global__ void __launch_bounds__(DB_THREADS) db_core_out_kernel(int n, const uint8_t* __restrict__ core, const int* __restrict__ sidx,
                                                                uint8_t* __restrict__ core_out) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) core_out[sidx[p]] = core[p] == 1;
}

__global__ void __launch_bounds__(DB_THREADS) db_core_in_kernel(int n, const uint8_t* __restrict__ core_in, const int* __restrict__ sidx,
                                                               uint8_t* __restrict__ core) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) core[p] = core_in[sidx[p]] ? 1 : (core[p] == 2 ? 2 : 0);
}

// single-GPU canonical numbering: the smallest core point of a component has key == its own index
__global__ void __launch_bounds__(DB_THREADS) db_rootflag_kernel(int n, const long long* __restrict__ comp_key, int* __restrict__ flags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flags[i] = comp_key[i] == (long long)i;
}

__global__ void __launch_bounds__(DB_THREADS) db_rank_labels_kernel(int n, const long long* __restrict__ comp_key, const int* __restrict__ rank,
                                                                   int32_t* __restrict__ labels) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long k = comp_key[i];
    labels[i] = k >= 0 ? rank[k] : -1;
}

__global__ void __launch_bounds__(DB_THREADS) db_relabel_kernel(int64_t n, const long long* __restrict__ keys, const long long* __restrict__ table_keys,
                                                               const int32_t* __restrict__ table_ids, int64_t m, int32_t* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long k = keys[i];
    int32_t id = -1;
    if (k >= 0 && m > 0) {
        int64_t lo = 0, hi = m;                                   // first entry >= k
        while (lo < hi) { int64_t mid = (lo + hi) >> 1; if (table_keys[mid] < k) lo = mid + 1; else hi = mid; }
        if (lo < m && table_keys[lo] == k) id = table_ids[lo];
    }
    out[i] = id;
}

template <typename T>
int scratch(rb_ctx* ctx, rb_slot slot, size_t count, T** out) {
    void* p;
    int rc = rb_scratch_get(ctx, slot, sizeof(T) * count, &p);
    *out = (T*)p;
    return rc;
}

// Host side: choose the grid. Tight cells when the times are integers and the bucket table fits the budget;
// otherwise cells at least eps wide, coarsened until the table fits.
int choose_grid(const float mn[4], const float mx[4], bool times_integer, int dim, int64_t n, double eps_space,
                float eps_time, int mode_opt, DbGrid* g, double* cell_out, double* wt_out) {
    double ext[3] = {0, 0, 0};
    for (int k = 0; k < 3; ++k) { g->lo[k] = 0; g->n[k] = 1; }
    for (int k = 0; k < dim; ++k) {
        g->lo[k] = mn[k];
        ext[k] = (double)mx[k] - (double)mn[k];
        if (!(ext[k] >= 0) || !isfinite(ext[k])) { rb_set_error("rb_stdbscan: non-finite coordinates"); return RB_ERR_ARG; }
    }
    double text = (double)mx[3] - (double)mn[3];
    if (!(text >= 0) || !isfinite(text)) { rb_set_error("rb_stdbscan: non-finite times"); return RB_ERR_ARG; }
    const double budget = fmin(fmax(16.0 * (double)n, 1048576.0), 134217728.0);
    double et = (double)eps_time;
    g->dim = dim;
    g->tmin = mn[3];
    g->tight = 0;
    g->R = 1;

    // ---- tight grid ---------------------------------------------------------------------------------
    if (mode_opt != 1 && times_integer && eps_space > 0 && et >= 0) {
        const double cell = eps_space * (1.0 - 1e-9) / sqrt((double)dim);
        double total = 1;
        for (int k = 0; k < dim; ++k) total *= floor(ext[k] / cell) + 1;
        const double nt = floor(text) + 1;
        total *= nt;
        if (total <= budget) {
            for (int k = 0; k < dim; ++k) g->n[k] = (int)(floor(ext[k] / cell) + 1);
            g->nt = (int)nt;
            g->inv_cell = 1.0 / cell;
            g->inv_wt = 1.0;
            g->tr = (int)fmin(floor(et), 1e6);
            g->R = 2;                                    // cell < eps <= 2 cells in every dimension (1-D included: a pair at
                                                         // cell < d <= eps can straddle a whole cell)
            g->tight = 1;
            *cell_out = cell;
            *wt_out = 1.0;
            return RB_OK;
        }
    }
    if (mode_opt == 2) { rb_set_error("rb_stdbscan: tight grid required (dbscan_mode=2) but not applicable"); return RB_ERR_ARG; }

    // ---- general grid ---------------------------------------------------------------------------------
    double max_ext = fmax(ext[0], fmax(ext[1], ext[2]));
    double cell = eps_space > 0 ? eps_space * (1.0 + 1e-7) : (max_ext > 0 ? max_ext / 1024.0 : 1.0);
    if (!(cell > 0) || !isfinite(cell)) cell = 1.0;
    double wt; int tr;
    if (!(et >= 0)) et = 0;                                 // negative eps_time: nothing matches anyway
    if (times_integer) {
        wt = 1.0;
        tr = (int)fmin(floor(et), 1e6);
    } else if (et > 0) {
        wt = et * (1.0 + 1e-6); tr = 1;
    } else {
        wt = text > 0 ? text / 256.0 : 1.0; tr = 0;         // equal times always share a bin
    }
    for (int iter = 0; iter < 200; ++iter) {
        double total = 1;
        for (int k = 0; k < dim; ++k) { double c = floor(ext[k] / cell) + 1; total *= c; }
        double nt = floor(text / wt) + 1;
        total *= nt;
        if (total <= budget) {
            for (int k = 0; k < dim; ++k) g->n[k] = (int)(floor(ext[k] / cell) + 1);
            g->nt = (int)nt;
            break;
        }
        // coarsen whichever axis family has more cells per search step
        double per_axis = 1;
        for (int k = 0; k < dim; ++k) per_axis = fmax(per_axis, floor(ext[k] / cell) + 1);
        if (nt / (2.0 * tr + 1.0) > per_axis / 3.0 && nt > 1) {
            wt *= 2.0;
            tr = (int)fmin(floor(et / wt) + 1, 1e6);
        } else {
            cell *= 2.0;
        }
        if (iter == 199) { rb_set_error("rb_stdbscan: could not fit a cell table"); return RB_ERR_ARG; }
    }
    g->inv_cell = 1.0 / cell;
    g->inv_wt = 1.0 / wt;
    g->tr = tr;
    *cell_out = cell;
    *wt_out = wt;
    return RB_OK;
}

}  // namespace

// ---- plan: everything the phases share, owned by the ctx ------------------------------------------------
struct rb_db_plan {
    bool valid = false;
    int dim = 0;
    int n = 0;
    DbGrid g;
    int64_t n_cells = 0;
    double eps2 = 0, cell = 0, wt = 0;
    float eps_t = 0;
    int min_samples = 0;
    int min_frames = 0;                          // > 0: PointCloudWorkF variant (extra core test + FIFO border rule)
    bool have_cores = false, have_components = false;
    // device arrays (scratch slots of the ctx)
    int *cell_start = nullptr, *sidx = nullptr, *scell = nullptr, *parent = nullptr, *flags = nullptr, *rank = nullptr, *slabel = nullptr;
    int *b_ncore = nullptr, *b_parent = nullptr, *b_label = nullptr, *core_start = nullptr, *cb_list = nullptr;
    int *cb_slot = nullptr, *cb_bbox = nullptr;
    long long *minkey = nullptr, *b_minkey = nullptr, *comp_key = nullptr;
    float *sx = nullptr, *sy = nullptr, *sz = nullptr, *st = nullptr;
    uint8_t* core = nullptr;
    int* d_misc = nullptr;                       // [0..15] bounds, then counters
    unsigned long long* d_ctr = nullptr;         // count, union, border tests; [3] low word = n_clusters
    int* d_ncb = nullptr;
};

void rb_db_plan_free(rb_ctx* ctx) {
    delete ctx->db_plan;
    ctx->db_plan = nullptr;
}

namespace {

Sorted sorted_view(const rb_db_plan& P) { return Sorted{P.sx, P.sy, P.sz, P.st, P.scell, P.cell_start}; }

template <int DIM>
int plan_build(rb_ctx* ctx, rb_db_plan& P, const DbPoints& pts, int64_t n64, double eps_space, float eps_time, int min_samples,
               cudaStream_t stream, const rb_stdbscan_hint* hint = nullptr) {
    const int n = (int)n64;
    const unsigned blocks = (unsigned)rb_div_up(n, DB_THREADS);
    P.valid = false;
    P.dim = DIM; P.n = n; P.eps2 = eps_space * eps_space; P.eps_t = eps_time; P.min_samples = min_samples;
    P.have_cores = P.have_components = false;
    P.min_frames = 0;

    // 1. bounds -> host
    RB_TRY(scratch(ctx, RB_S_MISC, 64, &P.d_misc));
    P.d_ctr = (unsigned long long*)(P.d_misc + 16);
    P.d_ncb = P.d_misc + 32;
    RB_CUDA(cudaMemsetAsync(P.d_ctr, 0, sizeof(unsigned long long) * 5, stream));     // [4] = "a point outside the hinted box"
    float mn[4], mx[4];
    bool times_integer;
    if (hint) {
        // the caller knows a box that contains every point and time (any superset is fine: the grid is only a
        // candidate filter) - no bounds pass, no sync
        for (int k = 0; k < 4; ++k) { mn[k] = hint->lo[k]; mx[k] = hint->hi[k]; }
        times_integer = hint->times_integer != 0;
    } else {
        RB_CUDA(rb_launch(ctx, db_bounds_init, dim3(1), dim3(32), 0, stream, P.d_misc));
        RB_LAUNCH_CHECK(ctx);
        const unsigned want_b = (unsigned)rb_div_up(n, DB_THREADS * 4);
        int bblocks = (int)(want_b < (unsigned)ctx->sm_count * 4 ? want_b : (unsigned)ctx->sm_count * 4);
        RB_CUDA(rb_launch(ctx, db_bounds_kernel, dim3(bblocks), dim3(DB_THREADS), 0, stream, pts, DIM, n64, P.d_misc));
        RB_LAUNCH_CHECK(ctx);
        int* h = (int*)ctx->pinned;
        RB_CUDA(cudaMemcpyAsync(h, P.d_misc, sizeof(int) * 9, cudaMemcpyDeviceToHost, stream));
        RB_CUDA(cudaStreamSynchronize(stream));
        for (int k = 0; k < 4; ++k) { mn[k] = ord2f(h[k]); mx[k] = ord2f(h[4 + k]); }
        times_integer = h[8] == 0;
    }

    // 2. grid
    RB_TRY(choose_grid(mn, mx, times_integer, DIM, n64, eps_space, eps_time, ctx->opt_dbscan_mode, &P.g, &P.cell, &P.wt));
    const DbGrid& g = P.g;
    P.n_cells = (int64_t)g.n[0] * g.n[1] * g.n[2] * g.nt;

    // 3. counting sort into the bucket table
    int *cell_id, *slot;
    RB_TRY(scratch(ctx, RB_S_CELL_ID, (size_t)n, &cell_id));
    RB_TRY(scratch(ctx, RB_S_CELL_FILL, (size_t)n, &slot));
    RB_TRY(scratch(ctx, RB_S_CELL_START, (size_t)P.n_cells + 1, &P.cell_start));
    RB_TRY(scratch(ctx, RB_S_SORT_IDX, (size_t)n * 2, &P.sidx));
    P.scell = P.sidx + n;
    RB_TRY(scratch(ctx, RB_S_SX, (size_t)n, &P.sx));
    RB_TRY(scratch(ctx, RB_S_SY, (size_t)n, &P.sy));
    RB_TRY(scratch(ctx, RB_S_SZ, (size_t)n, &P.sz));
    RB_TRY(scratch(ctx, RB_S_ST, (size_t)n, &P.st));
    RB_TRY(scratch(ctx, RB_S_CORE, (size_t)n, &P.core));
    RB_TRY(scratch(ctx, RB_S_PARENT, (size_t)n, &P.parent));
    RB_TRY(scratch(ctx, RB_S_MINORIG, (size_t)n, &P.minkey));
    RB_TRY(scratch(ctx, RB_S_FLAGS, (size_t)n + 1, &P.flags));
    RB_TRY(scratch(ctx, RB_S_RANK, (size_t)n + 1, &P.rank));
    RB_TRY(scratch(ctx, RB_S_SLABEL, (size_t)n, &P.slabel));
    RB_TRY(scratch(ctx, RB_S_COMP_KEY, (size_t)n, &P.comp_key));
    if (g.tight) {
        RB_TRY(scratch(ctx, RB_S_B_NCORE, (size_t)P.n_cells + 1, &P.b_ncore));
        RB_TRY(scratch(ctx, RB_S_B_PARENT, (size_t)P.n_cells, &P.b_parent));
        RB_TRY(scratch(ctx, RB_S_B_LABEL, (size_t)P.n_cells, &P.b_label));
        RB_TRY(scratch(ctx, RB_S_B_MINKEY, (size_t)P.n_cells, &P.b_minkey));
        RB_TRY(scratch(ctx, RB_S_CORE_START, (size_t)P.n_cells + 1, &P.core_start));
        RB_TRY(scratch(ctx, RB_S_CB_LIST, (size_t)(P.n_cells < n ? P.n_cells : n) * 7 + 8, &P.cb_list));
        P.cb_bbox = P.cb_list + (size_t)(P.n_cells < n ? P.n_cells : n) + 1;
        P.cb_slot = P.b_label;                   // the label array is free until the assign phase
    }
    RB_CUDA(cudaMemsetAsync(P.cell_start, 0, sizeof(int) * ((size_t)P.n_cells + 1), stream));
    RB_CUDA(rb_launch(ctx, db_cell_kernel, dim3(blocks), dim3(DB_THREADS), 0, stream, pts, g, n64, cell_id, slot, P.cell_start, hint ? (int*)(P.d_ctr + 4) : nullptr));
    RB_LAUNCH_CHECK(ctx);
    RB_TRY(rb_exclusive_scan_i32(ctx, P.cell_start, P.cell_start, P.n_cells + 1, nullptr, stream));
    RB_CUDA(rb_launch(ctx, db_scatter_kernel, dim3(blocks), dim3(DB_THREADS), 0, stream, pts, DIM, n64, cell_id, slot, P.cell_start, P.sidx, P.scell, P.sx, P.sy, P.sz,
                                                        P.st));
    RB_LAUNCH_CHECK(ctx);
    P.valid = true;
    return RB_OK;
}

template <int DIM>
int phase_cores(rb_ctx* ctx, rb_db_plan& P, cudaStream_t stream) {
    const unsigned blocks = (unsigned)rb_div_up(P.n, DB_THREADS);
    const Sorted s = sorted_view(P);
    const bool wf = P.min_frames > 0;
    if (P.g.tight && wf) RB_CUDA(rb_launch(ctx, dbt_count_kernel<DIM, true>, dim3(blocks), dim3(DB_THREADS), 0, stream, s, P.g, P.n, P.eps2, P.min_samples, P.min_frames, P.core, P.d_ctr + 0));
    else if (P.g.tight) RB_CUDA(rb_launch(ctx, dbt_count_kernel<DIM, false>, dim3(blocks), dim3(DB_THREADS), 0, stream, s, P.g, P.n, P.eps2, P.min_samples, 0, P.core, P.d_ctr + 0));
    else if (wf) RB_CUDA(rb_launch(ctx, dbg_count_kernel<DIM, true>, dim3(blocks), dim3(DB_THREADS), 0, stream, s, P.g, P.n, P.eps2, P.eps_t, P.min_samples, P.min_frames, P.core, P.d_ctr + 0));
    else RB_CUDA(rb_launch(ctx, dbg_count_kernel<DIM, false>, dim3(blocks), dim3(DB_THREADS), 0, stream, s, P.g, P.n, P.eps2, P.eps_t, P.min_samples, 0, P.core, P.d_ctr + 0));
    RB_LAUNCH_CHECK(ctx);
    P.have_cores = true;
    P.have_components = false;
    return RB_OK;
}

template <int DIM>
int phase_components(rb_ctx* ctx, rb_db_plan& P, const long long* gidx, cudaStream_t stream) {
    const int n = P.n;
    const unsigned blocks = (unsigned)rb_div_up(n, DB_THREADS);
    const Sorted s = sorted_view(P);
    if (P.g.tight) {
        const unsigned cblocks = (unsigned)rb_div_up(P.n_cells + 1, DB_THREADS);
        RB_CUDA(rb_launch(ctx, dbt_bucket_init_kernel, dim3(cblocks), dim3(DB_THREADS), 0, stream, P.n_cells, P.b_ncore, P.b_parent, P.b_minkey, P.d_ncb));
        RB_LAUNCH_CHECK(ctx);
        RB_CUDA(rb_launch(ctx, dbt_bucket_stats_kernel, dim3(blocks), dim3(DB_THREADS), 0, stream, n, P.core, P.scell, P.sidx, gidx, P.b_ncore, P.b_minkey));
        RB_LAUNCH_CHECK(ctx);
        const unsigned lblocks = (unsigned)rb_div_up(P.n_cells, (int64_t)DB_THREADS * LIST_PER_THREAD);
        RB_CUDA(rb_launch(ctx, dbt_bucket_list_kernel, dim3(lblocks), dim3(DB_THREADS), 0, stream, P.n_cells, P.b_ncore, P.cb_list, P.d_ncb, P.cb_slot, P.cb_bbox, P.b_parent));
        RB_LAUNCH_CHECK(ctx);
        RB_CUDA(rb_launch(ctx, dbt_bucket_bbox_kernel<DIM>, dim3(blocks), dim3(DB_THREADS), 0, stream, s, n, P.core, P.cb_slot, P.cb_bbox));
        RB_LAUNCH_CHECK(ctx);
        RB_TRY(rb_exclusive_scan_i32(ctx, P.b_ncore, P.core_start, P.n_cells + 1, nullptr, stream));
        const int64_t max_buckets = P.n_cells < n ? P.n_cells : n;
        const int64_t want = rb_div_up(max_buckets, DB_THREADS);         // one lane per core bucket
        const unsigned ublocks = (unsigned)(want < (int64_t)ctx->sm_count * 16 ? (want > 0 ? want : 1) : (int64_t)ctx->sm_count * 16);
        const int64_t want2 = rb_div_up(max_buckets, DB_THREADS);
        const unsigned mblocks = (unsigned)(want2 < (int64_t)ctx->sm_count * 8 ? (want2 > 0 ? want2 : 1) : (int64_t)ctx->sm_count * 8);
        RB_CUDA(rb_launch(ctx, dbt_link_time_kernel, dim3(mblocks), dim3(DB_THREADS), 0, stream, P.g, P.cb_list, P.d_ncb, P.b_ncore, P.b_parent));
        RB_LAUNCH_CHECK(ctx);
        RB_CUDA(rb_launch(ctx, dbt_flatten_kernel, dim3(mblocks), dim3(DB_THREADS), 0, stream, P.cb_list, P.d_ncb, P.b_parent));
        RB_LAUNCH_CHECK(ctx);
        RB_CUDA(rb_launch(ctx, dbt_union_kernel<DIM>, dim3(ublocks), dim3(DB_THREADS), 0, stream, s, P.g, P.cb_list, P.d_ncb, P.core, P.b_ncore, P.b_parent, P.cb_slot,
                                                                  P.cb_bbox, P.eps2, P.d_ctr + 1));
        RB_LAUNCH_CHECK(ctx);
        RB_CUDA(rb_launch(ctx, dbt_compmin_kernel, dim3(mblocks), dim3(DB_THREADS), 0, stream, P.cb_list, P.d_ncb, P.b_parent, P.b_minkey));
        RB_LAUNCH_CHECK(ctx);
        RB_CUDA(rb_launch(ctx, dbt_keyout_kernel, dim3(blocks), dim3(DB_THREADS), 0, stream, n, P.core, P.scell, P.sidx, P.b_parent, P.b_minkey, P.comp_key));
        RB_LAUNCH_CHECK(ctx);
    } else {
        RB_CUDA(rb_launch(ctx, dbg_init_kernel, dim3(blocks), dim3(DB_THREADS), 0, stream, n, P.parent, P.minkey));
        RB_LAUNCH_CHECK(ctx);
        RB_CUDA(rb_launch(ctx, dbg_union_kernel<DIM>, dim3(blocks), dim3(DB_THREADS), 0, stream, s, P.g, n, P.eps2, P.eps_t, P.core, P.parent, P.d_ctr + 1));
        RB_LAUNCH_CHECK(ctx);
        RB_CUDA(rb_launch(ctx, dbg_minkey_kernel, dim3(blocks), dim3(DB_THREADS), 0, stream, n, P.core, P.parent, P.sidx, gidx, P.minkey));
        RB_LAUNCH_CHECK(ctx);
        RB_CUDA(rb_launch(ctx, dbg_keyout_kernel, dim3(blocks), dim3(DB_THREADS), 0, stream, n, P.core, P.parent, P.sidx, P.minkey, P.comp_key));
        RB_LAUNCH_CHECK(ctx);
    }
    P.have_components = true;
    return RB_OK;
}

template <int DIM>
int phase_assign(rb_ctx* ctx, rb_db_plan& P, const int32_t* core_label, int32_t* labels, cudaStream_t stream) {
    const int n = P.n;
    const unsigned blocks = (unsigned)rb_div_up(n, DB_THREADS);
    const Sorted s = sorted_view(P);
    // labels of the core points and of the certain noise, bucket labels, list of the border candidates (P.rank is free here)
    int* open_list = P.rank;
    int* n_open = P.d_misc + 34;
    RB_CUDA(cudaMemsetAsync(n_open, 0, sizeof(int), stream));
    RB_CUDA(rb_launch(ctx, db_gather_labels_kernel, dim3(blocks), dim3(DB_THREADS), 0, stream, n, P.core, P.sidx, P.scell, core_label, P.slabel,
                      P.g.tight ? P.b_label : nullptr, labels, open_list, n_open));
    RB_LAUNCH_CHECK(ctx);
    const bool wf = P.min_frames > 0;
    const unsigned wblocks = (unsigned)(blocks < (unsigned)ctx->sm_count * 8 ? blocks : (unsigned)ctx->sm_count * 8);
    if (P.g.tight && wf)
        RB_CUDA(rb_launch(ctx, dbt_border_kernel<DIM, true>, dim3(wblocks), dim3(DB_THREADS), 0, stream, s, P.g, P.eps2, P.core, P.sidx, open_list, n_open,
                          P.b_ncore, P.core_start, P.b_label, P.b_parent, P.b_minkey, labels, P.d_ctr + 2));
    else if (P.g.tight)
        RB_CUDA(rb_launch(ctx, dbt_border_kernel<DIM, false>, dim3(wblocks), dim3(DB_THREADS), 0, stream, s, P.g, P.eps2, P.core, P.sidx, open_list, n_open,
                          P.b_ncore, P.core_start, P.b_label, P.b_parent, P.b_minkey, labels, P.d_ctr + 2));
    else if (wf)
        RB_CUDA(rb_launch(ctx, dbg_border_kernel<DIM, true>, dim3(wblocks), dim3(DB_THREADS), 0, stream, s, P.g, P.eps2, P.eps_t, P.core, P.slabel, P.sidx,
                          P.comp_key, open_list, n_open, labels, P.d_ctr + 2));
    else
        RB_CUDA(rb_launch(ctx, dbg_border_kernel<DIM, false>, dim3(wblocks), dim3(DB_THREADS), 0, stream, s, P.g, P.eps2, P.eps_t, P.core, P.slabel, P.sidx,
                          P.comp_key, open_list, n_open, labels, P.d_ctr + 2));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}

#define DB_DISPATCH(P, call)                                  \
    ((P).dim == 3 ? call<3> : (P).dim == 2 ? call<2> : call<1>)

int fetch_stats(rb_ctx* ctx, rb_db_plan& P, int64_t* n_clusters, cudaStream_t stream) {
    unsigned long long* hc = (unsigned long long*)ctx->pinned;
    RB_CUDA(cudaMemcpyAsync(hc, P.d_ctr, sizeof(unsigned long long) * 5, cudaMemcpyDeviceToHost, stream));
    RB_CUDA(cudaStreamSynchronize(stream));
    if (hc[4] != 0) {
        rb_set_error("ST-DBSCAN: the hinted box does not contain every point / time (rb_stdbscan_hint); the result is invalid");
        return RB_ERR_ARG;
    }
    rb_dbscan_stats& stt = ctx->last_stats;
    memset(&stt, 0, sizeof stt);
    stt.n_points = P.n;
    stt.n_cells = P.n_cells;
    stt.n_clusters = (int64_t)(int)(hc[3] & 0xffffffffu);
    stt.n_core = -1;
    stt.pair_tests_count = (int64_t)hc[0];
    stt.pair_tests_union = (int64_t)hc[1];
    stt.pair_tests_border = (int64_t)hc[2];
    stt.cell_size = P.cell;
    stt.time_bin = P.wt;
    stt.dims[0] = P.g.n[0]; stt.dims[1] = P.g.n[1]; stt.dims[2] = P.g.n[2]; stt.dims[3] = P.g.nt;
    stt.time_radius = P.g.tr;
    stt.tight = P.g.tight;
    if (n_clusters) *n_clusters = stt.n_clusters;
    return RB_OK;
}

}  // namespace

int rb_stdbscan_plan_hinted(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                            const float* times, int64_t n, double eps_space, float eps_time, int min_samples,
                            const rb_stdbscan_hint* hint, void* stream_);

extern "C" int rb_stdbscan_plan(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                                const float* times, int64_t n, double eps_space, float eps_time, int min_samples,
                                void* stream_) {
    return rb_stdbscan_plan_hinted(ctx, x, y, z, stride, times, n, eps_space, eps_time, min_samples, nullptr, stream_);
}

extern "C" int rb_stdbscan_plan_hinted(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                                       const float* times, int64_t n, double eps_space, float eps_time, int min_samples,
                                       const rb_stdbscan_hint* hint, void* stream_) {
    RB_REQUIRE(ctx, "ctx is NULL");
    RB_REQUIRE(n > 0 && n < ((int64_t)1 << 31) - 1, "point count out of range (1 .. 2^31-2)");
    RB_REQUIRE(x && times, "NULL argument");
    RB_REQUIRE(stride >= 1, "stride must be >= 1");
    RB_REQUIRE(!(z && !y), "z without y");
    RB_REQUIRE(eps_space >= 0 && isfinite(eps_space), "eps_space must be finite and >= 0");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!ctx->db_plan) ctx->db_plan = new rb_db_plan();
    rb_db_plan& P = *ctx->db_plan;
    DbPoints pts{x, y, z, stride, times};
    if (z) return plan_build<3>(ctx, P, pts, n, eps_space, eps_time, min_samples, stream, hint);
    if (y) return plan_build<2>(ctx, P, pts, n, eps_space, eps_time, min_samples, stream, hint);
    return plan_build<1>(ctx, P, pts, n, eps_space, eps_time, min_samples, stream, hint);
}

extern "C" int rb_stdbscan_cores(rb_ctx* ctx, uint8_t* core_out, void* stream_) {
    RB_REQUIRE(ctx && ctx->db_plan && ctx->db_plan->valid, "rb_stdbscan_cores: no plan (call rb_stdbscan_plan first)");
    cudaStream_t stream = (cudaStream_t)stream_;
    rb_db_plan& P = *ctx->db_plan;
    RB_TRY(DB_DISPATCH(P, phase_cores)(ctx, P, stream));
    if (core_out) {
        RB_CUDA(rb_launch(ctx, db_core_out_kernel, dim3((unsigned)rb_div_up(P.n, DB_THREADS)), dim3(DB_THREADS), 0, stream, P.n, P.core, P.sidx, core_out));
        RB_LAUNCH_CHECK(ctx);
    }
    return RB_OK;
}

extern "C" int rb_stdbscan_set_cores(rb_ctx* ctx, const uint8_t* core_in, void* stream_) {
    RB_REQUIRE(ctx && ctx->db_plan && ctx->db_plan->valid && ctx->db_plan->have_cores, "rb_stdbscan_set_cores: run rb_stdbscan_cores first");
    RB_REQUIRE(core_in, "core_in is NULL");
    cudaStream_t stream = (cudaStream_t)stream_;
    rb_db_plan& P = *ctx->db_plan;
    RB_CUDA(rb_launch(ctx, db_core_in_kernel, dim3((unsigned)rb_div_up(P.n, DB_THREADS)), dim3(DB_THREADS), 0, stream, P.n, core_in, P.sidx, P.core));
    RB_LAUNCH_CHECK(ctx);
    P.have_components = false;
    return RB_OK;
}

// rb_stdbscan_set_cores straight after a plan, without counting neighbours first: for a caller that already holds the
// exact core flag of every point of the plan (recording.cu). Without the count phase no point is known to have no
// neighbour at all (core state 2, which set_cores keeps): every non-core point stays a border candidate.
int rb_stdbscan_set_cores_planned(rb_ctx* ctx, const uint8_t* core_in, void* stream_) {
    RB_REQUIRE(ctx && ctx->db_plan && ctx->db_plan->valid, "rb_stdbscan_set_cores_planned: no plan");
    RB_CUDA(cudaMemsetAsync(ctx->db_plan->core, 0, (size_t)ctx->db_plan->n, (cudaStream_t)stream_));
    ctx->db_plan->have_cores = true;
    return rb_stdbscan_set_cores(ctx, core_in, stream_);
}

// device word the last plan raises when a point or time lies outside its hint box (valid until the next plan)
int rb_stdbscan_hint_flag(rb_ctx* ctx, const unsigned long long** flag) {
    RB_REQUIRE(ctx && ctx->db_plan && ctx->db_plan->valid && flag, "rb_stdbscan_hint_flag: no plan");
    *flag = ctx->db_plan->d_ctr + 4;
    return RB_OK;
}

extern "C" int rb_stdbscan_components(rb_ctx* ctx, const int64_t* global_index, int64_t* comp_key, void* stream_) {
    RB_REQUIRE(ctx && ctx->db_plan && ctx->db_plan->valid && ctx->db_plan->have_cores, "rb_stdbscan_components: run rb_stdbscan_cores first");
    cudaStream_t stream = (cudaStream_t)stream_;
    rb_db_plan& P = *ctx->db_plan;
    RB_TRY(DB_DISPATCH(P, phase_components)(ctx, P, (const long long*)global_index, stream));
    if (comp_key) RB_CUDA(cudaMemcpyAsync(comp_key, P.comp_key, sizeof(int64_t) * (size_t)P.n, cudaMemcpyDeviceToDevice, stream));
    return RB_OK;
}

extern "C" int rb_stdbscan_assign(rb_ctx* ctx, const int32_t* core_label, int32_t* labels, void* stream_) {
    RB_REQUIRE(ctx && ctx->db_plan && ctx->db_plan->valid && ctx->db_plan->have_cores, "rb_stdbscan_assign: run rb_stdbscan_cores first");
    RB_REQUIRE(core_label && labels, "NULL argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    rb_db_plan& P = *ctx->db_plan;
    return DB_DISPATCH(P, phase_assign)(ctx, P, core_label, labels, stream);
}

extern "C" int rb_relabel(rb_ctx* ctx, const int64_t* keys, int64_t n, const int64_t* table_keys, const int32_t* table_ids,
                          int64_t m, int32_t* out, void* stream_) {
    RB_REQUIRE(ctx, "ctx is NULL");
    RB_REQUIRE(n >= 0 && m >= 0, "negative size");
    if (n == 0) return RB_OK;
    RB_REQUIRE(keys && out && (m == 0 || (table_keys && table_ids)), "NULL argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    RB_CUDA(rb_launch(ctx, db_relabel_kernel, dim3((unsigned)rb_div_up(n, DB_THREADS)), dim3(DB_THREADS), 0, stream, n, (const long long*)keys, (const long long*)table_keys,
                                                                                    table_ids, m, out));
    RB_LAUNCH_CHECK(ctx);
    return RB_OK;
}

// everything of rb_stdbscan except reading the counters back: with a hint nothing here syncs
int rb_stdbscan_enqueue(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride, const float* times,
                        int64_t n, double eps_space, float eps_time, int min_samples, int32_t* labels, uint8_t* core,
                        const rb_stdbscan_hint* hint, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    RB_TRY(rb_stdbscan_plan_hinted(ctx, x, y, z, stride, times, n, eps_space, eps_time, min_samples, hint, stream_));
    rb_db_plan& P = *ctx->db_plan;
    RB_TRY(rb_stdbscan_cores(ctx, core, stream_));
    RB_TRY(rb_stdbscan_components(ctx, nullptr, nullptr, stream_));
    // canonical numbering: rank of every component's smallest core index
    const unsigned blocks = (unsigned)rb_div_up(P.n, DB_THREADS);
    RB_CUDA(rb_launch(ctx, db_rootflag_kernel, dim3(blocks), dim3(DB_THREADS), 0, stream, P.n, P.comp_key, P.flags));
    RB_LAUNCH_CHECK(ctx);
    int* d_total = (int*)(P.d_ctr + 3);
    RB_TRY(rb_exclusive_scan_i32(ctx, P.flags, P.rank, P.n, d_total, stream));
    RB_CUDA(rb_launch(ctx, db_rank_labels_kernel, dim3(blocks), dim3(DB_THREADS), 0, stream, P.n, P.comp_key, P.rank, labels));
    RB_LAUNCH_CHECK(ctx);
    return rb_stdbscan_assign(ctx, labels, labels, stream_);         // in place: core labels are copied before any write
}

int rb_stdbscan_fetch_stats(rb_ctx* ctx, int64_t* n_clusters, void* stream_) {
    RB_REQUIRE(ctx && ctx->db_plan && ctx->db_plan->valid, "no ST-DBSCAN plan");
    return fetch_stats(ctx, *ctx->db_plan, n_clusters, (cudaStream_t)stream_);
}

extern "C" int rb_stdbscan(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                           const float* times, int64_t n, double eps_space, float eps_time, int min_samples,
                           int32_t* labels, uint8_t* core, int64_t* n_clusters, void* stream_) {
    RB_REQUIRE(ctx, "ctx is NULL");
    RB_REQUIRE(n >= 0 && n < ((int64_t)1 << 31) - 1, "point count out of range");
    if (n_clusters) *n_clusters = 0;
    if (n == 0) return RB_OK;
    RB_REQUIRE(labels, "labels is NULL");
    RB_TRY(rb_stdbscan_enqueue(ctx, x, y, z, stride, times, n, eps_space, eps_time, min_samples, labels, core, nullptr, stream_));
    return rb_stdbscan_fetch_stats(ctx, n_clusters, stream_);
}

extern "C" int rb_stdbscan_wf(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                              const float* times, int64_t n, double eps_space, float eps_time, int min_samples, int min_frames,
                              int32_t* labels, uint8_t* core, int64_t* n_clusters, void* stream_) {
    RB_REQUIRE(ctx, "ctx is NULL");
    RB_REQUIRE(n >= 0 && n < ((int64_t)1 << 31) - 1, "point count out of range");
    RB_REQUIRE(min_frames >= 1, "min_frames must be >= 1");
    RB_REQUIRE(!(eps_time > 30.f), "rb_stdbscan_wf supports eps_time <= 30 (the frame set of a neighbourhood is a 64-bit mask)");
    if (n_clusters) *n_clusters = 0;
    if (n == 0) return RB_OK;
    RB_REQUIRE(labels, "labels is NULL");
    cudaStream_t stream = (cudaStream_t)stream_;
    RB_TRY(rb_stdbscan_plan(ctx, x, y, z, stride, times, n, eps_space, eps_time, min_samples, stream_));
    rb_db_plan& P = *ctx->db_plan;
    P.min_frames = min_frames;                                  // switches the core test and the border rule
    RB_TRY(rb_stdbscan_cores(ctx, core, stream_));
    RB_TRY(rb_stdbscan_components(ctx, nullptr, nullptr, stream_));
    const unsigned blocks = (unsigned)rb_div_up(P.n, DB_THREADS);
    RB_CUDA(rb_launch(ctx, db_rootflag_kernel, dim3(blocks), dim3(DB_THREADS), 0, stream, P.n, P.comp_key, P.flags));
    RB_LAUNCH_CHECK(ctx);
    int* d_total = (int*)(P.d_ctr + 3);
    RB_TRY(rb_exclusive_scan_i32(ctx, P.flags, P.rank, P.n, d_total, stream));
    RB_CUDA(rb_launch(ctx, db_rank_labels_kernel, dim3(blocks), dim3(DB_THREADS), 0, stream, P.n, P.comp_key, P.rank, labels));
    RB_LAUNCH_CHECK(ctx);
    RB_TRY(rb_stdbscan_assign(ctx, labels, labels, stream_));
    return rb_stdbscan_fetch_stats(ctx, n_clusters, stream_);
}

// After phases driven by the caller (rb_stdbscan_plan_hinted ... rb_stdbscan_assign): syncs the stream, refreshes the
// counters of rb_stdbscan_last_stats and fails if the plan's hint box did not contain every point and time.
extern "C" int rb_stdbscan_check(rb_ctx* ctx, void* stream_) {
    RB_REQUIRE(ctx && ctx->db_plan && ctx->db_plan->valid, "rb_stdbscan_check: no plan");
    return fetch_stats(ctx, *ctx->db_plan, nullptr, (cudaStream_t)stream_);
}

extern "C" int rb_stdbscan_last_stats(rb_ctx* ctx, rb_dbscan_stats* out) {
    RB_REQUIRE(ctx && out, "NULL argument");
    *out = ctx->last_stats;
    return RB_OK;
}
