/*
 * radarb200 — C ABI of the B200-native per-frame detection hot path
 * (spoke-to-point -> land/stationary persistence filter -> temporal ST-DBSCAN).
 *
 * The reference (SamuelCancilla2/radar-point-cloud-tracking) has no FFI/plugin interface: its
 * boundary for this path is the Python function surface of
 *   PointCloudWork/4_temporal_object_tracker.py            ("T4")
 *   PointCloudWork/3_stdbscan_point_clouds.py               ("T3")
 *   PointCloudWork/5_gain_fusion_ply_builder.py             ("T5")
 *   radar-pipeline/src/radar_pipeline/{core,processors}     ("PKG")
 * Each entry point below names the reference lines it replaces; INTEGRATION.md shows the ctypes
 * binding a maintainer of the reference would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only. Every data pointer is a DEVICE pointer unless
 *     the parameter comment says "host". The caller owns all buffers; the library owns only the
 *     scratch inside rb_ctx (grown on demand, freed by rb_destroy).
 *   - All work is enqueued on the caller's stream (`stream` is a cudaStream_t passed as void*;
 *     NULL = legacy default stream). A call synchronises that stream only where its comment says
 *     "syncs" (a count or a bound has to reach the host).
 *   - Return value: 0 = ok, negative = error (rb_last_error() gives the text). Nothing throws.
 *   - One rb_ctx per device and per host thread; a ctx is not thread safe.
 *   - There is no CPU fallback: without a CUDA device rb_create fails.
 */
#ifndef RADARB200_H
#define RADARB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RB_OK 0
#define RB_ERR_CUDA (-1)        /* a CUDA runtime call failed                     */
#define RB_ERR_ARG (-2)         /* bad argument                                   */
#define RB_ERR_CAPACITY (-3)    /* caller-provided output capacity too small      */
#define RB_ERR_NOMEM (-4)       /* scratch allocation failed                      */
#define RB_ERR_NCCL (-5)        /* collective layer (NCCL) failure                */

typedef struct rb_ctx rb_ctx;

/* ---- context ----------------------------------------------------------------------------- */
int rb_version(void);                               /* ABI version, currently 1 */
const char* rb_last_error(void);                    /* thread-local text of the last failure */
int rb_create(int device, rb_ctx** out);            /* fails without a usable CUDA device */
void rb_destroy(rb_ctx* ctx);
int rb_device_info(rb_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, int64_t* l2_bytes);
/* Scratch grows on demand; a buffer that was outgrown is kept until rb_destroy, because freeing device memory synchronises
 * the whole device. rb_trim frees those buffers: call it only when no work of this context is in flight and no collective of
 * the process waits for a peer (rb_detect_block does so itself after its final read-back). */
int rb_trim(rb_ctx* ctx);

/* ---- a1 + a2: spoke-to-point with threshold, stride and multi-gain concat fusion ------------
 * Replaces the numeric part of load_radar_csv (T4:200-232; twins PKG/core/transforms.py:13-79,
 * T5:97-121) for a whole batch of sweeps in ONE launch, and the concatenation of build_frame
 * (T4:322-344): sweeps are laid out frame-major / ascending-gain-minor, so the output of a frame
 * is exactly np.concatenate over its gains.
 *
 *   echo       [W][S][E] float32, row major (W = frames x gains sweeps)
 *   cos_tab    [W][S]  float32  np.cos(deg2rad(Angle.f32*360/8196)) computed by the HOST with
 *   sin_tab    [W][S]  float32  numpy (bit-exactness of trig is a host contract, see DESIGN.md)
 *   range_res  [W][S]  float32  Scale.f32 / E                                   (T4:213)
 *   ranges     [W][S][E] float32, OPTIONAL (NULL = use range_res*j): explicit range of every cell,
 *              for callers that hold a RadarSweep.ranges array (PKG/core/transforms.py:63); only
 *              the cells that are written are read.
 *   sweep_gain [W]     int32    gain label written for every point of the sweep (T4:333)
 * For sweep w, element (s, j) survives when echo > threshold (strict, T4:221); survivors are
 * ranked in row-major order and every `stride`-th one (rank % stride == 0, T4:227-230) is written:
 *   x = fl32(fl32(range_res*j) * cos), y = fl32(fl32(range_res*j) * sin), intensity = echo.
 * Outputs (capacity `cap` points each): x, y, inten float32; gain int32;
 *   sweep_base [W+1] int64: output offset of every sweep; sweep_base[W] = total points.
 * If the total exceeds `cap`, points beyond `cap` are dropped (never written) and sweep_base
 * still holds the true sizes, so the caller can detect it after its own sync. Does not sync.
 */
int rb_spoke_to_points(rb_ctx* ctx, const float* echo, const float* cos_tab, const float* sin_tab,
                       const float* range_res, const float* ranges, const int32_t* sweep_gain,
                       int64_t n_sweeps, int n_spokes, int n_bins,
                       float threshold, int stride,
                       float* x, float* y, float* inten, int32_t* gain, int64_t cap,
                       int64_t* sweep_base, void* stream);

/* The same with uint8 echoes (what the radar delivers: 0..255, a quarter of the bytes to move): survives when
 * (float)echo > threshold, intensity = (float)echo. Results are identical to rb_spoke_to_points on the same values
 * converted to float32. The TMA-staged kernel needs S*E % 16 == 0 and a 16-byte aligned pointer. */
int rb_spoke_to_points_u8(rb_ctx* ctx, const uint8_t* echo, const float* cos_tab, const float* sin_tab,
                          const float* range_res, const float* ranges, const int32_t* sweep_gain,
                          int64_t n_sweeps, int n_spokes, int n_bins,
                          float threshold, int stride,
                          float* x, float* y, float* inten, int32_t* gain, int64_t cap,
                          int64_t* sweep_base, void* stream);

/* polar_to_cartesian on a full grid (PKG/core/transforms.py:13-34): x = ranges*cos[:,None],
 * y = ranges*sin[:,None]; ranges/x/y float32 [n_rows][n_cols], cos/sin float32 [n_rows] from the
 * host's numpy. No sync. */
int rb_polar_to_cartesian(rb_ctx* ctx, const float* ranges, const float* cos_tab, const float* sin_tab,
                          int64_t n_rows, int n_cols, float* x, float* y, void* stream);

/* frame_off[f] = sweep_base[f*gains_per_frame], f = 0..n_frames (int64, device). No sync. */
int rb_frame_offsets(rb_ctx* ctx, const int64_t* sweep_base, int64_t n_frames, int gains_per_frame,
                     int64_t* frame_off, void* stream);

/* times[i] = frame_ids[f] for frame_off[f] <= i < frame_off[f+1]  (T4:460,467: float32 frame
 * ids per point). frame_ids float32[n_frames] device. No sync. */
int rb_expand_frame_times(rb_ctx* ctx, const int64_t* frame_off, const float* frame_ids,
                          int64_t n_frames, int64_t n_points, float* times, void* stream);

/* ---- a3: max fusion on a grid (T5:222-273 fuse_gains_max) --------------------------------------
 * Pools n points on a grid anchored at (x_min, y_min): cell = trunc((v - v_min)/res) in float32
 * (T5:258-259), keeps the max intensity per cell (T5:263) and emits occupied cells in y-major
 * order (T5:267): cell_ix, cell_iy int32 and max intensity float32, capacity cap_cells.
 * x_min / y_min / nx / ny are the caller's float32 values (T5:251-256). n_cells_out: host
 * int64. Runs on the kernels of rb_fuse_max_frames (one frame, the caller's grid). Syncs. */
int rb_fuse_max(rb_ctx* ctx, const float* x, const float* y, const float* inten, int64_t n,
                float x_min, float y_min, float resolution, int nx, int ny,
                int32_t* cell_ix, int32_t* cell_iy, float* cell_max, int64_t cap_cells,
                int64_t* n_cells_out, void* stream);

/* Max fusion of many frames per call: for every frame f (points [frame_off[f], frame_off[f+1]) of x, y, inten; frame_off
 * int64[F+1] device, from 0 to n), exactly what fuse_gains_max returns for that frame's points:
 *   bounds = the float32 min / max of the frame's points, nx = int(ceil((x_max - x_min) / res)) + 1 and likewise ny, and
 *   cell = trunc((v - v_min) / res), all in float32 with res = (float)resolution (numpy >= 2, T5:251-259); max intensity
 *   per cell starting from 0 (T5:262-263); cells > 0 in y-major order (T5:267) with float64 centres
 *   x_min + ix * resolution + resolution / 2 evaluated left to right with the full double resolution (T5:269-270).
 * Outputs (device): cell_x, cell_y float64 and cell_max float32 with capacity cap_cells (n always suffices: a frame has at
 * most one cell per point); cell_off int64[F+1] delimits the frames. n_cells_out: host int64, the total.
 * A frame's grid must have fewer than 2^30 cells (RB_ERR_ARG naming the frame otherwise). Frames are pooled in groups of
 * consecutive frames whose grids fit a scratch bound together (2^28 cells, rb_set_option "fuse_group_cells"; a larger
 * frame is a group alone). RB_ERR_ARG before anything is enqueued for a resolution that is not finite and > 0, F < 0,
 * or NULL pointers. Syncs twice, whatever F: grid sizes, then the total. */
int rb_fuse_max_frames(rb_ctx* ctx, const float* x, const float* y, const float* inten, int64_t n,
                       const int64_t* frame_off, int64_t n_frames, double resolution,
                       double* cell_x, double* cell_y, float* cell_max, int64_t cap_cells,
                       int64_t* cell_off, int64_t* n_cells_out, void* stream);

/* HOST function: rb_fuse_max_frames' grouping. cells[F] = grid cells of each frame; consecutive frames join a group while
 * their cells add up to at most max_cells (a frame above it is a group alone). Writes the group cuts (frame indices,
 * cuts[0] = 0 ... cuts[K] = F; at most cap entries) and returns K, or a negative RB_ERR_* for bad arguments. */
int64_t rb_fuse_plan_groups(const int64_t* cells, int64_t n_frames, int64_t max_cells, int64_t* cuts, int64_t cap);

/* ---- a4-a6: land / stationary persistence filter --------------------------------------------- */
/* Global bounds (T4:365-369): out4 = device float32 {x_min, x_max, y_min, y_max}. No sync. */
int rb_bounds(rb_ctx* ctx, const float* x, const float* y, int64_t n, float* out4, void* stream);
/* Same over the first min(*n_dev, n_max) points, the count still being on the device (e.g. sweep_base[W] of
 * rb_spoke_to_points): lets a caller enqueue spoke-to-point + bounds and read count and bounds back with ONE sync. */
int rb_bounds_counted(rb_ctx* ctx, const float* x, const float* y, const int64_t* n_dev, int64_t n_max, float* out4,
                      void* stream);

/* build_occupancy_grid accumulation (T4:378-389): for every point
 *   ix = clip(searchsorted_right(x_edges, (double)x) - 1, 0, n_x_edges - 2)      (T4:384)
 *   count[ix][iy] += 1 (int32);  isum[ix][iy] += intensity (float64)            (T4:388-389)
 * x_edges / y_edges are the float64 np.arange edges computed on the host (T4:372-373) and copied
 * to the device. count/isum must be zeroed by the caller; the call accumulates. No sync. Exact for integer-valued
 * intensities, checked on the device - see rb_land_accumulate_status below. */
int rb_land_accumulate(rb_ctx* ctx, const float* x, const float* y, const float* inten, int64_t n,
                       const double* x_edges, int n_x_edges, const double* y_edges, int n_y_edges,
                       int32_t* count, double* isum, void* stream);

/* rb_land_accumulate's float64 sums equal np.add.at's for INTEGER-valued intensities in [0, 65535] (a radar's echoes are
 * 0..255): integer addition is exact in any order, and the kernel checks that every intensity is one. Otherwise a flag is
 * raised on the device and the grids of that call must not be used: zero them again and call
 * rb_land_accumulate_ordered, which adds every cell's points one after the other in the reference's order (slower; a
 * stable partition by cell first). rb_land_accumulate_status: host int32 out, 1 = some call since the last query saw
 * such an intensity; syncs and clears the flag. _status_async: the same into `dst` (device or pinned host memory) as a
 * copy enqueued on the stream, for callers that read several things back with one sync. rb_detect_block does all of
 * this by itself. */
int rb_land_accumulate_status(rb_ctx* ctx, int32_t* inexact, void* stream);
int rb_land_accumulate_status_async(rb_ctx* ctx, int32_t* dst, void* stream);
int rb_land_accumulate_ordered(rb_ctx* ctx, const float* x, const float* y, const float* inten, int64_t n,
                               const double* x_edges, int n_x_edges, const double* y_edges, int n_y_edges,
                               int32_t* count, double* isum, void* stream);

/* identify_land_cells (T4:394-410) in float64 on the device:
 *   land = (count / max(num_frames,1) >= persistence) & ((count>0 ? isum/count : 0) >= min_intensity)
 * land = uint8[n_cells]. No sync. */
int rb_land_cells(rb_ctx* ctx, const int32_t* count, const double* isum, int64_t n_cells,
                  int64_t num_frames, double persistence, double min_intensity,
                  uint8_t* land, void* stream);

/* filter_land_from_frame for all frames at once (T4:413-436): order-preserving removal of points
 * whose cell is land; frame_off_out[f] = new start of frame f. Outputs have capacity n.
 * keep_mask (optional, may be NULL) receives the uint8 keep flag per input point. No sync. */
int rb_land_filter(rb_ctx* ctx, const float* x, const float* y, const float* inten,
                   const int32_t* gain, int64_t n, const int64_t* frame_off, int64_t n_frames,
                   const double* x_edges, int n_x_edges, const double* y_edges, int n_y_edges,
                   const uint8_t* land,
                   float* x_out, float* y_out, float* inten_out, int32_t* gain_out,
                   int64_t* frame_off_out, uint8_t* keep_mask, void* stream);

/* ---- a7: temporal ST-DBSCAN ------------------------------------------------------------------
 * Replaces st_dbscan (T4:443-506 label computation; T3:101-136; PKG/processors/clustering.py:
 * 49-115; native precedent radar-pipeline-rs/src/processors/clustering.rs:209-325).
 *   neighbour(p,q) <=> sum_d (double(p_d)-double(q_d))^2 <= eps_space^2  (float64, inclusive,
 *                      self included: sklearn BallTree semantics, T4:474-475)
 *                  and |t_p - t_q| <= (float)eps_time in float32          (T4:485-486)
 *   core <=> |N| >= min_samples; clusters = connected components of cores;
 *   labels are the reference's own numbering: id = rank of the component's smallest core index;
 *   border points take the smallest id among their core neighbours; noise = -1.
 * Coordinates: component d of point i is at x[i*stride], y[i*stride], z[i*stride] (z NULL = 2-D),
 * so both SoA (stride 1) and a row-major [N][D] array (x=base, y=base+1, z=base+2, stride D) work.
 *   times  float32[n];  labels int32[n] out;  core uint8[n] out (optional, may be NULL)
 *   n_clusters: host int64 out (optional).  Syncs (grid dimensions are chosen on the host).
 */
int rb_stdbscan(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                const float* times, int64_t n, double eps_space, float eps_time, int min_samples,
                int32_t* labels, uint8_t* core, int64_t* n_clusters, void* stream);

/* The "paper" variant of the same clustering (PointCloudWorkF/stdbscan_denoising_pipeline.py:264-369, SURVEY.md
 * section 8 f rank 3): a point is core only if its neighbours ALSO span at least min_frames distinct int32(times)
 * (WF:308-315), and border points follow the rule of its FIFO expansion (WF:337-366): a border point joins the
 * smallest-id cluster among those of its core neighbours that either started (smallest core index) before the
 * border point's own index or whose start point itself is the neighbour. Labels are identical to the reference
 * function's. eps_time <= 30. Syncs. */
int rb_stdbscan_wf(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                   const float* times, int64_t n, double eps_space, float eps_time, int min_samples, int min_frames,
                   int32_t* labels, uint8_t* core, int64_t* n_clusters, void* stream);

/* Work counters of the last rb_stdbscan on this ctx (host): pair tests per neighbour sweep, grid
 * cells, cell size. For bench/roofline reporting only. */
typedef struct rb_dbscan_stats {
    int64_t n_points, n_cells, n_core, n_clusters;
    int64_t pair_tests_count, pair_tests_union, pair_tests_border;
    double cell_size, time_bin;
    int32_t dims[4];            /* nx, ny, nz, nt */
    int32_t time_radius;
    int32_t tight;              /* 1 = tight-cell bucket algorithm, 0 = general algorithm */
} rb_dbscan_stats;
int rb_stdbscan_last_stats(rb_ctx* ctx, rb_dbscan_stats* out);

/* Optional knowledge of the caller about the points of an ST-DBSCAN call: a box that contains every coordinate
 * and time (lo/hi = x, y, z, t; any superset is fine) and whether all times are integers. With a hint the plan
 * phase needs no bounds pass and does not sync. */
typedef struct rb_stdbscan_hint {
    float lo[4], hi[4];
    int32_t times_integer;
} rb_stdbscan_hint;

/* ---- a7 in phases (what rb_stdbscan runs back to back) -------------------------------------------
 * For callers that must exchange data between the phases - the time-sharded multi-GPU driver
 * (SURVEY.md section 8 e): every rank clusters its own frames plus a floor(eps_time)-frame halo,
 * replaces the core flags of the halo points by their owner's, and numbers components globally.
 * The plan (grid, sorted copies, bucket table) lives in the ctx until the next rb_stdbscan_plan /
 * rb_stdbscan; the coordinate and time buffers are only read by rb_stdbscan_plan.
 *
 *   rb_stdbscan_plan        same inputs as rb_stdbscan. Syncs (the grid is chosen on the host).
 *   rb_stdbscan_cores       core flags (neighbour count >= min_samples); core_out uint8[n]
 *                           (original order) optional.
 *   rb_stdbscan_set_cores   overwrite the core flags (uint8[n], original order).
 *   rb_stdbscan_components  connected components of the core points. global_index int64[n]
 *                           (optional; NULL = 0..n-1) gives every point its key; comp_key int64[n]
 *                           (optional output) = smallest key among the core points of the point's
 *                           component, -1 for non-core points.
 *   rb_stdbscan_assign      core_label int32[n]: final cluster id of every core point (ignored for
 *                           the others); labels int32[n] out: core points keep their id, border
 *                           points take the smallest id among their core neighbours, noise = -1.
 *                           labels may alias core_label.
 *   rb_relabel              out[i] = ids[j] with table_keys[j] == keys[i] (table_keys sorted
 *                           ascending, int64[m]); -1 when keys[i] < 0 or absent.
 * None of these sync except rb_stdbscan_plan. */
int rb_stdbscan_plan(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                     const float* times, int64_t n, double eps_space, float eps_time, int min_samples,
                     void* stream);
/* A hint that does NOT contain every point / time would put points into wrong buckets: the plan flags it on the device;
 * rb_stdbscan / rb_detect_block fail with RB_ERR_ARG at their final read-back, and a caller that drives the phases itself
 * asks with rb_stdbscan_check (syncs; also refreshes rb_stdbscan_last_stats). */
int rb_stdbscan_check(rb_ctx* ctx, void* stream);
int rb_stdbscan_plan_hinted(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                            const float* times, int64_t n, double eps_space, float eps_time, int min_samples,
                            const rb_stdbscan_hint* hint /* host, may be NULL */, void* stream);
int rb_stdbscan_cores(rb_ctx* ctx, uint8_t* core_out, void* stream);
int rb_stdbscan_set_cores(rb_ctx* ctx, const uint8_t* core_in, void* stream);
int rb_stdbscan_components(rb_ctx* ctx, const int64_t* global_index, int64_t* comp_key, void* stream);
int rb_stdbscan_assign(rb_ctx* ctx, const int32_t* core_label, int32_t* labels, void* stream);
int rb_relabel(rb_ctx* ctx, const int64_t* keys, int64_t n, const int64_t* table_keys,
               const int32_t* table_ids, int64_t m, int32_t* out, void* stream);

/* ---- the whole hot path for one block of frames in ONE call ----------------------------------------
 * What run_pipeline does between "CSV parsed" and "labels known" (T4:941-977) for F frames of G gains:
 * spoke-to-point + gain concat (a1, a2) -> if frames_built > land_min_frames: occupancy grid over the block,
 * land cells, land filter (a4-a6; the np.arange edges are reproduced on the host side of the library) ->
 * ST-DBSCAN over the (filtered) points with time = frame id (a7). All launches, the two small read-backs in
 * between (point count + bounds; filtered count) and the final counter read-back happen inside the library.
 *
 *   echo [F*G][S][E], cos/sin/range_res [F*G][S], sweep_gain int32[F*G]: device, as rb_spoke_to_points
 *   frame_ids: HOST float32[F]
 * Outputs (device unless noted), all with capacity buf->cap points:
 *   raw points x,y,inten,gain + frame_off int64[F+1]; filtered points fx,fy,finten,fgain + f_frame_off[F+1]
 *   (when the land filter did not run, res->filtered_is_raw = 1 and the f* arrays are not written: use the raw
 *   ones); labels int32; land grids count/isum/land with capacity max_cells; edges: HOST double arrays with
 *   capacity max_edges each.
 * Returns RB_ERR_CAPACITY (and the needed sizes in *res) when cap / max_cells / max_edges are too small. Syncs. */
typedef struct rb_detect_params {
    int32_t n_frames, gains_per_frame, n_spokes, n_bins;
    float intensity_threshold;
    int32_t point_stride;
    int32_t land_filter;            /* 0 = skip a4-a6 */
    int32_t land_min_frames;        /* the reference filters only when len(frames) > 10 (T4:954) */
    double land_resolution, land_persistence, land_min_intensity;
    double eps_space;
    float eps_time;
    int32_t min_samples;
    int32_t cluster;                /* 0 = stop after the land filter */
    int32_t echo_u8;                /* 1 = `echo` points at uint8 cells (rb_spoke_to_points_u8) */
    int32_t cluster_3d;             /* 1 = cluster on (x, y, z = intensity) like 3_stdbscan_point_clouds.py (T3:177-182:
                                       coords = column_stack((x, y, z))) instead of (x, y) */
} rb_detect_params;

typedef struct rb_detect_buffers {
    float *x, *y, *inten; int32_t* gain; int64_t* frame_off;
    float *fx, *fy, *finten; int32_t* fgain; int64_t* f_frame_off;
    int32_t* labels;
    int64_t cap;
    int32_t* count; double* isum; uint8_t* land; int64_t max_cells;
    double *x_edges, *y_edges; int32_t max_edges;             /* host */
} rb_detect_buffers;

typedef struct rb_detect_result {                            /* host */
    int64_t n_raw, n_points, n_clusters;
    int32_t frames_built, land_applied, filtered_is_raw;
    int32_t n_x_edges, n_y_edges;
    float bounds[4];                                          /* x_min, x_max, y_min, y_max of the raw points */
    int32_t land_ordered;                                     /* 1 = non-integer intensities: the ordered accumulation ran */
} rb_detect_result;

int rb_detect_block(rb_ctx* ctx, const float* echo, const float* cos_tab, const float* sin_tab, const float* range_res,
                    const int32_t* sweep_gain, const float* frame_ids, const rb_detect_params* prm,
                    const rb_detect_buffers* buf, rb_detect_result* res, void* stream);

/* ---- a8: per-frame cluster records on the device (SURVEY section 8 f, rank 1) -----------------------------------
 * What st_dbscan builds after the labels are known (T4:511-534) and what ObjectTracker.update (T4:553) and
 * save_tracking_results (T4:873-886) read: for every (frame, cluster id) that occurs - a SEGMENT - the number of points,
 * centroid = np.mean(points, axis=0) and mean intensity = np.mean(intensities), bit for bit in numpy's float32 arithmetic
 * (rows added in order per column; numpy's pairwise sum for the 1-D intensities; float32 division), plus the points grouped
 * by segment in their original order (a stable partition), so the host's per-cluster arrays are slices instead of masks.
 *   x, y, inten float32[n], labels int32[n] (-1 = noise, ids < n_clusters), frame_off int64[n_frames + 1]: device.
 *   Table columns (device, capacity cap_segments), segments ordered by frame, then label (-1 first):
 *     frame  int32  index of the frame in the block          label  int32  cluster id, -1 = the frame's noise entry
 *     first  int32  index INSIDE the frame of the segment's first point (the order of first occurrences is what decides
 *                   the iteration order of `set(frame_labels)`, T4:518-521: the host replays it)
 *     count  int32  points                                   start  int64  offset in gx / gy / gi (-1 for noise)
 *     cx, cy, mean_intensity float32 (0 for noise)
 *   gx, gy, gi float32[n]: grouped points (noise points are not copied).
 *   n_segments, n_grouped: host int64 out. RB_ERR_CAPACITY (with *n_segments set) when cap_segments is too small, or when
 *   n_frames * (n_clusters + 1) exceeds the slot table (2^27): pass fewer frames per call - frames are independent.
 * Syncs once. */
typedef struct rb_cluster_table {
    int32_t *frame, *label, *first, *count;
    int64_t* start;
    float *cx, *cy, *mean_intensity;
} rb_cluster_table;
int rb_cluster_records(rb_ctx* ctx, const float* x, const float* y, const float* inten, const int32_t* labels, int64_t n,
                       const int64_t* frame_off, int64_t n_frames, int64_t n_clusters, const rb_cluster_table* table,
                       int64_t cap_segments, float* gx, float* gy, float* gi, int64_t* n_segments, int64_t* n_grouped,
                       void* stream);

/* np.arange(lo, fl32(hi + step), step) as build_occupancy_grid computes its edges (T4:372-373: float32 scalar
 * bounds, float64 result): out[0] = lo, out[1] = lo + step, out[i] = lo + i*(out[1] - lo). Host function.
 * Returns the number of edges (> cap: nothing written beyond cap). */
int64_t rb_arange_edges(float lo, float hi, double step, double* out, int64_t cap);

/* HOST function of the time-sharded multi-GPU path (sharded.py): global cluster numbering from the ranks' local
 * components. keys[n_keys] = every rank's distinct local component keys (key = smallest global core-point index the rank
 * saw in the component; duplicates allowed). pair_a/pair_b[n_pairs] = the keys under which two neighbouring ranks hold
 * the SAME boundary core point: each pair ties two local components together. Writes the sorted distinct keys to
 * table_keys and, per key, the final cluster id to table_ids - the id of a cluster being the rank of its smallest key
 * among all clusters, which is the reference's numbering (first core point in index order starts cluster 0; T4:481-500,
 * SURVEY.md N4). Returns the table size (<= cap) or a negative RB_ERR_*; *n_clusters = number of clusters. */
int64_t rb_stitch_components(const int64_t* keys, int64_t n_keys, const int64_t* pair_a, const int64_t* pair_b,
                             int64_t n_pairs, int64_t* table_keys, int32_t* table_ids, int64_t cap, int64_t* n_clusters);

/* ---- a7 over a whole recording: ST-DBSCAN in time windows (DESIGN.md section 3.8) ----------------------------------
 * The labels, core flags and n_clusters of rb_stdbscan on the same points with times = the frame id of each point, for
 * any number of points (int64; no 2^31 limit on the total) and any valid choice of windows. Points are frame-ordered:
 * frame f holds points [frame_off_host[f], frame_off_host[f+1]) of x/y/z (component d of point i at x[i*stride] ...,
 * z NULL = 2-D). frame_ids_host float32[F]: integers, strictly increasing, magnitude < 2^24. cuts_host[n_windows+1]:
 * frame indices, strictly increasing from 0 to F; window k owns frames [cuts[k], cuts[k+1]) and with more than one
 * window each is at least h = floor(eps_time) frames long. Its local problem is frames [cuts[k]-h, cuts[k+1]+h), clipped
 * to the recording; each local problem must stay under 2^31-1 points, and the scratch follows the largest one (plus one
 * byte per point of the recording when `core` is NULL). One window is rb_stdbscan itself; with K > 1 windows every
 * window is planned three times (cores; components; labels) and the host stitches the components in between.
 *   hint: host, optional: a box containing every x, y, z (its time range is ignored: each window's comes from the ids);
 *         with it no plan syncs (a box that misses a point fails the call with RB_ERR_ARG at the end).
 *   labels int32[N] out; core uint8[N] out (optional); n_clusters host int64 out (optional).
 * RB_ERR_ARG before any work when the ids, offsets or cuts break the rules above. Syncs. */
int rb_stdbscan_windowed(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                         const int64_t* frame_off_host, const float* frame_ids_host, int64_t n_frames,
                         const int64_t* cuts_host, int64_t n_windows, double eps_space, float eps_time, int min_samples,
                         const rb_stdbscan_hint* hint, int32_t* labels, uint8_t* core, int64_t* n_clusters, void* stream);

/* rb_stdbscan_windowed with the PointCloudWorkF rules: the labels, core flags and n_clusters of rb_stdbscan_wf on the
 * same points with times = the frame id of each point, for any number of points and any valid choice of windows. Same
 * arguments, windows, scratch and hint as rb_stdbscan_windowed, plus min_frames (>= 1). A window's components only know
 * the part of a cluster inside its local problem, while the WF border rule compares a border point's index with the start
 * of the WHOLE cluster (its smallest core index): between the second and third pass the host takes every cluster's start
 * from the stitched key table and uploads it, and the third pass assigns border points with recording-wide indices and
 * those starts (DESIGN.md section 3.8). One window is rb_stdbscan_wf itself.
 * RB_ERR_ARG before any work when min_frames < 1, eps_time is not <= 30 (NaN included), or the ids, offsets or cuts break the rules of
 * rb_stdbscan_windowed. Syncs. */
int rb_stdbscan_windowed_wf(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                            const int64_t* frame_off_host, const float* frame_ids_host, int64_t n_frames,
                            const int64_t* cuts_host, int64_t n_windows, double eps_space, float eps_time, int min_samples,
                            int min_frames, const rb_stdbscan_hint* hint, int32_t* labels, uint8_t* core, int64_t* n_clusters,
                            void* stream);

/* The three passes of rb_stdbscan_windowed(_wf) as entries of their own, over a LOCAL problem: frames [0, n_frames) of
 * x/y/z with host frame offsets and ids as above, of which the windows (cuts_host[n_windows+1], from own_fa to own_fb)
 * cover only the OWNED frames [own_fa, own_fb); the frames before and after are halo frames that a window's local
 * problem may reach (h = floor(eps_time) of them on each side where a neighbour exists). Point i of the local problem
 * has the global index index_base + i (components are keyed by it). min_frames 0 = the T4 rules, >= 1 = the
 * PointCloudWorkF variant (eps_time <= 30). core uint8[frame_off_host[n_frames]] spans the whole local problem; the
 * hint and its flag work as in rb_stdbscan_windowed. The multi-GPU recording (sharded.py, ShardedRecording) runs them on
 * every rank with the halo exchanges and the stitch of all ranks' windows in between:
 *   _pass_cores   the exact core flags of the owned points into core (clears the hint flag of the context)
 *   _pass_keys    after the halo slots of core hold their owners' flags: windows [first_window, first_window + n_encode)
 *                 encode their zones in rb_shard_pack_keys' format into vec int64[n_encode * (9 + 2 cap_keys)] (window k
 *                 at (k - first_window) (9 + 2 cap_keys); entries beyond cap_keys are dropped, the counts stay true). The
 *                 left zones of the first window and the right zones of the last one are encoded when left_neighbour /
 *                 right_neighbour say that a neighbour holds the frames beyond. hint_outside (device, optional): the hint
 *                 flag of passes 1 and 2 is OR-ed into it.
 *   _pass_labels  with the stitched table (host: sorted keys, their ids) and, for min_frames, every cluster's start (host
 *                 int64[n_start], its smallest global core index): labels int32 of the owned points (labels[0] = the
 *                 first owned point). Syncs; fails with RB_ERR_ARG when the hint missed a point.
 * None but _pass_labels syncs. RB_ERR_ARG before any work when the ids, offsets, owned range or cuts break the rules. */
int rb_stdbscan_windowed_pass_cores(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                                    const int64_t* frame_off_host, const float* frame_ids_host, int64_t n_frames, int64_t own_fa,
                                    int64_t own_fb, const int64_t* cuts_host, int64_t n_windows, int64_t index_base, double eps_space,
                                    float eps_time, int min_samples, int min_frames, const rb_stdbscan_hint* hint, uint8_t* core,
                                    void* stream);
int rb_stdbscan_windowed_pass_keys(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                                   const int64_t* frame_off_host, const float* frame_ids_host, int64_t n_frames, int64_t own_fa,
                                   int64_t own_fb, const int64_t* cuts_host, int64_t n_windows, int64_t index_base, double eps_space,
                                   float eps_time, int min_samples, int min_frames, const rb_stdbscan_hint* hint, int left_neighbour,
                                   int right_neighbour, const uint8_t* core, int64_t first_window, int64_t n_encode, int64_t cap_keys,
                                   int64_t* vec, unsigned long long* hint_outside, void* stream);
int rb_stdbscan_windowed_pass_labels(rb_ctx* ctx, const float* x, const float* y, const float* z, int64_t stride,
                                     const int64_t* frame_off_host, const float* frame_ids_host, int64_t n_frames, int64_t own_fa,
                                     int64_t own_fb, const int64_t* cuts_host, int64_t n_windows, int64_t index_base, double eps_space,
                                     float eps_time, int min_samples, int min_frames, const rb_stdbscan_hint* hint, const uint8_t* core,
                                     const int64_t* table_keys_host, const int32_t* table_ids_host, int64_t n_table,
                                     const int64_t* start_of_host, int64_t n_start, int32_t* labels, void* stream);

/* HOST function: the pairing of two run-length encodings of the SAME boundary points (rb_shard_pack_keys' zone format:
 * keys[j] holds from position starts[j] of the zone to the next start, -1 = not a core point; starts[0] = 0) into the
 * distinct (key_a, key_b) pairs of the core points, sorted. Cost follows the number of runs, not of points. Writes at
 * most cap pairs and returns their total number, or a negative RB_ERR_* when the encodings disagree on which points
 * are core points or are malformed. */
int64_t rb_pair_zone_runs(const int64_t* keys_a, const int64_t* starts_a, int64_t n_a, const int64_t* keys_b,
                          const int64_t* starts_b, int64_t n_b, int64_t* pair_a, int64_t* pair_b, int64_t cap);

/* ---- multi-GPU: time sharding (SURVEY section 8 e) -----------------------------------------------------------------
 * One process per GPU; rank r owns a contiguous block of frames and clusters it together with a floor(eps_time)-frame
 * halo from each neighbour (radar_point_cloud_tracking_b200/sharded.py drives the protocol, DESIGN.md section 6). The
 * collectives are NCCL calls made BY THE LIBRARY on the caller's stream; the library binds to the NCCL the process already
 * holds (the one PyTorch loaded; RB_NCCL_LIBRARY names another). A context owns one communicator; a rank that keeps
 * several blocks in flight uses one context - hence one communicator - per block slot.
 *   rb_comm_unique_id   HOST: a fresh NCCL unique id (128 bytes), to be created on one rank and handed to all others
 *                       by whatever means the application has (torch.distributed broadcast, MPI, a file)
 *   rb_comm_init        collective over all ranks: joins the communicator `unique_id` as `rank` of `world`
 *   rb_comm_all_gather  send[bytes_per_rank] of every rank -> recv[world * bytes_per_rank] on every rank
 *   rb_comm_all_reduce_sum / _grids   in-place sums (dtype 0 = int32, 1 = float64); _grids: the land filter's count and
 *                       intensity grids in one NCCL group (sums of integers: exact in any order)
 *   rb_comm_exchange    neighbour exchange in one NCCL group: part k of to_left goes to rank - 1, of to_right to rank + 1,
 *                       from_left / from_right receive the neighbours' parts; sizes in bytes, 0 = nothing; device pointers
 * None of these sync the stream. */
int rb_comm_unique_id(uint8_t* out128);
int rb_comm_init(rb_ctx* ctx, const uint8_t* unique_id128, int rank, int world);
int rb_comm_destroy(rb_ctx* ctx);
int rb_comm_info(rb_ctx* ctx, int* rank, int* world);
int rb_comm_all_gather(rb_ctx* ctx, const void* send, void* recv, int64_t bytes_per_rank, void* stream);
int rb_comm_all_reduce_sum(rb_ctx* ctx, void* buf, int64_t count, int dtype, void* stream);
int rb_comm_all_reduce_grids(rb_ctx* ctx, int32_t* count, double* isum, int64_t cells, void* stream);
int rb_comm_exchange(rb_ctx* ctx, int n_parts, const void* const* to_left, const int64_t* to_left_bytes,
                     const void* const* to_right, const int64_t* to_right_bytes, void* const* from_left,
                     const int64_t* from_left_bytes, void* const* from_right, const int64_t* from_right_bytes, void* stream);

/* What the collectives of a block carry, assembled on the device (no sync, a few small launches each):
 *   rb_shard_pack_stats   out7 float64 = [frames with points, points, x_min, x_max, y_min, y_max, capacity] from the raw
 *                         frame offsets (int64[F+1]) and rb_bounds_counted's output
 *   rb_shard_pack_layout  out int64[2 + 4 hh] = [points owned, first point of the last hh frames, ids and point counts of
 *                         the first hh frames, ids and point counts of the last hh frames]; frame_ids: HOST int64[F]
 *   rb_shard_local_index  times float32[n_loc] and global point index int64[n_loc] of the local problem
 *                         [left halo (nl) | owned (n_own) | right halo (nr)]; head / ids: HOST arrays describing its
 *                         frames (head[f] = first local point of frame f, head[n_local_frames] = n_loc); the three parts
 *                         start at the global indices lbase / gbase / rbase
 *   rb_shard_pack_keys    vec int64[9 + 2 cap_keys] = [5 running entry counts | 4 zone lengths | keys[cap_keys] | starts[cap_keys]]:
 *                         the component keys (rb_stdbscan_components) of four zones [a, b) of the local problem (zones8: HOST
 *                         int64[8]) RUN-LENGTH ENCODED over all their points - an entry is a key (-1 = not a core point) and the
 *                         position in the zone from which it holds; two ranks' encodings of the same boundary points are
 *                         merged by position on the host, at a cost that follows the number of runs, not of points - followed
 *                         by the keys that are their own global index (one per local component). Entries beyond cap_keys are
 *                         dropped; the counts stay true (the caller repeats with a larger vector) */
int rb_shard_pack_stats(rb_ctx* ctx, const int64_t* frame_off, int64_t n_frames, const float* bounds4, int64_t cap, double* out7,
                        void* stream);
int rb_shard_pack_layout(rb_ctx* ctx, const int64_t* frame_off, int64_t n_frames, const int64_t* frame_ids_host, int hh, int64_t* out,
                         void* stream);
int rb_shard_local_index(rb_ctx* ctx, const int64_t* head_host, const float* ids_host, int64_t n_local_frames, int64_t nl,
                         int64_t n_own, int64_t nr, int64_t lbase, int64_t gbase, int64_t rbase, float* times, int64_t* gidx,
                         void* stream);
int rb_shard_pack_keys(rb_ctx* ctx, const int64_t* key, const int64_t* gidx, int64_t n_loc, const int64_t* zones8_host, int64_t cap_keys,
                       int64_t* vec, void* stream);

/* ---- ingest (SURVEY section 8 f, rank 2) --------------------------------------------------------------------------
 * One radar sweep CSV parsed on the device; replaces the numeric part of pd.read_csv in load_radar_csv
 * (4_temporal_object_tracker.py:189-206: header row skipped, columns Status, Scale, Range, Gain, Angle,
 * Echo_0..Echo_{E-1}, NaN echoes -> 0). text[n_bytes] = the file's bytes on the device. Outputs, for data row r
 * (line r + 1 of the file): echo[r * E + c] = Echo_c as uint8 (feeds rb_spoke_to_points_u8 directly);
 * row_start[r] / prefix_end[r] = byte offsets of the row's first character and of its fifth comma - the caller parses
 * the five leading fields [row_start, prefix_end) on the host with the reference's own parser (Scale may be a decimal).
 * info[0] = number of lines in the file (rows = info[0] - 1), info[1] = OR of RB_CSV_* bits: 0 means every echo field
 * was empty or 1..3 digits <= 255 and every row had exactly E + 5 fields. Any other input only sets a bit; the caller
 * then parses that file with the reference's parser, so unusual files keep the reference's exact behaviour.
 * max_rows = capacity of echo / row_start / prefix_end in rows. Enqueues only; read info after a stream sync. */
#define RB_CSV_NOT_INTEGER 1   /* an echo field is not 1..3 plain digits (sign, decimal point, blank, quote, ...), or a
                                  carriage return that is not followed by a line feed (pandas ends a line there)   */
#define RB_CSV_OUT_OF_RANGE 2  /* an echo value above 255                                                         */
#define RB_CSV_RAGGED 4        /* a row without exactly E + 5 fields                                              */
#define RB_CSV_BLANK_LINE 8    /* an empty line among the rows                                                    */
#define RB_CSV_CAPACITY 16     /* more rows than max_rows                                                         */
int rb_csv_parse_sweep(rb_ctx* ctx, const uint8_t* text, int64_t n_bytes, int n_echo_columns, int64_t max_rows,
                       uint8_t* echo, int32_t* row_start, int32_t* prefix_end, int32_t* info, void* stream);

/* Many sweep CSVs per launch, in two calls with one read-back between them. text[n_bytes] (device, n_bytes < 2^31)
 * holds W files; file w is text[file_off[w], file_off[w] + file_len[w]), file_off[w] is a multiple of 4096 and files do
 * not overlap: file_off[w] + file_len[w] <= file_off[w + 1] (file_off, file_len: int64 device arrays; the kernels give a
 * chunk to the last file starting at or before it, so overlapping files would get wrong row counts). Same grammar and status bits as rb_csv_parse_sweep, decided per file: a
 * file's status never depends on its neighbours.
 * rb_csv_sweeps_lines: chunk_base[ceil(n_bytes / 4096) + 1] (device) receives the newline scan (chunk_base[last] = all
 * newlines), rows[w] the data rows of file w (lines minus the header), status[w] the line-level bits (lone CR, blank
 * line, RB_CSV_CAPACITY = more lines than rows of E + 5 fields could fill; rows[w] is then 0).
 * rb_csv_parse_sweeps: the caller reads back rows and status, sets row_base[w] = sum of rows[v < w] over the files it
 * wants parsed (0 rows for the others; row_base[W] = n_rows) and passes n_newlines = chunk_base[last]. For row r of
 * file w, row R = row_base[w] + r: echo[R * E + c] = Echo_c (uint8), row_start[R] / prefix_end[R] = file-relative offsets
 * of the row and of its fifth comma, angle[R] / scale[R] = Angle and Scale as float32; gain[w] = Gain of row 0.
 * Leading fields: Angle and Scale of every row and Gain of row 0 must be -?D+ or -?D+.D+ (Gain: -?D+, within int32) with
 * at most 15 digits and not a negative zero; the value is the digits as an exact double divided once by 10^(fraction
 * digits), rounded to float32 - bit for bit what pandas' C parser gives. Anything else sets RB_CSV_LEAD_FIELDS: the
 * echoes stay valid, the caller parses that file's leading fields itself. status[w] accumulates across both calls. */
#define RB_CSV_LEAD_FIELDS 32  /* a leading field outside the device grammar (echoes still valid)                   */
int rb_csv_sweeps_lines(rb_ctx* ctx, const uint8_t* text, int64_t n_bytes, const int64_t* file_off, const int64_t* file_len,
                        int n_files, int n_echo_columns, int32_t* chunk_base, int32_t* rows, int32_t* status, void* stream);
int rb_csv_parse_sweeps(rb_ctx* ctx, const uint8_t* text, int64_t n_bytes, const int64_t* file_off, const int64_t* file_len,
                        int n_files, int n_echo_columns, const int32_t* chunk_base, int64_t n_newlines, const int64_t* row_base,
                        int64_t n_rows, uint8_t* echo, int32_t* row_start, int32_t* prefix_end, float* angle, float* scale,
                        int32_t* gain, int32_t* status, void* stream);

/* ---- PLY output (SURVEY section 8 f, rank 4) ------------------------------------------------------------------------
 * HOST function: appends the vertex lines of an ASCII PLY to the file at `path` - the bytes that
 * np.savetxt(fh, data, fmt="%.4f %.4f %.4f %d %d %d") writes in write_ply_fast (5_gain_fusion_ply_builder.py:370-403;
 * identical to write_ply's per-point loop T5:345-367 and to the ASCII branch of
 * PointCloudWorkF/stdbscan_denoising_pipeline.py:828-851) for float32 coordinates and uint8 colours rgb[n][3].
 * All pointers are host pointers. The header is the caller's business. */
int rb_ply_append_ascii(const char* path, const float* x, const float* y, const float* z, const uint8_t* rgb, int64_t n);

/* The same vertex lines formatted on the device, for every float32 value (no printf): the lines of x, y, z float32[n]
 * and rgb uint8[n][3], concatenated into text (capacity cap bytes), and line_end int64[n] = the end offset of every line
 * in text. total: device int64[1] = the bytes of all lines. When total > cap nothing is written to text (line_end and
 * total still are): the caller reads total back and calls again with a larger buffer. Three launches, no sync. */
int rb_ply_format_ascii(rb_ctx* ctx, const float* x, const float* y, const float* z, const uint8_t* rgb, int64_t n,
                        char* text, int64_t cap, int64_t* line_end, int64_t* total, void* stream);

/* The 15-byte little-endian records of write_ply_binary (WF:797-827): out[15 * i ..] = x, y, z float32 then r, g, b.
 * One launch, no sync. */
int rb_ply_pack_binary(rb_ctx* ctx, const float* x, const float* y, const float* z, const uint8_t* rgb, int64_t n,
                       uint8_t* out, void* stream);

/* intensity_to_rgb (T5:292-327) of values[n], float32 (is_f64 = 0) or float64 (is_f64 = 1), with numpy >= 2's dtype rules
 * (all arithmetic in the input's dtype, ramps truncated to uint8), into rgb uint8[n][3]. normalize = 1 first applies
 * normalize_intensity (T5:276-289) to each frame [frame_off[f], frame_off[f+1]) of frame_off int64[n_frames + 1] (numpy's
 * linear 99th percentile and the minimum of the frame; elements outside every frame are not written). A NaN or a value
 * outside [0, 255] after the optional normalisation has no defined colour in the reference: it sets bit 0 of status
 * (device int32[1], cleared by the call) and is coloured black. One launch (normalize: one block per frame), no sync. */
int rb_ply_colors_intensity(rb_ctx* ctx, const void* values, int is_f64, int64_t n, const int64_t* frame_off,
                            int64_t n_frames, int normalize, uint8_t* rgb, int32_t* status, void* stream);

/* gain_to_rgb (T5:330-342): the GAIN_COLORS colour of each int32 gain, black for any other gain. One launch, no sync. */
int rb_ply_colors_gain(rb_ctx* ctx, const int32_t* gains, int64_t n, uint8_t* rgb, void* stream);

/* ---- test/bench infrastructure (not part of the reference surface) ---------------------------
 * Device twin of radar_point_cloud_tracking_b200.synthetic.synth_echo: fills echo[W][S][E] for
 * sweeps w0 .. w0+n_sweeps-1 of the data set. sweep_keys uint32[n_sweeps], clutter_thr
 * uint32[n_sweeps], rects int32[n_rects][10], rect_off int32[n_frames+1] (all device). */
int rb_synth_echo(rb_ctx* ctx, float* echo, int64_t n_sweeps, int n_spokes, int n_bins,
                  int gains_per_frame, int64_t first_frame,
                  const uint32_t* sweep_keys, const uint32_t* clutter_thr,
                  const int32_t* rects, const int32_t* rect_off, void* stream);

/* Diagnostic switches. "spoke_profile" = 1: rb_spoke_to_points records CUDA events (on the launch stream)
 * around each of its three kernels; read them back with rb_get_info. "spoke_mask_variant": 0 = auto (the
 * TMA-staged mask kernel when S*E % 4 == 0 and echo is 16-byte aligned, else the register-staged one),
 * 1 = always register-staged, 2 = require TMA-staged (error when the shape is not eligible).
 * "dbscan_mode": 0 = auto (tight-cell bucket algorithm when the times are integers and the bucket table
 * fits the budget), 1 = always the general algorithm, 2 = require the tight one. */
int rb_set_option(rb_ctx* ctx, const char* name, int64_t value);
/* "launches"; "spoke_last_variant" (1 = register-staged, 2 = TMA-staged); "land_last_variant" (accumulation kernel of the last
 * rb_land_accumulate / rb_land_accumulate_ordered: 1 = shared-memory histogram, 2 = global atomics, 3 = ordered); "spoke_mask_ns" / "spoke_offsets_ns" / "spoke_emit_ns" = device time of the kernels of the
 * last profiled rb_spoke_to_points (syncs on its last event); -1 for unknown names or nothing recorded. */
int64_t rb_get_info(rb_ctx* ctx, const char* name);

/* Number of kernels this library has launched on this ctx since creation (bench "gpu_launches"). */
int64_t rb_launch_count(rb_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* RADARB200_H */
