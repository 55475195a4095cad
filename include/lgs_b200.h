/* lgs_b200.h -- C ABI of the B200-native scan-matching / occupancy-grid backend.
 *
 * This is the drop-in boundary (SURVEY.md section 8(b)): the C++ adapters that subclass the
 * reference's ScanMatcher / LoopDetector (adapters/, INTEGRATION.md) call ONLY these entry
 * points.  Conventions: extern "C", opaque handles, int status return (0 = LGS_OK), no
 * exceptions across the boundary, caller-owned host buffers, callee-owned device buffers
 * freed by the matching *_destroy.  One lgs_ctx owns one CUDA stream + scratch and may be
 * used by one host thread at a time; different contexts may be used concurrently (the
 * reference calls OptimizePose from the front-end thread and Detect from the back-end
 * thread, lidar_graph_slam_backend.cpp:39-40).  There is no CPU fallback: every call fails
 * with LGS_ERR_CUDA when no sm_100-class device is usable.
 *
 * Reference interfaces replaced (file:line under the reference tree):
 *   lgs_grid_*                 GridMap<T> storage read through Value(x, y, unknown)
 *                              (grid_map/grid_map.hpp:859-873) and
 *                              WorldCoordinateToGridCellIndex (grid_map.hpp:779-790)
 *   lgs_precompute*            PrecomputeGridMap / PrecomputeGridMaps / SlidingWindowMaxRow /
 *                              SlidingWindowMaxCol (mapping/grid_map_builder.cpp:403-536,
 *                              util.hpp:199-253)
 *   lgs_rtcsm_*                ScanMatcherRealTimeCorrelative::OptimizePose(grid, coarse, scan,
 *                              pose, thr) incl. ComputeSearchStep / ComputeScanIndices /
 *                              ComputeScore / EvaluateHighResolutionMap
 *                              (mapping/scan_matcher_real_time_correlative.cpp:50-256)
 *   lgs_bb_*                   ScanMatcherBranchBound::OptimizePose(grid, pyramids, scan, pose,
 *                              thr) + ScorePixelAccurate::Score
 *                              (mapping/scan_matcher_branch_bound.cpp:47-163,
 *                              mapping/score_function_pixel_accurate.cpp:19-76)
 *   lgs_grid_integrate_scans   GridMapBuilder::UpdateGridMap / ConstructMapFromScans scan
 *                              integration loops (mapping/grid_map_builder.cpp:170-186, :311-328),
 *                              Bresenham (util.hpp:257-303), BinaryBayesGridCell::Update
 *                              (grid_map/binary_bayes_grid_cell.hpp:75-119)
 *
 * Matchers return window INDICES + score; the adapter rebuilds the pose with the reference's
 * own expression (sensorPose.mX + bestWinX * stepX, scan_matcher_real_time_correlative.cpp:
 * 122-125) and runs the host tail (Cost, ComputeCovariance, MoveBackward) unchanged.
 */
#ifndef LGS_B200_H
#define LGS_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define LGS_OK            0
#define LGS_ERR_INVALID   1   /* bad argument */
#define LGS_ERR_CUDA      2   /* CUDA runtime error or no usable device */
#define LGS_ERR_NOMEM     3
#define LGS_ERR_APRON     4   /* search window wider than the grid's zero apron */
#define LGS_ERR_OVERFLOW  5   /* an internal work list overflowed its capacity */

typedef struct lgs_ctx lgs_ctx;
typedef struct lgs_grid lgs_grid;
typedef struct lgs_rtcsm_batch lgs_rtcsm_batch;
typedef struct lgs_pyramid lgs_pyramid;
typedef struct lgs_bb_batch lgs_bb_batch;

/* ---- context --------------------------------------------------------------------------- */
int lgs_device_count(void);                 /* usable CUDA devices (0 without a driver / GPU) */
int lgs_ctx_create(int device, lgs_ctx** out);
int lgs_ctx_destroy(lgs_ctx* ctx);
const char* lgs_ctx_last_error(const lgs_ctx* ctx);
int lgs_ctx_synchronize(lgs_ctx* ctx);
/* Stream order across two contexts of one device: everything enqueued on `ctx` after this call runs
 * after everything enqueued on `other` before it (an event wait, nothing blocks on the host).  Used by
 * callers that pipeline steps over two contexts and need step k's record exchange to get its SMs
 * before step k + 1's persistent kernel takes all of them. */
int lgs_ctx_wait_ctx(lgs_ctx* ctx, lgs_ctx* other);
/* The cudaStream_t every call on this context is ordered on (for event timing). */
void* lgs_ctx_stream(lgs_ctx* ctx);
/* CUDA-event stopwatch on the context stream: start, enqueue work, stop -> milliseconds. */
int lgs_ctx_timer_start(lgs_ctx* ctx);
int lgs_ctx_timer_stop(lgs_ctx* ctx, float* ms);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
long long lgs_ctx_launch_count(const lgs_ctx* ctx);
/* Page-lock / unlock a caller-owned host buffer (cudaHostRegister) so that the H2D copies of the
 * upload calls run at full PCIe / C2C speed and asynchronously; optional, any host memory works. */
int lgs_host_pin(lgs_ctx* ctx, void* ptr, unsigned long long bytes);
int lgs_host_unpin(lgs_ctx* ctx, void* ptr);
/* Raw device buffers for record exchange (gather / send / receive buffers of loop detection): plain
 * cudaMalloc memory of the context's device, so it is reachable from peer devices once peer access is
 * enabled (lgs_group_create) and registrable with a collective library. */
int lgs_device_alloc(lgs_ctx* ctx, unsigned long long bytes, void** out);
int lgs_device_free(lgs_ctx* ctx, void* ptr);
/* device -> host on the context stream, waits. */
int lgs_device_download(lgs_ctx* ctx, const void* device_ptr, void* host, unsigned long long bytes);
const char* lgs_version(void);
/* Diagnostic (bench.py roofline): measured bandwidth, in GB/s of useful bytes, of warp-wide 8-byte
 * gathers of `row_lanes` (25 or 32) consecutive doubles from an nx x ny array -- the access shape of
 * the scoring kernels.  aligned: rows start on 256-byte boundaries; local: successive rows move by a
 * few cells (L1 hits) instead of uniformly at random (L2 hits). */
int lgs_measure_gather_peak(lgs_ctx* ctx, int nx, int ny, int row_lanes, int aligned, int local,
                            double* gbps);
/* Per-context tuning / diagnostic / test hooks; none of them changes results.  The LGS_* environment
 * variables only supply the DEFAULTS of a new context (read once inside lgs_ctx_create); no run path
 * reads the environment or any process-global state afterwards.  Names:
 *   "edge_eps"          width (in cells) of the guard band around cell edges inside which a projected
 *                       point is re-derived exactly (default 1e-9; values outside (0, 0.5) restore it).
 *                       Raising it only moves more points onto the exact paths.
 *   "csm_flat"          correlative sweep: flattened one-hypothesis-per-thread kernel      (LGS_CSM_FLAT)
 *   "bb_sync"/"bb_table" branch-and-bound: level-synchronous exact path only       (LGS_BB_SYNC / _TABLE)
 *   "bb_warp_below"     exact path: node count below which a level scores a warp per node
 *   "bb_resolve_ulps"   device-only run: half width, in ulps of cos / sin, of the interval that decides
 *                       near-edge points on the device (default 8; huge values force the exact fallback)
 *   "bb_blocks_per_sm", "bb_cost_g1" / "_g4" / "_g8" / "_g32"   residency and per-pass cost model (us)
 *                       of the persistent kernel's warp mappings
 *   "bb_host_timing", "integ_host_timing", "integ_timing", "integ_diag"   timing reports on stderr
 *   "integ_side_words"  integration side-buffer size in words (tests shrink it)    (LGS_INTEG_SIDE_WORDS)
 *   "integ_resolve_ulps" lgs_grid_construct_many: half width, in ulps of cos / sin, of the interval around the
 *                       device's value (default 8; huge values send every hit and every bbox side to the host)
 *   "gs_tables"         grid search through the index tables instead of the fused kernel (LGS_GS_TABLES) */
int lgs_ctx_set_option(lgs_ctx* ctx, const char* name, double value);
int lgs_ctx_get_option(const lgs_ctx* ctx, const char* name, double* value);

/* ---- dense device grid ---------------------------------------------------------------------
 * Row-major double[ny][nx], 0.0 = unknown, surrounded by `apron` zero cells on every side so
 * that out-of-map reads return 0.0 exactly like GridMap::Value(x, y, unknown).  Cell (0,0)'s
 * lower-left corner is at (min_x, min_y); index = floor((p - min) / res). */
int lgs_grid_create(lgs_ctx* ctx, int nx, int ny, double min_x, double min_y, double res,
                    int apron, lgs_grid** out);
int lgs_grid_destroy(lgs_grid* g);
int lgs_grid_upload(lgs_grid* g, const double* dense);       /* host [ny][nx] -> device */
int lgs_grid_download(const lgs_grid* g, double* dense);     /* device -> host [ny][nx] */
/* Cells [x0, x0 + w) x [y0, y0 + h) only: row r of the region goes to dst + r * dst_pitch (pitch in
 * doubles, >= w).  What a builder needs after integrating one scan: only the scan's bounding box can
 * have changed (grid_map_builder.cpp:152-186). */
int lgs_grid_download_region(const lgs_grid* g, int x0, int y0, int w, int h, double* dst,
                             long long dst_pitch);
/* Device -> device: `dst` takes the geometry (size, placement, window) and the cells of `src`,
 * keeping its own apron (which stays 0.0).  The grids may belong to different contexts of the same
 * device; the copy runs on dst's stream after src's stream has drained.  This is the hand-over of
 * the builder's device-resident latest map to the matcher (no host round trip of the map,
 * lidar_graph_slam.cpp:99 / lidar_graph_slam_frontend.cpp:93-107). */
int lgs_grid_copy(const lgs_grid* src, lgs_grid* dst);
/* Large maps split into row bands (one per GPU): declare this grid to hold cells
 * [off_x, off_x + nx) x [off_y, off_y + ny) of a larger map whose cell (0, 0) has its lower-left
 * corner at (min_x, min_y).  World -> cell conversion stays floor((p - min) / res) of the WHOLE map,
 * so results are bit-identical to matching against it as long as every cell a match reads lies
 * inside the band (the caller sizes the margin).  Honoured by lgs_precompute / lgs_pyramid_* (which
 * are geometry free) and lgs_bb_*; the correlative matcher and the integration reject windows. */
int lgs_grid_set_window(lgs_grid* g, int off_x, int off_y);
int lgs_grid_info(const lgs_grid* g, int* nx, int* ny, double* min_x, double* min_y,
                  double* res, int* apron);

/* Mirror of GridMap::Resize's patch copy (grid_map.hpp:652-711): the grid becomes nx x ny cells
 * at (min_x, min_y); new cell (x, y) takes old cell (x + shift_x, y + shift_y), 0.0 elsewhere. */
int lgs_grid_resize(lgs_grid* g, int nx, int ny, double min_x, double min_y, int shift_x,
                    int shift_y);
int lgs_grid_clear(lgs_grid* g);                             /* GridMap::Reset */

/* ---- occupancy-grid scan integration ---------------------------------------------------------
 * Per scan: sensor position and the hit points of the beams that passed the range filter, in
 * beam order, exactly as ComputeBoundingBoxAndScanPoints / ConstructMapFromScans produce them
 * (grid_map_builder.cpp:335-380, :240-277).  Scans are applied in order; every touched cell
 * must already be inside the grid (expand first).  n_updates (optional) receives the number of
 * BinaryBayesGridCell::Update calls the CPU would have made.  The one-map calls (integrate_scans,
 * _submit) are lgs_grid_integrate_many's code with one map; they refuse (LGS_ERR_INVALID) a windowed
 * grid and a grid on another device, and a call without scans returns LGS_OK before any grid check. */
typedef struct lgs_hit_batch {
    int n_scans;
    const double* sensor_xy;    /* [n_scans][2]           */
    const int* hit_begin;       /* [n_scans + 1]          */
    const double* hit_xy;       /* [hit_begin[n_scans]][2] */
} lgs_hit_batch;
int lgs_grid_integrate_scans(lgs_ctx* ctx, lgs_grid* grid, const lgs_hit_batch* scans,
                             double p_hit, double p_miss, long long* n_updates);
/* The same call in two halves, for a caller that streams scans (config C3): submit returns once the
 * call's work is queued (it waits only for the pre-pass that bounds the scans, and fails before anything
 * touches the grid if a scan leaves it); wait returns the update count of the OLDEST submitted call.  Up
 * to two calls may be in flight: the host-to-device copy and the pre-pass of call k + 1 then run under
 * the passes of call k (staging is double buffered).  The host arrays of a call must stay valid until
 * submit returns; cells are folded in submission order.  The grid is defined again -- for downloads,
 * matchers, resizes, copies -- once every submitted call has been waited for. */
int lgs_grid_integrate_submit(lgs_ctx* ctx, lgs_grid* grid, const lgs_hit_batch* scans,
                              double p_hit, double p_miss);
int lgs_grid_integrate_wait(lgs_ctx* ctx, long long* n_updates);
/* Many maps in one synchronous call: scans[i] into grids[i], i < n_maps -- every cell and n_updates[i]
 * (optional) exactly as n_maps calls of lgs_grid_integrate_scans would leave them.  The rebuild after a
 * loop closure (GridMapBuilder::AfterLoopClosure, grid_map_builder.cpp:62-80: every local map again from
 * its corrected poses) is the intended caller -- GridMapBuilderCuda::AfterLoopClosure.  One staging copy,
 * one pre-pass and one host sync for the whole call; a round of launches takes the next chunk of <= 64
 * scans of every map, so maps of <= 64 scans cost a constant number of launches however many there are.
 * All or nothing: if any scan of any map touches a cell outside its grid, the call fails with
 * LGS_ERR_INVALID naming the map and the scan before any grid is written.  Grids may differ in size,
 * resolution and apron and may belong to other contexts of the same device (ordered like lgs_grid_copy);
 * maps without scans and scans without hits are allowed.  Refused (LGS_ERR_INVALID): a grid twice, a
 * windowed grid, a grid on another device, and a call while a submitted integration on `ctx` has not
 * been waited for. */
int lgs_grid_integrate_many(lgs_ctx* ctx, int n_maps, lgs_grid* const* grids,
                            const lgs_hit_batch* scans, double p_hit, double p_miss,
                            long long* n_updates);

/* Diagnostics: cells (cumulative over this context) whose fast candidate search disagreed with
 * the mark pass and were redone by the exhaustive exact path; expected to stay 0. */
long long lgs_ctx_integrate_fallback_cells(const lgs_ctx* ctx);

/* Host helpers (glibc arithmetic, no device work) for callers that do not link the reference:
 * range filter + HitPoint + bounding box of one scan; GridMap::Resize / Expand geometry. */
typedef struct lgs_geometry {
    int nx, ny;                 /* cells (multiples of patch) */
    double min_x, min_y, res;
    int patch;                  /* cells per patch side       */
} lgs_geometry;

/* GridMapBuilder::ConstructMapFromScans (grid_map_builder.cpp:227-332) for many maps in one synchronous call,
 * from raw scans.  Map i: scans[i] holds its nodes' scans in node order, sensor_pose[k] = Compound(node pose,
 * RelativeSensorPose()), range_min[k] / range_max[k] = max(UsableRangeMin, MinRange()) / min(UsableRangeMax,
 * MaxRange()) (both arrays required).  A beam is used unless r >= range_max or r <= range_min (:365-366); its hit
 * is HitPoint's.  The bbox covers every hit and sensor position, from min = DBL_MAX and max = DBL_MIN (:236-237);
 * the new geometry is lgs_geometry_resize(cur[i], bbox) -- cur[i] is the map's current geometry, whose origin
 * anchors the patch lattice (a fresh map: 0 x 0 cells at its anchor) -- and grids[i] takes it with every cell
 * unknown (Resize + Reset) before every hit is integrated as lgs_grid_integrate_many would.  geometry_out[i],
 * bbox_out[i] = {min_x, min_y, max_x, max_y} (optional) and n_updates[i] (optional) return what was used.
 * Every cell, geometry and bbox is bit-identical to lgs_scan_hit_points per scan, then the bbox, then
 * lgs_geometry_resize, then lgs_grid_integrate_many: beams are projected on the device with an interval that
 * contains glibc's cos / sin ("integ_resolve_ulps"), and the few hits that interval cannot settle -- near a
 * cell edge, or possibly a bbox extreme -- are re-derived on the host (lgs_ctx_construct_host_points).  The
 * extra launches do not depend on n_maps.  Intended callers: GridMapBuilderCuda::AfterLoopClosure (every local
 * map plus the latest map in one call), UpdateLatestMap and ConstructGlobalMap.  Refused (LGS_ERR_INVALID)
 * before any grid changes: the refusals of lgs_grid_integrate_many, a map without scans, NULL range arrays,
 * a non-finite sensor pose or range window, and a non-finite angle or range on a beam that is used. */
struct lgs_scan_batch;          /* defined with the scans below */
int lgs_grid_construct_many(lgs_ctx* ctx, int n_maps, lgs_grid* const* grids,
                            const struct lgs_scan_batch* scans, const lgs_geometry* cur,
                            double p_hit, double p_miss, lgs_geometry* geometry_out,
                            double* bbox_out, long long* n_updates);
/* Points lgs_grid_construct_many re-derived on the host (cumulative over this context): bbox candidates
 * and near-edge hits. */
int lgs_ctx_construct_host_points(const lgs_ctx* ctx, long long* bbox_points, long long* edge_points);
int lgs_scan_hit_points(const double* sensor_pose, int n, const double* angles,
                        const double* ranges, double range_min, double range_max,
                        double* hit_xy, int* n_hit, double* bbox);
int lgs_geometry_resize(const lgs_geometry* cur, double min_x, double min_y, double max_x,
                        double max_y, lgs_geometry* out, int* shift_x, int* shift_y);
int lgs_geometry_expand(const lgs_geometry* cur, double min_x, double min_y, double max_x,
                        double max_y, double enlarge_step, lgs_geometry* out, int* shift_x,
                        int* shift_y, int* changed);

/* ---- sliding-window-max precompute ---------------------------------------------------------
 * out(x,y) = max grid[xs..xs+w) x [ys..ys+w), xs = min(x, max(nx-w, 0)) (the reference repeats
 * the last full window at the upper edges).  `out` must have the geometry of `in`. */
int lgs_precompute(lgs_ctx* ctx, const lgs_grid* in, int win, lgs_grid* out);
/* Levels 0..height_max with windows 1, 2, ..., 2^height_max (PrecomputeGridMaps):
 * lgs_pyramid_create_many with one grid. */
int lgs_pyramid_create(lgs_ctx* ctx, const lgs_grid* in, int height_max, lgs_pyramid** out);
/* The pyramids of n grids at once: out[i] is an ordinary pyramid of grids[i] (its own slab, freed by
 * lgs_pyramid_destroy), level by level identical to a build of grids[i] alone.  The apron clear, the
 * level-0 copy and each doubling level are one launch over all grids, so the launch count (height_max + 2)
 * does not depend on n.  The loop detector's pyramid cache, refilled after every loop closure, is the
 * intended caller.  Grids may belong to other contexts of the same device; a grid on another device is
 * refused (LGS_ERR_INVALID).  If an allocation fails, everything made so far is released, out[] is all
 * NULL and the call returns LGS_ERR_NOMEM. */
int lgs_pyramid_create_many(lgs_ctx* ctx, int n, const lgs_grid* const* grids, int height_max,
                            lgs_pyramid** out);
int lgs_pyramid_destroy(lgs_pyramid* p);
int lgs_pyramid_download(const lgs_pyramid* p, int level, double* dense);
int lgs_pyramid_levels(const lgs_pyramid* p);

/* ---- scans -------------------------------------------------------------------------------- */
typedef struct lgs_scan_batch {
    int n_scans;
    const int* beam_begin;      /* [n_scans + 1] offsets into angles / ranges              */
    const double* angles;       /* ScanData::Angles()                                       */
    const double* ranges;       /* ScanData::Ranges()                                       */
    const double* sensor_pose;  /* [n_scans][3] Compound(initialPose, RelativeSensorPose()) */
    const double* range_min;    /* [n_scans] ScanData::MinRange(), NULL = 0 (branch-and-bound only) */
    const double* range_max;    /* [n_scans] ScanData::MaxRange(), NULL = +inf                      */
} lgs_scan_batch;

typedef struct lgs_match_result {
    int found;                  /* scoreMax > scoreThreshold                               */
    int ix, iy, it;             /* bestWinX / bestWinY / bestWinTheta                      */
    int win_x, win_y, win_t;    /* window half sizes derived like the reference            */
    int n_fixups;               /* projected points re-derived on the host (near cell edge)*/
    double step_x, step_y, step_t;
    double score;               /* scoreMax (un-normalised sum), = threshold if !found     */
    long long n_scored;         /* hypotheses / nodes actually summed on the device        */
    int exact_replay;           /* 1 if the sequential CPU-order replay decided the winner */
    int reserved;
} lgs_match_result;

/* ---- real-time correlative matcher ------------------------------------------------------ */
typedef struct lgs_rtcsm_params {
    int low_res;                /* mLowResolution  */
    double range_x, range_y;    /* mRangeX, mRangeY (metres) */
    double range_theta;         /* mRangeTheta (radians)     */
    double scan_range_max;      /* mScanRangeMax             */
} lgs_rtcsm_params;

/* A batch object owns the device copies of the scans and all scratch (projected indices,
 * score tables).  upload = host prep + H2D; run = kernels only (asynchronous on the context
 * stream, inputs resident); results = D2H of the result records (+ rare host fix-ups). */
int lgs_rtcsm_batch_create(lgs_ctx* ctx, const lgs_rtcsm_params* params, lgs_rtcsm_batch** out);
int lgs_rtcsm_batch_destroy(lgs_rtcsm_batch* b);
/* norm_threshold: [n_scans] normalised score thresholds, or NULL for DBL_MIN (the 1-argument
 * OptimizePose overload).  `grid` supplies the geometry the window is derived from. */
int lgs_rtcsm_batch_upload(lgs_rtcsm_batch* b, const lgs_grid* grid, const lgs_scan_batch* scans,
                           const double* norm_threshold);
int lgs_rtcsm_batch_run(lgs_rtcsm_batch* b, const lgs_grid* grid, const lgs_grid* coarse);
/* Windows of >= 512 hypotheses are scored exactly but not exhaustively: every coarse hypothesis, then only
 * the fine tiles whose coarse scores can still reach the match's best fine score (the reference scores a
 * fine block only when its coarse score beats the running best).  This needs `coarse` to be
 * lgs_precompute(grid, low_res) of `grid`, as the reference's precomputed map is.
 * Same as run, but brackets the stages with CUDA events and waits:
 * ms[0] = projection, ms[1] = scoring (coarse scores, bound, work list, fine scores), ms[2] = selection. */
int lgs_rtcsm_batch_run_timed(lgs_rtcsm_batch* b, const lgs_grid* grid, const lgs_grid* coarse,
                              float* ms);
int lgs_rtcsm_batch_results(lgs_rtcsm_batch* b, const lgs_grid* grid, const lgs_grid* coarse,
                            lgs_match_result* out);
/* Test/diagnostic access to the per-match scratch of scan `m` after a run:
 * fine[nT][nyw][nxw], coarse[nT][nbx][nby], cells[nT][nKept][2] (projected cell indices,
 * un-clamped), dims = {nT, nxw, nyw, nbx, nby, nKept}.  Any pointer may be NULL.
 * After a pruned run, the first call that asks for `fine` or `coarse` scores the whole batch again with
 * the exhaustive sweep against the grids of that run, which must still exist unchanged, and waits for it
 * (about the time of a run without pruning); later calls only copy. */
int lgs_rtcsm_batch_debug(lgs_rtcsm_batch* b, int m, int* dims, double* fine, double* coarse,
                          int* cells);
/* Algorithmic work of the last upload: hypotheses (fine + coarse) and gathered cells.  These count
 * every hypothesis of each window, the window the result is exact over, also where the run prunes. */
int lgs_rtcsm_batch_work(const lgs_rtcsm_batch* b, long long* hypotheses, long long* gathers);
/* Diagnostic: fine tiles the last scoring pass of run (or of results' re-scoring) summed, and the tiles
 * of the exhaustive sweep.  A tile is one warp's share of the row sweep: up to 32 x offsets, 4-5 window
 * rows, 2 theta slices.  Windows of the flattened sweep (< 512 hypotheses) are never pruned; for them
 * both counts are that sweep's warps.  Waits for the stream. */
int lgs_rtcsm_batch_fine_tiles(lgs_rtcsm_batch* b, long long* scored, long long* total);
/* Convenience: upload + run + results. */
int lgs_rtcsm_match(lgs_ctx* ctx, const lgs_grid* grid, const lgs_grid* coarse,
                    const lgs_rtcsm_params* params, const lgs_scan_batch* scans,
                    const double* norm_threshold, lgs_match_result* out);

/* ---- branch-and-bound matcher (loop detection) ------------------------------------------------
 * One query = (scan, sensor pose, submap pyramid).  All queries of a batch are searched
 * breadth-first, level by level, together. */
typedef struct lgs_bb_params {
    int node_height_max;            /* mNodeHeightMax (pyramids need levels 0..node_height_max) */
    double range_x, range_y;        /* mRangeX, mRangeY (metres) */
    double range_theta;             /* mRangeTheta (radians)     */
    double scan_range_max;          /* mScanRangeMax             */
    double score_range_min;         /* ScorePixelAccurate::mUsableRangeMin */
    double score_range_max;         /* ScorePixelAccurate::mUsableRangeMax */
} lgs_bb_params;

int lgs_bb_batch_create(lgs_ctx* ctx, const lgs_bb_params* params, lgs_bb_batch** out);
int lgs_bb_batch_destroy(lgs_bb_batch* b);
/* scans->n_scans queries; pyramids[q] is the submap query q is matched against (pyramids may
 * repeat); norm_threshold[q] as for the correlative matcher.
 * Precondition of the device-only run: the cells of the submaps are occupancy probabilities, 0 (unknown)
 * or within (0, 1] -- the reference's BinaryBayesGridCell values are clamped to [0.001, 0.999].  The run
 * stops a node's sum once `partial + remaining beams <= threshold` ("bb_early_reject", default on); for
 * grids with larger values switch the option off (lgs_ctx_set_option) or take the exact path ("bb_sync"). */
int lgs_bb_batch_upload(lgs_bb_batch* b, const lgs_scan_batch* scans,
                        lgs_pyramid* const* pyramids, const double* norm_threshold);
/* Same, for scans shared by several queries: pair q matches scans[pair_scan[q]] against
 * pyramids[q]; the scan is projected once (config C4: 1 scan x 500 submaps). */
int lgs_bb_batch_upload_pairs(lgs_bb_batch* b, const lgs_scan_batch* scans, int n_pairs,
                              const int* pair_scan, lgs_pyramid* const* pyramids,
                              const double* norm_threshold);
/* Asynchronous: ONE persistent kernel launch on the context stream (hit points, all tree levels with
 * device-side node counts, winner, verification / CPU-order replay, result records); nothing comes
 * back to the host until results / records / settle. */
int lgs_bb_batch_run(lgs_bb_batch* b);
/* Waits for the run.  A run that met a near-edge point the device could not decide, or a node pool
 * that was too small, is transparently repeated on the level-synchronous exact path (host-computed
 * index tables for the near-edge points) before anything is returned. */
int lgs_bb_batch_results(lgs_bb_batch* b, lgs_match_result* out);
/* The exchange format of loop detection (SURVEY.md 8(e)): one 32-byte record per (scan, submap) pair.
 * Replaces the per-pair outcome of LoopDetectorBranchBound::Detect's inner loop
 * (mapping/loop_detector_branch_bound.cpp:63-88) before the host tail. */
typedef struct lgs_loop_record {
    int found;                  /* scoreMax > scoreThreshold */
    int ix, iy, it;             /* bestWinX / bestWinY / bestWinTheta */
    double score;               /* scoreMax, = threshold if !found */
    long long id;               /* caller's pair id (lgs_bb_batch_set_record_ids), default: index in the batch */
} lgs_loop_record;
/* ids[q] is copied into record q by the finalize phase of every later run; takes effect with the
 * next upload, whose pair count must equal n (n = 0 restores the default). */
int lgs_bb_batch_set_record_ids(lgs_bb_batch* b, const long long* ids, int n);
/* Device-side record sink: the finalize phase of every later run stores record q at
 * device_records[first_slot + q].  The pointer may be memory of ANOTHER GPU mapped into this device
 * (peer access): the records then cross NVLink as plain stores from the kernel itself, with no host
 * staging and no separate copy.  NULL restores the batch's own buffer.  The caller orders its reads
 * after the run (lgs_bb_batch_settle / lgs_ctx_synchronize).  One STATUS record follows the batch's
 * records, at device_records[first_slot + n_pairs] (so the sink needs room for n_pairs + 1): id = -1,
 * found = 1 if the run stands, -1 if it has to be repeated on the exact path (lgs_bb_batch_settle does
 * that and rewrites records and status) -- ranks that only see the exchanged buffer learn it from there. */
int lgs_bb_batch_set_record_sink(lgs_bb_batch* b, lgs_loop_record* device_records, long long first_slot);
int lgs_bb_batch_records(lgs_bb_batch* b, lgs_loop_record* out);    /* host copy of the records, waits */
int lgs_bb_batch_settle(lgs_bb_batch* b);    /* wait + validate (+ exact repeat) without copying results out */
void* lgs_bb_batch_device_records(lgs_bb_batch* b);                 /* the batch's own device record buffer */
/* Diagnostic (option "bb_host_timing" on before the run): microseconds spent in the phases of the last
 * device-only run -- [0] hit points, [1] root level, [2 ..] levels H-1 .. 0, then winner, finalize --
 * and (optional) the lanes-per-node mapping the scoring phases used. */
int lgs_bb_batch_phase_times(lgs_bb_batch* b, double* us, int* mapping, int n);
/* Beams the last device-only run left out through early rejection ("bb_early_reject": a node whose
 * partial sum plus one per remaining beam cannot exceed its threshold is pruned by the CPU whatever the
 * rest of its sum is; grid cells are probabilities <= 1).  lgs_bb_batch_work counts every beam of every
 * node -- the reference's cost; the difference was actually gathered. */
long long lgs_bb_batch_skipped_gathers(const lgs_bb_batch* b);
/* With the context option "bb_count_nodes" (or "bb_host_timing") on: nodes[q] = nodes below the root
 * level scored for query q by the last device-only run (n >= queries of the batch) -- the per-submap
 * cost a placement can balance; lgs_match_result::n_scored is then per query too (roots + these). */
int lgs_bb_batch_query_nodes(lgs_bb_batch* b, long long* nodes, int n);
/* How many runs of this batch object were device-only and how many went through the exact path. */
int lgs_bb_batch_path(const lgs_bb_batch* b, long long* device_runs, long long* exact_runs);
/* Nodes scored per tree level (index = height) and gathered cells during the last run. */
int lgs_bb_batch_work(const lgs_bb_batch* b, long long* nodes_per_level, int n_levels,
                      long long* gathers);
/* Test hook: force the sequential CPU-order replay for every query of the next runs. */
int lgs_bb_batch_force_replay(lgs_bb_batch* b, int on);
/* Convenience: upload + run + results. */
int lgs_bb_match(lgs_ctx* ctx, const lgs_bb_params* params, const lgs_scan_batch* scans,
                 lgs_pyramid* const* pyramids, const double* norm_threshold,
                 lgs_match_result* out);

/* ---- loop detection across the GPUs of one box (SURVEY.md 8(e)) ---------------------------------------
 * LoopDetectorBranchBound::Detect's pair loop (mapping/loop_detector_branch_bound.cpp:38-90) carries
 * nothing from one (node, local map) pair to the next, so the pairs shard by the submap they name.
 *
 * lgs_group: ONE process drives all devices -- one lgs_ctx and one persistent host thread per device,
 * peer access between all members.  Build the grids / pyramids of submap i with lgs_group_ctx(g, i % G);
 * lgs_group_bb_detect then runs every pair on the device that holds its pyramid (one persistent kernel
 * per member, all members concurrently) and each member's kernel stores its 32-byte records straight
 * into the root device's gather buffer over NVLink (peer stores, no host staging); one device -> host
 * copy returns them.  Results are in pair order and identical to a single-device lgs_bb_batch run. */
typedef struct lgs_group lgs_group;
typedef struct lgs_group_bb lgs_group_bb;
int lgs_group_create(const int* devices, int n, lgs_group** out);
int lgs_group_destroy(lgs_group* g);
int lgs_group_size(const lgs_group* g);
lgs_ctx* lgs_group_ctx(lgs_group* g, int member);
const char* lgs_group_last_error(const lgs_group* g);
int lgs_group_bb_create(lgs_group* g, const lgs_bb_params* params, lgs_group_bb** out);
int lgs_group_bb_destroy(lgs_group_bb* d);
int lgs_group_bb_detect(lgs_group_bb* d, const lgs_scan_batch* scans, int n_pairs, const int* pair_scan,
                        lgs_pyramid* const* pyramids, const double* norm_threshold, lgs_match_result* out);
int lgs_group_bb_records(const lgs_group_bb* d, lgs_loop_record* out);   /* the exchanged records, pair order */

/* lgs_comm: one process PER device (torchrun-style launch).  An all-gather of fixed-size loop records
 * on the context stream, device to device, through NCCL (libnccl.so.2 is resolved at run time).  Rank 0
 * creates the 128-byte id and hands it to the others over any host channel.  With send_device == NULL the
 * all-gather runs IN PLACE: rank r's records are expected in its own slice recv_device[r * count ..), which
 * is where a batch whose sink is (recv_device, r * count) has written them. */
typedef struct lgs_comm lgs_comm;
int lgs_comm_unique_id(void* id128);
int lgs_comm_create(lgs_ctx* ctx, int world, int rank, const void* id128, lgs_comm** out);
int lgs_comm_destroy(lgs_comm* c);
int lgs_comm_all_gather_records(lgs_comm* c, const void* send_device, void* recv_device, int count);

/* ---- exhaustive grid-search matcher ------------------------------------------------------------
 * Replaces ScanMatcherGridSearch::OptimizePose (scan_matcher_grid_search.cpp:45-114) with
 * ScorePixelAccurate::Score (score_function_pixel_accurate.cpp:19-76), the matcher behind
 * LoopDetectorGridSearch (loop_detector_grid_search.cpp:26-118).  Offsets are ACCUMULATED like the
 * reference's loops (`for (d = -range / 2; d <= range / 2; d += step)`), visit order y, x, theta,
 * first strictly greater score wins.  Winner and score are bit-identical to the CPU code. */
typedef struct lgs_gs_params {
    double range_x, range_y, range_theta;   /* mRangeX, mRangeY, mRangeTheta */
    double step_x, step_y, step_theta;      /* mStepX, mStepY, mStepTheta    */
    double score_range_min;                 /* ScorePixelAccurate::mUsableRangeMin */
    double score_range_max;                 /* ScorePixelAccurate::mUsableRangeMax */
} lgs_gs_params;
/* Query q = scan q of the batch (sensor_pose = Compound(initialPose, RelativeSensorPose())) against
 * grids[q].  Results: found, ix / iy / it = LOOP COUNTERS of the winning dx / dy / dt (-1 if not
 * found), win_x / win_y / win_t = the three loop lengths, score = winning score.  The winning offset
 * itself is lgs_gs_offsets(...)[counter]; the pose is sensor_pose + offset.  score_table (optional,
 * one query only): [win_t][win_y][win_x] scores of every hypothesis. */
int lgs_gs_match(lgs_ctx* ctx, const lgs_gs_params* params, const lgs_scan_batch* scans,
                 const lgs_grid* const* grids, const double* norm_threshold, lgs_match_result* out,
                 double* score_table);
/* The offsets the reference's accumulating loop visits for (range, step): n values, the first
 * min(n, cap) written to out (may be NULL).  Host arithmetic only. */
int lgs_gs_offsets(double range, double step, double* out, int cap, int* n);

/* ---- CostGreedyEndpoint: the tail both matchers run on the winning pose ------------------------
 * Replaces CostGreedyEndpoint::Cost / ComputeGradient / ComputeCovariance
 * (cost_function_greedy_endpoint.cpp:32-171) as called from
 * scan_matcher_real_time_correlative.cpp:126-138 and scan_matcher_branch_bound.cpp:143-162.
 * Fields are the constructor's arguments in the constructor's meaning
 * (cost_function_greedy_endpoint.hpp:19-25; note that slam_launcher.cpp:70-72 passes
 * StandardDeviation and ScalingFactor swapped -- a caller that wants the launcher's behaviour swaps
 * them the same way).  Results are bit-identical to the CPU code. */
typedef struct lgs_cost_params {
    double usable_range_min, usable_range_max;
    double hit_and_missed_dist;
    double occupancy_threshold;
    int kernel_size;                /* 0..7 */
    double scaling_factor;
    double standard_deviation;
} lgs_cost_params;
/* Cost() of n_poses sensor poses (poses[n_poses][3]); pose p uses scan pose_scan[p] of the batch
 * (NULL: n_poses == n_scans, pose p uses scan p).  scans->sensor_pose is not read; range_min /
 * range_max are ScanData::MinRange / MaxRange.  n_fixups (optional): near-edge beams re-derived
 * on the host. */
int lgs_cost_greedy_endpoint(lgs_ctx* ctx, const lgs_grid* grid, const lgs_cost_params* params,
                             const lgs_scan_batch* scans, int n_poses, const int* pose_scan,
                             const double* poses, double* cost, int* n_fixups);
/* The whole tail for one best sensor pose per scan (best_sensor_pose[n_scans][3]):
 * normalized_cost[m] = Cost / NumOfScans, covariance[m][9] = row-major ComputeCovariance.
 * Either output may be NULL. */
int lgs_cost_tail(lgs_ctx* ctx, const lgs_grid* grid, const lgs_cost_params* params,
                  const lgs_scan_batch* scans, const double* best_sensor_pose,
                  double* normalized_cost, double* covariance, int* n_fixups);

#ifdef __cplusplus
}
#endif
#endif /* LGS_B200_H */
