// lgs_csm.cu -- real-time correlative scan matcher on sm_100a.
//
// Replaces ScanMatcherRealTimeCorrelative::OptimizePose(grid, coarse, scan, pose, thr)
// (mapping/scan_matcher_real_time_correlative.cpp:50-145) and its helpers ComputeSearchStep
// (:156-175), ComputeScanIndices (:178-203), ComputeScore (:207-224) and
// EvaluateHighResolutionMap (:227-256).
//
// Exactness strategy (SURVEY.md H1, H2, H5, H6, H12):
//  * csm_project_kernel projects every kept beam once per theta with the reference's exact
//    operation order (IEEE add/mul/div intrinsics, never fused).  Only sin/cos can differ from
//    glibc by an ulp, which can change floor() only within the edge guard band of a cell edge; such
//    points are flagged and re-derived on the host with glibc before the result is accepted.
//  * the sweep (csm_sweep_rows_kernel: lanes = the x offsets of one window row, 4-5 rows of
//    kThetaGroup theta slices per thread; csm_sweep_kernel: one thread per hypothesis, for small
//    windows) sums the gathered cells of every hypothesis in beam order in double: the score is
//    bit-identical to the CPU loop by construction, so no epsilon logic is needed anywhere.
//  * csm_select_kernel computes each coarse block's fine maximum with first-visit argmax and
//    then reproduces the CPU's pruned visit sequence: a parallel (score desc, visit asc)
//    reduction when every coarse score bounds its block, otherwise a sequential replay of
//    `if (C[b] > best && F[b] > best) best = F[b]` in the CPU's visit order.
//
// Data layout: projected points are stored per (match, theta) as int32 offsets into the
// apron-padded grid, clamped so that every out-of-map read lands in the zero apron; the sweep
// stages the offsets of its theta slice(s) in shared memory and each thread gathers
// grid[base + off[i]].
#include <cfloat>
#include <cmath>

#include "lgs_internal.cuh"

namespace {

constexpr int kBeamPad = 8;          // kept-beam count is padded to a multiple of this
constexpr int kFlagCap = 1 << 16;    // initial capacity of the near-edge fix-up list (grown on demand)
constexpr int kThetaGroup = 2;       // row-mapped sweep: theta slices per thread (profiles/r3_csm_theta_reuse.md)
constexpr int kRowsUnroll = 4;       // row-mapped sweep: beams per loop iteration

struct CsmDesc {
    double sx, sy, st;       // sensor pose
    double stepT;            // angular step
    double thrAbs;           // normalizedScoreThreshold * NumOfScans()
    int winT, nT;            // theta half window, 2 * winT + 1
    int nKept, nKeptPad;     // beams with range < scanRangeMax
    int beamBegin;           // into the kept angle / range arrays
    int pad0;
    long long offBegin;      // into offs  : nT * nKeptPad
    long long cellBegin;     // into cells : nT * nKept (int2)
    long long fineBegin;     // into fine table   : nT * nyw * nxw
    long long coarseBegin;   // into coarse table : nT * nbx * nby
};

struct CsmWindow {           // identical for every match of a batch (depends on grid + params)
    int winX, winY;
    int nbx, nby;            // coarse blocks per axis
    int nxw, nyw;            // fine hypotheses per axis = nb * lowRes
    int lowRes;
    int tilesFine, tilesCoarse;   // thread blocks per theta
    int block;               // threads per block
    int hpt;                 // fine hypotheses per thread (1 or 4)
    int slots;               // thread slots per theta = ceil(nHyp / hpt) rounded up to a warp
    int rows;                // > 0: row-mapped sweep, fine rows per thread (4 or 5)
    int xChunks, rowGroups;  // warps per theta = xChunks * rowGroups (lanes = 32 consecutive x)
};

struct GridGeom {
    double minX, minY, res;
    int nx, ny, pitch;
};

struct DevResult {
    double score;
    int found, ix, iy, it;
    int exactReplay;
    int needFull;            // pruned select found a coarse score below its block: score every tile again
};

struct FlagEntry { int m, t, i; };

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// ---- K1: scan projection ----------------------------------------------------------------------
// One thread per (match, theta, kept beam).  scan_matcher_real_time_correlative.cpp:88-96,
// :178-203; sensor_data.hpp:162-173; grid_map.hpp:779-790.
__global__ void csm_project_kernel(const CsmDesc* __restrict__ descs,
                                   const double* __restrict__ angles,
                                   const double* __restrict__ ranges, GridGeom g, CsmWindow w, double eps,
                                   int* __restrict__ offs, int2* __restrict__ cells,
                                   FlagEntry* __restrict__ flags, int flagCap, int* __restrict__ flagCount,
                                   int* __restrict__ noBound) {
    const CsmDesc d = descs[blockIdx.y];
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)d.nT * d.nKeptPad) return;
    const int t = (int)(idx / d.nKeptPad);
    const int i = (int)(idx - (long long)t * d.nKeptPad);
    // Clamp targets: every window offset of a clamped point reads the zero apron.
    const int xLo = -w.winX, xHi = -w.winX + w.nxw - 1;
    const int yLo = -w.winY, yHi = -w.winY + w.nyw - 1;
    if (i >= d.nKept) {   // padding beam: contributes exactly +0.0
        offs[d.offBegin + idx] = (-yHi - 1) * g.pitch + (-xHi - 1);
        return;
    }
    const double theta = __dadd_rn(d.st, __dmul_rn(d.stepT, (double)(t - d.winT)));
    const double a = __dadd_rn(theta, angles[d.beamBegin + i]);
    double s, c;
    sincos(a, &s, &c);
    const double r = ranges[d.beamBegin + i];
    const double hx = __dadd_rn(d.sx, __dmul_rn(r, c));
    const double hy = __dadd_rn(d.sy, __dmul_rn(r, s));
    const double qx = __ddiv_rn(__dsub_rn(hx, g.minX), g.res);
    const double qy = __ddiv_rn(__dsub_rn(hy, g.minY), g.res);
    const double fx = floor(qx), fy = floor(qy);
    const double rx = qx - fx, ry = qy - fy;
    const bool edge = !(rx >= eps && rx <= 1.0 - eps && ry >= eps && ry <= 1.0 - eps);
    if (edge) {
        const int k = atomicAdd(flagCount, 1);
        if (k < flagCap) flags[k] = FlagEntry{(int)blockIdx.y, t, i};
    }
    const int cx = __double2int_rd(qx), cy = __double2int_rd(qy);
    cells[d.cellBegin + (long long)t * d.nKept + i] = make_int2(cx, cy);
    const int ccx = clampi(cx, -xHi - 1, g.nx - xLo);
    const int ccy = clampi(cy, -yHi - 1, g.ny - yLo);
    offs[d.offBegin + idx] = ccy * g.pitch + ccx;
    // "coarse may not bound" (K2c): a coarse read of this point in (-lowRes, 0) on either axis
    const int e = edge ? 1 : 0;
    bool band = false;
    for (int c = -e; c <= e; ++c) {
        for (int bx = 0; bx < w.nbx; ++bx) {
            const int rx = ccx + c - w.winX + bx * w.lowRes;
            band |= rx > -w.lowRes && rx < 0;
        }
        for (int by = 0; by < w.nby; ++by) {
            const int ry = ccy + c - w.winY + by * w.lowRes;
            band |= ry > -w.lowRes && ry < 0;
        }
    }
    if (band) noBound[blockIdx.y] = 1;
}

// ---- K2: the sweep (hot kernel) -------------------------------------------------------------------
// grid = (tilesFine + tilesCoarse, maxNT, matches).  One thread per hypothesis; the theta's
// offsets are staged in shared memory; each thread sums grid[base + off[i]] in beam order.
// Lanes are consecutive x offsets so a warp's gathers for one beam fall in 1-3 cache lines.
// scan_matcher_real_time_correlative.cpp:98-102 (coarse), :207-224, :239-244 (fine).
template <int UNROLL, int HPT>
__global__ void __launch_bounds__(256)
csm_sweep_kernel(const CsmDesc* __restrict__ descs, const double* __restrict__ fineGrid,
                 const double* __restrict__ coarseGrid, int pitch, CsmWindow w,
                 const int* __restrict__ offs, double* __restrict__ fineTab,
                 double* __restrict__ coarseTab) {
    extern __shared__ int sOff[];
    const CsmDesc d = descs[blockIdx.z];
    const int t = blockIdx.y;
    if (t >= d.nT) return;
    {   // stage this theta's offsets (nKeptPad is a multiple of 4 ints = 16 B)
        const int4* src = reinterpret_cast<const int4*>(offs + d.offBegin + (long long)t * d.nKeptPad);
        int4* dst = reinterpret_cast<int4*>(sOff);
        for (int k = threadIdx.x; k < d.nKeptPad / 4; k += blockDim.x) dst[k] = src[k];
    }
    __syncthreads();
    const int n = d.nKeptPad;   // multiple of kBeamPad >= UNROLL

    if (blockIdx.x >= (unsigned)w.tilesFine) {
        // Coarse hypotheses (stride lowRes on the win-max map), one per thread.
        const int h = (blockIdx.x - w.tilesFine) * blockDim.x + threadIdx.x;
        if (h >= w.nbx * w.nby) return;
        const int oy = h / w.nbx, ox = h - oy * w.nbx;
        const double* __restrict__ gp =
            coarseGrid + (-w.winY + oy * w.lowRes) * pitch + (-w.winX + ox * w.lowRes);
        double acc = 0.0;
#pragma unroll 1
        for (int i = 0; i < n; i += UNROLL) {
            double v[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) v[u] = __ldg(gp + sOff[i + u]);
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) acc = __dadd_rn(acc, v[u]);
        }
        // stored in the CPU's visit order: x outer, y inner
        coarseTab[d.coarseBegin + ((long long)t * w.nbx + ox) * w.nby + oy] = acc;
        return;
    }

    // Fine hypotheses: thread slot j owns hypotheses j, j + S, ..., j + (HPT-1) S of the flattened
    // (y, x) window, so one shared-memory offset load feeds HPT gathers and a warp's lanes stay
    // on consecutive x cells for every one of them.
    const int nHyp = w.nxw * w.nyw;
    const int S = w.slots;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= S) return;
    const double* __restrict__ gp[HPT];
    double acc[HPT];
#pragma unroll
    for (int k = 0; k < HPT; ++k) {
        const int h = min(j + k * S, nHyp - 1);          // out-of-range slots alias the last one
        const int oy = h / w.nxw, ox = h - oy * w.nxw;
        gp[k] = fineGrid + (-w.winY + oy) * pitch + (-w.winX + ox);
        acc[k] = 0.0;
    }
#pragma unroll 1
    for (int i = 0; i < n; i += UNROLL) {
        double v[UNROLL][HPT];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const int o = sOff[i + u];
#pragma unroll
            for (int k = 0; k < HPT; ++k) v[u][k] = __ldg(gp[k] + o);
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u)
#pragma unroll
            for (int k = 0; k < HPT; ++k) acc[k] = __dadd_rn(acc[k], v[u][k]);   // beam order, like the CPU
    }
#pragma unroll
    for (int k = 0; k < HPT; ++k) {
        const int h = j + k * S;
        if (h < nHyp) {
            const int oy = h / w.nxw, ox = h - oy * w.nxw;
            fineTab[d.fineBegin + ((long long)t * w.nyw + oy) * w.nxw + ox] = acc[k];
        }
    }
}

// ---- K2b: the sweep, row mapped and theta grouped ----------------------------------------------------
// Same arithmetic as csm_sweep_kernel, different ownership: a warp's lanes are the x offsets of ONE
// window row (25 of 32 lanes for config C2) and a thread owns ROWS consecutive rows of TG consecutive
// theta slices.  A 32-lane request touches the 2-3 cache lines of a single 25-cell row (2.5 L1
// wavefronts on average) instead of the 3.8 lines of 1.28 rows of the flattened mapping, and the L1
// data pipe is what bounds this kernel (profiles/r1_kernels_v2.md).
//
// Theta grouping gathers fewer bytes for the same sums.  Slices t and t + 1 differ by one angular step,
// so a beam usually projects to the same cell in both, or to the cell directly above or below.  The
// rows a thread gathered for slice t are then exactly the rows slice t + 1 needs, or the same rows
// shifted by one, and only the missing row is loaded (on C2: 0.67 of the loads at TG = 2, 0.50 at TG = 4).
// TG = 2 is the fastest measured: larger groups need more accumulator registers and lose more occupancy
// than they save in loads (profiles/r3_csm_theta_reuse.md).  Each decision compares two staged offsets of
// the same beam, which every lane of the block shares: the branches never diverge, and an equal address
// cannot give a different value.
// The adds stay acc[t][k] += v[k] in beam order, so every score is the one the CPU loop computes.
//
// Shared memory holds the group's offsets interleaved [beam][t]: one broadcast load per beam feeds all
// TG slices.  A slice past the match's nT (last group; matches of one batch can differ in nT) repeats
// the last valid slice's offsets, so it takes the equal-offset branch, loads nothing and is not stored.
template <int TG>
__device__ __forceinline__ void load_theta_group(const int* s, int (&o)[TG]) {
    if constexpr (TG % 4 == 0) {
#pragma unroll
        for (int q = 0; q < TG / 4; ++q) {
            const int4 v = reinterpret_cast<const int4*>(s)[q];
            o[4 * q] = v.x; o[4 * q + 1] = v.y; o[4 * q + 2] = v.z; o[4 * q + 3] = v.w;
        }
    } else if constexpr (TG == 2) {
        const int2 v = *reinterpret_cast<const int2*>(s);
        o[0] = v.x; o[1] = v.y;
    } else {
#pragma unroll
        for (int t = 0; t < TG; ++t) o[t] = s[t];
    }
}

// Stages the offsets of slices t0 .. t0 + TG of match d into s ([beam][TG]); threads tid of nthr take part.
template <int TG>
__device__ __forceinline__ void stage_theta_group(const CsmDesc& d, const int* __restrict__ offs, int t0, int nTg,
                                                  int* s, int tid, int nthr) {
    const int n4 = d.nKeptPad / 4;   // nKeptPad is a multiple of 4 ints = 16 B
    const int* src = offs + d.offBegin + (long long)t0 * d.nKeptPad;
    for (int k = tid; k < TG * n4; k += nthr) {
        const int t = k / n4, q = k - t * n4;
        const int4 v = reinterpret_cast<const int4*>(src + (long long)min(t, nTg - 1) * d.nKeptPad)[q];
        int* dst = s + 4 * q * TG + t;
        dst[0] = v.x; dst[TG] = v.y; dst[2 * TG] = v.z; dst[3 * TG] = v.w;
    }
}

// Coarse hypothesis h (stride lowRes on the win-max map) of TG slices, beams in order.  Only the equal-offset
// reuse applies: a thread holds a single row.
template <int UNROLL, int TG>
__device__ __forceinline__ void coarse_theta_group(const CsmDesc& d, const CsmWindow& w, const int* sOff,
                                                   const double* __restrict__ coarseGrid, int pitch, int h, int t0,
                                                   int nTg, double* __restrict__ coarseTab) {
    const int n = d.nKeptPad;   // multiple of kBeamPad >= UNROLL
    const int oy = h / w.nbx, ox = h - oy * w.nbx;
    const double* __restrict__ gp =
        coarseGrid + (-w.winY + oy * w.lowRes) * pitch + (-w.winX + ox * w.lowRes);
    double acc[TG];
#pragma unroll
    for (int t = 0; t < TG; ++t) acc[t] = 0.0;
#pragma unroll 1
    for (int i = 0; i < n; i += UNROLL) {
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            int o[TG];
            load_theta_group<TG>(sOff + (i + u) * TG, o);
            double v = __ldg(gp + o[0]);
            acc[0] = __dadd_rn(acc[0], v);
#pragma unroll
            for (int t = 1; t < TG; ++t) {
                if (o[t] != o[t - 1]) v = __ldg(gp + o[t]);
                acc[t] = __dadd_rn(acc[t], v);
            }
        }
    }
#pragma unroll
    for (int t = 0; t < TG; ++t)
        if (t < nTg) coarseTab[d.coarseBegin + ((long long)(t0 + t) * w.nbx + ox) * w.nby + oy] = acc[t];
}

// Fine rows of warp wg (x chunk wg % xChunks, row group wg / xChunks) of one theta group; lane = x in the chunk.
template <int UNROLL, int ROWS, int TG>
__device__ __forceinline__ void fine_theta_group(const CsmDesc& d, const CsmWindow& w, const int* sOff,
                                                 const double* __restrict__ fineGrid, int pitch, int wg, int lane,
                                                 int t0, int nTg, double* __restrict__ fineTab) {
    const int n = d.nKeptPad;   // multiple of kBeamPad >= UNROLL
    const int xc = wg % w.xChunks, rg = wg / w.xChunks;
    const int ox = xc * 32 + lane;
    if (rg >= w.rowGroups || ox >= w.nxw) return;
    const int oy0 = rg * ROWS;
    const double* __restrict__ gp = fineGrid + (-w.winY + oy0) * pitch + (-w.winX + ox);
    double acc[TG][ROWS];
#pragma unroll
    for (int t = 0; t < TG; ++t)
#pragma unroll
        for (int k = 0; k < ROWS; ++k) acc[t][k] = 0.0;
    const int nRows = min(ROWS, w.nyw - oy0);
    if (nRows == ROWS) {
        // the thread's ROWS window rows; row k of slice t is row[k] + o[t]
        const double* __restrict__ row[ROWS];
#pragma unroll
        for (int k = 0; k < ROWS; ++k) row[k] = gp + k * pitch;
#pragma unroll 1
        for (int i = 0; i < n; i += UNROLL) {
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                int o[TG];
                load_theta_group<TG>(sOff + (i + u) * TG, o);
                double v[ROWS];   // rows o[t] + k * pitch, k < ROWS, of the current slice
#pragma unroll
                for (int k = 0; k < ROWS; ++k) v[k] = __ldg(row[k] + o[0]);
#pragma unroll
                for (int k = 0; k < ROWS; ++k) acc[0][k] = __dadd_rn(acc[0][k], v[k]);   // beam order, like the CPU
#pragma unroll
                for (int t = 1; t < TG; ++t) {
                    if (o[t] == o[t - 1]) {
                        // same cell: all ROWS rows are already held
                    } else if (o[t] == o[t - 1] + pitch) {        // one row up the map: shift, load the top row
#pragma unroll
                        for (int k = 0; k < ROWS - 1; ++k) v[k] = v[k + 1];
                        v[ROWS - 1] = __ldg(row[ROWS - 1] + o[t]);
                    } else if (o[t] == o[t - 1] - pitch) {        // one row down: shift, load the bottom row
#pragma unroll
                        for (int k = ROWS - 1; k > 0; --k) v[k] = v[k - 1];
                        v[0] = __ldg(row[0] + o[t]);
                    } else {
#pragma unroll
                        for (int k = 0; k < ROWS; ++k) v[k] = __ldg(row[k] + o[t]);
                    }
#pragma unroll
                    for (int k = 0; k < ROWS; ++k) acc[t][k] = __dadd_rn(acc[t][k], v[k]);
                }
            }
        }
    } else {                                   // last row group of a window whose height is no multiple of ROWS
#pragma unroll 1
        for (int i = 0; i < n; ++i) {
#pragma unroll
            for (int t = 0; t < TG; ++t) {
                const double* __restrict__ q = gp + sOff[i * TG + t];
#pragma unroll
                for (int k = 0; k < ROWS; ++k)
                    if (k < nRows) acc[t][k] = __dadd_rn(acc[t][k], __ldg(q + k * pitch));
            }
        }
    }
#pragma unroll
    for (int t = 0; t < TG; ++t)
#pragma unroll
        for (int k = 0; k < ROWS; ++k)
            if (t < nTg && k < nRows)
                fineTab[d.fineBegin + ((long long)(t0 + t) * w.nyw + oy0 + k) * w.nxw + ox] = acc[t][k];
}

// The exhaustive row sweep: grid = (tilesFine + tilesCoarse, theta groups, matches).  It fills the whole fine
// and coarse tables; lgs_rtcsm_batch_debug runs it to return them after a pruned run.
template <int UNROLL, int ROWS, int TG>
__global__ void __launch_bounds__(256)
csm_sweep_rows_kernel(const CsmDesc* __restrict__ descs, const double* __restrict__ fineGrid,
                      const double* __restrict__ coarseGrid, int pitch, CsmWindow w,
                      const int* __restrict__ offs, double* __restrict__ fineTab,
                      double* __restrict__ coarseTab) {
    extern __shared__ int sOff[];   // [beam][TG]
    const CsmDesc d = descs[blockIdx.z];
    const int t0 = blockIdx.y * TG;
    if (t0 >= d.nT) return;
    const int nTg = min(TG, d.nT - t0);   // valid slices of this group
    stage_theta_group<TG>(d, offs, t0, nTg, sOff, threadIdx.x, blockDim.x);
    __syncthreads();
    if (blockIdx.x >= (unsigned)w.tilesFine) {
        const int h = (blockIdx.x - w.tilesFine) * blockDim.x + threadIdx.x;
        if (h < w.nbx * w.nby) coarse_theta_group<UNROLL, TG>(d, w, sOff, coarseGrid, pitch, h, t0, nTg, coarseTab);
        return;
    }
    fine_theta_group<UNROLL, ROWS, TG>(d, w, sOff, fineGrid, pitch, blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5),
                                       threadIdx.x & 31, t0, nTg, fineTab);
}

// ---- K2c: the pruned sweep of row-mapped windows ------------------------------------------------------
// The reference scores a fine block only when its coarse score beats the running best, so its answer depends
// only on blocks with C[b] >= F* (F* = the match's best fine score) whenever every coarse score bounds its
// block.  The device therefore scores every coarse hypothesis (csm_coarse_kernel), takes a lower bound L <= F*
// from the fine blocks of the kSeedBlocks best coarse blocks (csm_prune_kernel), and scores only the warp tiles
// (theta group x warp of the row sweep) that hold a block with C[b] >= L and C[b] > thrAbs
// (csm_sweep_tiles_kernel).  Matches whose projection may break the bound (csm_project_kernel's noBound flag)
// get every tile, and csm_select_kernel treats them as it treats the exhaustive tables.
//
// Why C[b] >= F[b] holds for every block of an unflagged match: C[b] and each fine score of block b are sums
// over the same beams in the same order, of coarse[p + o_b] and of fine[p + o_b + f] (0 <= f.x, f.y < L).
// IEEE addition is monotone, so termwise coarse >= fine gives C >= F bit for bit.  coarse is the win-max of
// fine over [c, c + L) on each axis (lgs_precompute), with the window moved to [n - L, n) at the upper map
// edge, which still covers every in-map cell of [c, c + L); cells past the map read the zero apron on both
// maps.  The one failure is a coarse index c in (-L, 0) on either axis: it reads 0 while fine cells
// c + f >= 0 are in the map (SURVEY.md H12).  The projection flags every kept beam whose clamped cell plus a
// block origin falls there (clamping keeps out-of-window points at c <= -L, so they never reach the band).
// Near-edge points, which results() may re-derive one cell away on the host, are tested at cell +- 1.
constexpr int kSeedBlocks = 4;       // coarse blocks whose fine blocks give the bound L
constexpr int kPruneThreads = 128;   // csm_prune_kernel block
constexpr int kTilesWarps = 4;       // csm_sweep_tiles_kernel warps per block

// One warp per (theta group, match): grid = (theta groups, matches).
template <int UNROLL, int TG>
__global__ void __launch_bounds__(32)
csm_coarse_kernel(const CsmDesc* __restrict__ descs, const double* __restrict__ coarseGrid, int pitch, CsmWindow w,
                  const int* __restrict__ offs, double* __restrict__ coarseTab) {
    extern __shared__ int sOff[];   // [beam][TG]
    const CsmDesc d = descs[blockIdx.y];
    const int t0 = blockIdx.x * TG;
    if (t0 >= d.nT) return;
    const int nTg = min(TG, d.nT - t0);
    stage_theta_group<TG>(d, offs, t0, nTg, sOff, threadIdx.x, 32);
    __syncwarp();
    for (int h = threadIdx.x; h < w.nbx * w.nby; h += 32)
        coarse_theta_group<UNROLL, TG>(d, w, sOff, coarseGrid, pitch, h, t0, nTg, coarseTab);
}

// (c, v) beats (bc, bv) in the order (score desc, visit asc)
__device__ __forceinline__ bool csm_before(double c, int v, double bc, int bv) {
    return c > bc || (c == bc && v < bv);
}

// Block-wide (score desc, visit asc) minimum of every thread's (c, v); every thread gets it.
__device__ void csm_block_best(double& c, int& v, double* sC, int* sV) {
    __syncthreads();
    sC[threadIdx.x] = c; sV[threadIdx.x] = v;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s && csm_before(sC[threadIdx.x + s], sV[threadIdx.x + s], sC[threadIdx.x], sV[threadIdx.x])) {
            sC[threadIdx.x] = sC[threadIdx.x + s];
            sV[threadIdx.x] = sV[threadIdx.x + s];
        }
        __syncthreads();
    }
    c = sC[0]; v = sV[0];
}

__device__ __forceinline__ bool csm_keep(double c, double bound, double thrAbs) { return c >= bound && c > thrAbs; }

// One block per match.  Seed: the kSeedBlocks best coarse blocks in (C desc, visit asc) order; their fine
// 5x5 (lowRes x lowRes) blocks are summed in beam order like the sweep, so L = their maximum is a fine score
// of the window and L <= F*.  Keep: C[b] >= L (a tie with F* at an earlier visit must be scored) and
// C[b] > thrAbs (no block at or below the threshold can make the match found).  Every warp tile of the row
// sweep that holds a kept block of one of its slices goes to the work list; a flagged match lists them all.
__global__ void __launch_bounds__(kPruneThreads)
csm_prune_kernel(const CsmDesc* __restrict__ descs, const double* __restrict__ fineGrid, int pitch, CsmWindow w,
                 const int* __restrict__ offs, const double* __restrict__ coarseTab,
                 const int* __restrict__ noBound, double* __restrict__ bound, int tileG, int2* __restrict__ tiles,
                 int* __restrict__ tileCount) {
    __shared__ double sC[kPruneThreads];
    __shared__ int sV[kPruneThreads];
    const int m = blockIdx.x;
    const CsmDesc d = descs[m];
    const int nbxy = w.nbx * w.nby, nB = d.nT * nbxy;
    const double* C = coarseTab + d.coarseBegin;
    const bool full = noBound[m] != 0;
    double L = -INFINITY;
    if (!full) {
        int seed[kSeedBlocks];
        double pc = INFINITY;
        int pv = -1;
#pragma unroll
        for (int k = 0; k < kSeedBlocks; ++k) {   // k-th best: the best of those after the (k-1)-th
            double bc = -INFINITY;
            int bv = 0x7fffffff;
            for (int v = threadIdx.x; v < nB; v += blockDim.x) {
                const double c = C[v];
                if (csm_before(pc, pv, c, v) && csm_before(c, v, bc, bv)) { bc = c; bv = v; }
            }
            csm_block_best(bc, bv, sC, sV);
            seed[k] = bv < nB ? bv : -1;
            pc = bc; pv = bv;
        }
        const int cells = w.lowRes * w.lowRes;
        double best = -INFINITY;
        for (int p = threadIdx.x; p < kSeedBlocks * cells; p += blockDim.x) {
            int v = -1;
#pragma unroll
            for (int k = 0; k < kSeedBlocks; ++k) if (p / cells == k) v = seed[k];
            if (v < 0) continue;
            const int t = v / nbxy, bx = (v / w.nby) % w.nbx, by = v % w.nby;
            const int f = p % cells;
            const double* __restrict__ gp = fineGrid + (-w.winY + by * w.lowRes + f % w.lowRes) * pitch +
                                            (-w.winX + bx * w.lowRes + f / w.lowRes);
            const int* __restrict__ o = offs + d.offBegin + (long long)t * d.nKeptPad;
            double acc = 0.0;
#pragma unroll 4
            for (int i = 0; i < d.nKeptPad; ++i) acc = __dadd_rn(acc, __ldg(gp + __ldg(o + i)));   // beam order
            best = fmax(best, acc);
        }
        int dummy = 0;
        csm_block_best(best, dummy, sC, sV);
        L = best;
    }
    if (threadIdx.x == 0) bound[m] = L;
    const int wpt = w.xChunks * w.rowGroups;        // warps per slice group
    const int nG = (d.nT + tileG - 1) / tileG;
    for (int p = threadIdx.x; p < nG * wpt; p += blockDim.x) {
        const int g = p / wpt, wg = p - g * wpt;
        bool need = full;
        if (!need) {
            const int xc = wg % w.xChunks, rg = wg / w.xChunks;
            const int x0 = xc * 32, x1 = min(x0 + 32, w.nxw) - 1;
            const int y0 = rg * w.rows, y1 = min(y0 + w.rows, w.nyw) - 1;
            for (int t = g * tileG; t < min(d.nT, (g + 1) * tileG) && !need; ++t)
                for (int bx = x0 / w.lowRes; bx <= x1 / w.lowRes && !need; ++bx)
                    for (int by = y0 / w.lowRes; by <= y1 / w.lowRes && !need; ++by)
                        need = csm_keep(C[(t * w.nbx + bx) * w.nby + by], L, d.thrAbs);
        }
        if (need) tiles[atomicAdd(tileCount, 1)] = make_int2(m, p);
    }
}

// Grid-stride over the work list, one tile per warp; each warp stages its own group's offsets.
template <int UNROLL, int ROWS, int TG>
__global__ void __launch_bounds__(kTilesWarps * 32)
csm_sweep_tiles_kernel(const CsmDesc* __restrict__ descs, const double* __restrict__ fineGrid, int pitch,
                       CsmWindow w, const int* __restrict__ offs, const int2* __restrict__ tiles,
                       const int* __restrict__ tileCount, int warpSmem, double* __restrict__ fineTab) {
    extern __shared__ int sAll[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    int* sOff = sAll + warp * warpSmem;
    const int n = *tileCount;
    const int wpt = w.xChunks * w.rowGroups;
    for (int k = blockIdx.x * wpb + warp; k < n; k += gridDim.x * wpb) {
        const int2 tile = tiles[k];
        const CsmDesc d = descs[tile.x];
        const int g = tile.y / wpt, wg = tile.y - g * wpt;
        const int t0 = g * TG, nTg = min(TG, d.nT - t0);
        __syncwarp();   // the previous tile's reads of sOff are done
        stage_theta_group<TG>(d, offs, t0, nTg, sOff, lane, 32);
        __syncwarp();
        fine_theta_group<UNROLL, ROWS, TG>(d, w, sOff, fineGrid, pitch, wg, lane, t0, nTg, fineTab);
    }
}

// ---- K3: block maxima + CPU-order selection -----------------------------------------------------
// One thread block per match.  After the pruned sweep (noBound != nullptr) an unflagged match considers only
// the kept blocks: the others were not scored, and every one of them is below F* or at most the threshold.
// Should a kept block still show C < F there (a coarse map that is not lgs_precompute's win-max of the grid),
// the match is flagged and marked needFull, and results() scores it again with every tile.
__global__ void __launch_bounds__(256)
csm_select_kernel(const CsmDesc* __restrict__ descs, CsmWindow w,
                  const double* __restrict__ fineTab, const double* __restrict__ coarseTab,
                  double* __restrict__ blockMax, int* __restrict__ blockArg,
                  int* __restrict__ noBound, const double* __restrict__ bound,
                  DevResult* __restrict__ results) {
    const CsmDesc d = descs[blockIdx.x];
    const int nB = d.nT * w.nbx * w.nby;
    double* F = blockMax + d.coarseBegin;
    int* A = blockArg + d.coarseBegin;
    const double* C = coarseTab + d.coarseBegin;
    const double* fine = fineTab + d.fineBegin;
    const bool pruned = noBound && !noBound[blockIdx.x];
    const double L = pruned ? bound[blockIdx.x] : 0.0;
    __shared__ int sInvalid;
    __shared__ double sBest[256];
    __shared__ int sIdx[256];
    if (threadIdx.x == 0) sInvalid = 0;
    __syncthreads();

    // Phase 1: F[v] = max of the lowRes x lowRes fine scores of block v, first visit wins
    // (x outer, y inner; strict '<' update: scan_matcher_real_time_correlative.cpp:239-251).
    double myBest = -1.0;
    int myIdx = 0x7fffffff;
    bool invalid = false;
    for (int v = threadIdx.x; v < nB; v += blockDim.x) {
        if (pruned && !csm_keep(C[v], L, d.thrAbs)) continue;
        const int by = v % w.nby;
        const int bx = (v / w.nby) % w.nbx;
        const int t = v / (w.nby * w.nbx);
        const double* ft = fine + (long long)t * w.nyw * w.nxw;
        double m = -1.0;
        int arg = 0;
        for (int fx = 0; fx < w.lowRes; ++fx)
            for (int fy = 0; fy < w.lowRes; ++fy) {
                const double s = ft[(by * w.lowRes + fy) * w.nxw + bx * w.lowRes + fx];
                if (m < s) { m = s; arg = fx * w.lowRes + fy; }
            }
        F[v] = m;
        A[v] = arg;
        if (C[v] < m) invalid = true;   // the coarse value is not an upper bound (H12)
        if (m > myBest) { myBest = m; myIdx = v; }   // v ascending per thread: first visit kept
    }
    if (invalid) atomicOr(&sInvalid, 1);
    sBest[threadIdx.x] = myBest;
    sIdx[threadIdx.x] = myIdx;
    __syncthreads();

    DevResult r;
    r.needFull = 0;
    if (sInvalid && pruned) {
        if (threadIdx.x != 0) return;
        noBound[blockIdx.x] = 1;
        r.needFull = 1; r.exactReplay = 0;
        r.found = 0; r.score = d.thrAbs;
        r.ix = -w.winX; r.iy = -w.winY; r.it = -d.winT;
        results[blockIdx.x] = r;
        return;
    }
    if (!sInvalid) {
        // Every C[v] >= F[v]: the pruned CPU loop returns the first visit of the global maximum.
        for (int s = blockDim.x / 2; s > 0; s >>= 1) {
            if (threadIdx.x < s) {
                const double ob = sBest[threadIdx.x + s];
                const int oi = sIdx[threadIdx.x + s];
                if (ob > sBest[threadIdx.x] || (ob == sBest[threadIdx.x] && oi < sIdx[threadIdx.x])) {
                    sBest[threadIdx.x] = ob;
                    sIdx[threadIdx.x] = oi;
                }
            }
            __syncthreads();
        }
        if (threadIdx.x != 0) return;
        r.exactReplay = 0;
        if (nB > 0 && sBest[0] > d.thrAbs) {
            const int v = sIdx[0];
            const int by = v % w.nby, bx = (v / w.nby) % w.nbx, t = v / (w.nby * w.nbx);
            r.found = 1; r.score = sBest[0];
            r.ix = -w.winX + bx * w.lowRes + A[v] / w.lowRes;
            r.iy = -w.winY + by * w.lowRes + A[v] % w.lowRes;
            r.it = t - d.winT;
        } else {
            r.found = 0; r.score = d.thrAbs;
            r.ix = -w.winX; r.iy = -w.winY; r.it = -d.winT;
        }
        results[blockIdx.x] = r;
        return;
    }
    // Sequential replay of the CPU's visit sequence (:88-114).
    if (threadIdx.x != 0) return;
    double best = d.thrAbs;
    int bv = -1;
    for (int v = 0; v < nB; ++v) {
        if (C[v] <= best) continue;
        if (best < F[v]) { best = F[v]; bv = v; }
    }
    r.exactReplay = 1;
    if (bv >= 0) {
        const int by = bv % w.nby, bx = (bv / w.nby) % w.nbx, t = bv / (w.nby * w.nbx);
        r.found = 1; r.score = best;
        r.ix = -w.winX + bx * w.lowRes + A[bv] / w.lowRes;
        r.iy = -w.winY + by * w.lowRes + A[bv] % w.lowRes;
        r.it = t - d.winT;
    } else {
        r.found = 0; r.score = d.thrAbs;
        r.ix = -w.winX; r.iy = -w.winY; r.it = -d.winT;
    }
    results[blockIdx.x] = r;
}

__global__ void csm_patch_kernel(const int* __restrict__ where, const int* __restrict__ offVal,
                                 const int2* __restrict__ cellVal, const long long* cellWhere,
                                 int n, int* offs, int2* cells) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    (void)where;
    offs[cellWhere[2 * k]] = offVal[k];
    cells[cellWhere[2 * k + 1]] = cellVal[k];
}

int pick_block(int nHyp) {
    // Threads per block: the multiple of 32 in [64, 256] wasting the fewest lanes, larger wins ties.
    int best = 128;
    long long bestWaste = 1LL << 60;
    for (int b = 256; b >= 64; b -= 32) {
        const long long tiles = (nHyp + b - 1) / b;
        const long long waste = tiles * b - nHyp;
        if (waste < bestWaste) { bestWaste = waste; best = b; }
    }
    return best;
}

}  // namespace

struct lgs_rtcsm_batch {
    lgs_ctx* ctx = nullptr;
    lgs_rtcsm_params params{};
    int nMatch = 0;
    int maxNT = 0, maxKeptPad = 0;
    size_t sweepSmem = 0;                        // dynamic shared memory of the sweep launch
    CsmWindow win{};
    GridGeom geom{};
    std::vector<CsmDesc> descs;
    std::vector<double> hAngles, hRanges;        // kept beams, host copy (for fix-ups)
    std::vector<double> stepT;
    std::vector<int> fixups;
    long long nOff = 0, nCell = 0, nFine = 0, nCoarse = 0;
    long long workHyp = 0, workGather = 0;
    DevBuf<CsmDesc> dDescs;
    DevBuf<double> dAngles, dRanges, dFine, dCoarse, dBlockMax;
    DevBuf<int> dOffs, dBlockArg, dFlagCount;
    DevBuf<int2> dCells;
    DevBuf<FlagEntry> dFlags;
    int flagCap = kFlagCap;
    // near-edge fix-up values (results()): kept with the batch, no per-call cudaMalloc
    DevBuf<int> dFixOff;
    DevBuf<int2> dFixCell;
    DevBuf<long long> dFixWhere;
    DevBuf<DevResult> dResults;
    PinBuf<DevResult> hResults;
    PinBuf<int> hFlagCount;
    PinBuf<CsmDesc> hDescs;
    PinBuf<double> hStage;
    // pruned sweep of row-mapped windows (K2c)
    long long nTilesAll = 0;                     // warp tiles of the exhaustive fine sweep
    int tilesGrid = 0;                           // csm_sweep_tiles_kernel blocks (all resident)
    size_t tilesSmem = 0;
    bool tablesFull = false;                     // dFine / dCoarse hold every hypothesis of every match
    const lgs_grid* lastGrid = nullptr;          // maps of the last run (debug() re-scores against them)
    const lgs_grid* lastCoarse = nullptr;
    DevBuf<int> dNoBound, dTileCount;
    DevBuf<double> dBound;
    DevBuf<int2> dTiles;
    bool uploaded = false, ran = false;
};

static int csm_launch_sweep(lgs_rtcsm_batch* b, const lgs_grid* grid, const lgs_grid* coarse) {
    lgs_ctx* c = b->ctx;
    const CsmWindow& w = b->win;
    for (int m0 = 0; m0 < b->nMatch; m0 += 65535) {
        const int nm = std::min(65535, b->nMatch - m0);
        // the row-mapped sweep takes kThetaGroup slices per block row
        const int tiles = w.rows ? (b->maxNT + kThetaGroup - 1) / kThetaGroup : b->maxNT;
        dim3 gridDim(w.tilesFine + w.tilesCoarse, tiles, nm);
        const size_t smem = b->sweepSmem;
        if (w.rows == 5)
            csm_sweep_rows_kernel<kRowsUnroll, 5, kThetaGroup><<<gridDim, w.block, smem, c->stream>>>(
                b->dDescs.p + m0, grid->origin(), coarse->origin(), grid->pitch, w, b->dOffs.p,
                b->dFine.p, b->dCoarse.p);
        else if (w.rows == 4)
            csm_sweep_rows_kernel<kRowsUnroll, 4, kThetaGroup><<<gridDim, w.block, smem, c->stream>>>(
                b->dDescs.p + m0, grid->origin(), coarse->origin(), grid->pitch, w, b->dOffs.p,
                b->dFine.p, b->dCoarse.p);
        else if (w.hpt == 4)
            csm_sweep_kernel<4, 4><<<gridDim, w.block, smem, c->stream>>>(
                b->dDescs.p + m0, grid->origin(), coarse->origin(), grid->pitch, w, b->dOffs.p,
                b->dFine.p, b->dCoarse.p);
        else
            csm_sweep_kernel<kBeamPad, 1><<<gridDim, w.block, smem, c->stream>>>(
                b->dDescs.p + m0, grid->origin(), coarse->origin(), grid->pitch, w, b->dOffs.p,
                b->dFine.p, b->dCoarse.p);
        LGS_LAUNCH_CHECK(c);
    }
    b->tablesFull = true;
    return LGS_OK;
}

// Steps 2-5 of a run (coarse scores, bound, work list, fine scores): the exhaustive sweep for windows of the
// flattened sweep, the pruned chain (K2c) for row-mapped ones.  Stream ordered, no host synchronisation.
static int csm_launch_score(lgs_rtcsm_batch* b, const lgs_grid* grid, const lgs_grid* coarse) {
    const CsmWindow& w = b->win;
    if (!w.rows) return csm_launch_sweep(b, grid, coarse);
    lgs_ctx* c = b->ctx;
    LGS_CUDA(c, cudaMemsetAsync(b->dTileCount.p, 0, sizeof(int), c->stream));
    const int nG = (b->maxNT + kThetaGroup - 1) / kThetaGroup;
    for (int m0 = 0; m0 < b->nMatch; m0 += 65535) {
        const int nm = std::min(65535, b->nMatch - m0);
        csm_coarse_kernel<kRowsUnroll, kThetaGroup><<<dim3(nG, nm), 32, b->sweepSmem, c->stream>>>(
            b->dDescs.p + m0, coarse->origin(), grid->pitch, w, b->dOffs.p, b->dCoarse.p);
        LGS_LAUNCH_CHECK(c);
    }
    csm_prune_kernel<<<b->nMatch, kPruneThreads, 0, c->stream>>>(
        b->dDescs.p, grid->origin(), grid->pitch, w, b->dOffs.p, b->dCoarse.p, b->dNoBound.p, b->dBound.p,
        kThetaGroup, b->dTiles.p, b->dTileCount.p);
    LGS_LAUNCH_CHECK(c);
    const int warpSmem = kThetaGroup * b->maxKeptPad;
    if (w.rows == 5)
        csm_sweep_tiles_kernel<kRowsUnroll, 5, kThetaGroup><<<b->tilesGrid, kTilesWarps * 32, b->tilesSmem, c->stream>>>(
            b->dDescs.p, grid->origin(), grid->pitch, w, b->dOffs.p, b->dTiles.p, b->dTileCount.p, warpSmem,
            b->dFine.p);
    else
        csm_sweep_tiles_kernel<kRowsUnroll, 4, kThetaGroup><<<b->tilesGrid, kTilesWarps * 32, b->tilesSmem, c->stream>>>(
            b->dDescs.p, grid->origin(), grid->pitch, w, b->dOffs.p, b->dTiles.p, b->dTileCount.p, warpSmem,
            b->dFine.p);
    LGS_LAUNCH_CHECK(c);
    b->tablesFull = false;
    return LGS_OK;
}

static int csm_launch_select(lgs_rtcsm_batch* b) {
    lgs_ctx* c = b->ctx;
    const bool pruned = b->win.rows != 0;
    csm_select_kernel<<<b->nMatch, 256, 0, c->stream>>>(b->dDescs.p, b->win, b->dFine.p,
                                                        b->dCoarse.p, b->dBlockMax.p,
                                                        b->dBlockArg.p, pruned ? b->dNoBound.p : nullptr,
                                                        b->dBound.p, b->dResults.p);
    LGS_LAUNCH_CHECK(c);
    return LGS_OK;
}

// Scores and selects again (after near-edge fix-ups, or for matches the select marked needFull) and waits for
// the result records.
static int csm_rescore_results(lgs_rtcsm_batch* b, const lgs_grid* grid, const lgs_grid* coarse) {
    lgs_ctx* c = b->ctx;
    int rc = csm_launch_score(b, grid, coarse);
    if (rc == LGS_OK) rc = csm_launch_select(b);
    if (rc != LGS_OK) return rc;
    LGS_CUDA(c, cudaMemcpyAsync(b->hResults.p, b->dResults.p, b->nMatch * sizeof(DevResult),
                                cudaMemcpyDeviceToHost, c->stream));
    LGS_CUDA(c, cudaStreamSynchronize(c->stream));
    return LGS_OK;
}

extern "C" {

int lgs_rtcsm_batch_create(lgs_ctx* ctx, const lgs_rtcsm_params* p, lgs_rtcsm_batch** out) {
    if (!ctx || !p || !out) return LGS_ERR_INVALID;
    *out = nullptr;
    if (p->low_res < 1 || !(p->range_x >= 0) || !(p->range_y >= 0) || !(p->range_theta >= 0))
        return lgs_fail(ctx, LGS_ERR_INVALID, "rtcsm_batch_create: bad parameters");
    lgs_rtcsm_batch* b = new lgs_rtcsm_batch();
    b->ctx = ctx;
    b->params = *p;
    *out = b;
    return LGS_OK;
}

int lgs_rtcsm_batch_destroy(lgs_rtcsm_batch* b) {
    if (!b) return LGS_OK;
    cudaSetDevice(b->ctx->device);
    cudaStreamSynchronize(b->ctx->stream);
    b->dDescs.release(); b->dAngles.release(); b->dRanges.release(); b->dFine.release();
    b->dCoarse.release(); b->dBlockMax.release(); b->dOffs.release(); b->dBlockArg.release();
    b->dFlagCount.release(); b->dCells.release(); b->dFlags.release(); b->dResults.release();
    b->dFixOff.release(); b->dFixCell.release(); b->dFixWhere.release();
    b->dNoBound.release(); b->dTileCount.release(); b->dBound.release(); b->dTiles.release();
    b->hResults.release(); b->hFlagCount.release(); b->hDescs.release(); b->hStage.release();
    delete b;
    return LGS_OK;
}

int lgs_rtcsm_batch_upload(lgs_rtcsm_batch* b, const lgs_grid* grid, const lgs_scan_batch* scans,
                           const double* normThr) {
    if (!b || !grid || !scans) return LGS_ERR_INVALID;
    lgs_ctx* c = b->ctx;
    const int n = scans->n_scans;
    if (n < 0 || (n > 0 && (!scans->beam_begin || !scans->sensor_pose)))
        return lgs_fail(c, LGS_ERR_INVALID, "rtcsm_batch_upload: bad scan batch");
    if (grid->off_x || grid->off_y)
        return lgs_fail(c, LGS_ERR_INVALID, "rtcsm_batch_upload: windowed grids (lgs_grid_set_window) are not supported");
    LGS_CUDA(c, cudaSetDevice(c->device));
    const lgs_rtcsm_params& p = b->params;
    b->uploaded = false; b->ran = false;
    b->nMatch = n;

    // Search step and window: scan_matcher_real_time_correlative.cpp:61-73, :156-175.
    const double stepX = grid->res, stepY = grid->res;
    CsmWindow& w = b->win;
    w.lowRes = p.low_res;
    w.winX = static_cast<int>(std::ceil(0.5 * p.range_x / stepX));
    w.winY = static_cast<int>(std::ceil(0.5 * p.range_y / stepY));
    // for (x = -winX; x <= winX; x += lowRes): SURVEY.md H2 (asymmetric window).
    w.nbx = (2 * w.winX) / w.lowRes + 1;
    w.nby = (2 * w.winY) / w.lowRes + 1;
    w.nxw = w.nbx * w.lowRes;
    w.nyw = w.nby * w.lowRes;
    if (std::max(w.nxw, w.nyw) > grid->apron)
        return lgs_fail(c, LGS_ERR_APRON, "rtcsm: window %dx%d cells needs apron >= %d, grid has %d",
                        w.nxw, w.nyw, std::max(w.nxw, w.nyw), grid->apron);
    w.hpt = (w.nxw * w.nyw >= 512) ? 4 : 1;
    w.slots = (((w.nxw * w.nyw + w.hpt - 1) / w.hpt) + 31) / 32 * 32;
    w.block = pick_block(w.slots);
    w.tilesFine = (w.slots + w.block - 1) / w.block;
    w.rows = 0; w.xChunks = 1; w.rowGroups = 0;
    if (w.hpt == 4 && !c->opt.csmFlat) {
        // row-mapped sweep: lanes = x offsets of one window row, ROWS rows per thread
        w.rows = (w.nyw % 5 == 0) ? 5 : 4;
        w.xChunks = (w.nxw + 31) / 32;
        w.rowGroups = (w.nyw + w.rows - 1) / w.rows;
        const int warps = w.xChunks * w.rowGroups;
        int wpb = std::min(8, warps);                        // warps per block: fewest idle warps, larger wins
        long long bestWaste = 1LL << 60;
        for (int cand = std::min(8, warps); cand >= 2; --cand) {
            const long long waste = (long long)((warps + cand - 1) / cand) * cand - warps;
            if (waste < bestWaste) { bestWaste = waste; wpb = cand; }
        }
        w.block = wpb * 32;
        w.tilesFine = (warps + wpb - 1) / wpb;
    }
    w.tilesCoarse = (w.nbx * w.nby + w.block - 1) / w.block;
    b->geom = GridGeom{grid->min_x, grid->min_y, grid->res, grid->nx, grid->ny, grid->pitch};

    b->descs.assign(n, CsmDesc{});
    b->stepT.assign(n, 0.0);
    b->fixups.assign(n, 0);
    b->hAngles.clear(); b->hRanges.clear();
    b->maxNT = 0; b->maxKeptPad = kBeamPad;
    long long nOff = 0, nCell = 0, nFine = 0, nCoarse = 0;
    b->workHyp = 0; b->workGather = 0; b->nTilesAll = 0;
    for (int m = 0; m < n; ++m) {
        const int b0 = scans->beam_begin[m], b1 = scans->beam_begin[m + 1];
        const int nb = b1 - b0;
        if (nb <= 0) return lgs_fail(c, LGS_ERR_INVALID, "rtcsm: scan %d has no beams", m);
        CsmDesc& d = b->descs[m];
        d.sx = scans->sensor_pose[3 * m]; d.sy = scans->sensor_pose[3 * m + 1];
        d.st = scans->sensor_pose[3 * m + 2];
        double maxR = scans->ranges[b0];
        for (int i = b0 + 1; i < b1; ++i) maxR = std::max(maxR, scans->ranges[i]);   // :163-164
        const double maxRange = std::min(maxR, p.scan_range_max);                        // :165
        const double th = grid->res / maxRange;                                          // :166
        d.stepT = std::acos(1.0 - 0.5 * th * th);                                       // :170
        b->stepT[m] = d.stepT;
        d.winT = static_cast<int>(std::ceil(0.5 * p.range_theta / d.stepT));             // :72-73
        if (!(d.stepT > 0.0) || d.winT < 0 || d.winT > (1 << 20))
            return lgs_fail(c, LGS_ERR_INVALID, "rtcsm: scan %d gives stepTheta=%g winTheta=%d", m,
                            d.stepT, d.winT);
        d.nT = 2 * d.winT + 1;
        const double thr = normThr ? normThr[m] : DBL_MIN;                               // :46-47
        d.thrAbs = thr * static_cast<double>(static_cast<size_t>(nb));                   // :77-78
        d.beamBegin = (int)b->hAngles.size();
        for (int i = b0; i < b1; ++i) {
            if (scans->ranges[i] >= p.scan_range_max) continue;                          // :192-193
            b->hAngles.push_back(scans->angles[i]);
            b->hRanges.push_back(scans->ranges[i]);
        }
        d.nKept = (int)b->hAngles.size() - d.beamBegin;
        d.nKeptPad = std::max(kBeamPad, (d.nKept + kBeamPad - 1) / kBeamPad * kBeamPad);
        d.offBegin = nOff; d.cellBegin = nCell; d.fineBegin = nFine; d.coarseBegin = nCoarse;
        nOff += (long long)d.nT * d.nKeptPad;
        nCell += (long long)d.nT * d.nKept;
        nFine += (long long)d.nT * w.nxw * w.nyw;
        nCoarse += (long long)d.nT * w.nbx * w.nby;
        b->maxNT = std::max(b->maxNT, d.nT);
        b->maxKeptPad = std::max(b->maxKeptPad, d.nKeptPad);
        const long long hyp = (long long)d.nT * ((long long)w.nxw * w.nyw + (long long)w.nbx * w.nby);
        b->workHyp += hyp;
        b->workGather += hyp * d.nKept;
        b->nTilesAll += w.rows ? (long long)((d.nT + kThetaGroup - 1) / kThetaGroup) * w.xChunks * w.rowGroups
                               : (long long)d.nT * (w.slots / 32);
    }
    if (b->maxNT > 65535)
        return lgs_fail(c, LGS_ERR_INVALID, "rtcsm: %d theta slices exceed the launch grid", b->maxNT);
    // the row-mapped sweep stages the offsets of kThetaGroup slices, the flattened one of one slice
    b->sweepSmem = (size_t)(w.rows ? kThetaGroup : 1) * b->maxKeptPad * sizeof(int);
    if (b->sweepSmem > 200 * 1024)
        return lgs_fail(c, LGS_ERR_INVALID, "rtcsm: %d beams exceed shared memory", b->maxKeptPad);
    b->nOff = nOff; b->nCell = nCell; b->nFine = nFine; b->nCoarse = nCoarse;
    if (n == 0) { b->uploaded = true; return LGS_OK; }

    const size_t nk = b->hAngles.size();
    LGS_CUDA(c, b->dDescs.reserve(n));
    LGS_CUDA(c, b->dAngles.reserve(std::max<size_t>(nk, 1)));
    LGS_CUDA(c, b->dRanges.reserve(std::max<size_t>(nk, 1)));
    LGS_CUDA(c, b->dOffs.reserve(nOff));
    LGS_CUDA(c, b->dCells.reserve(std::max<long long>(nCell, 1)));
    LGS_CUDA(c, b->dFine.reserve(nFine));
    LGS_CUDA(c, b->dCoarse.reserve(nCoarse));
    LGS_CUDA(c, b->dBlockMax.reserve(nCoarse));
    LGS_CUDA(c, b->dBlockArg.reserve(nCoarse));
    LGS_CUDA(c, b->dFlagCount.reserve(1));
    LGS_CUDA(c, b->dFlags.reserve(b->flagCap));
    LGS_CUDA(c, b->dResults.reserve(n));
    LGS_CUDA(c, b->dNoBound.reserve(n));
    LGS_CUDA(c, b->dBound.reserve(n));
    LGS_CUDA(c, b->dTileCount.reserve(1));
    if (w.rows) LGS_CUDA(c, b->dTiles.reserve(b->nTilesAll));
    LGS_CUDA(c, b->hResults.reserve(n));
    LGS_CUDA(c, b->hFlagCount.reserve(1));
    LGS_CUDA(c, b->hDescs.reserve(n));
    LGS_CUDA(c, b->hStage.reserve(2 * std::max<size_t>(nk, 1)));
    // Stage through pinned memory so the copies are truly asynchronous.
    memcpy(b->hDescs.p, b->descs.data(), n * sizeof(CsmDesc));
    memcpy(b->hStage.p, b->hAngles.data(), nk * sizeof(double));
    memcpy(b->hStage.p + nk, b->hRanges.data(), nk * sizeof(double));
    LGS_CUDA(c, cudaMemcpyAsync(b->dDescs.p, b->hDescs.p, n * sizeof(CsmDesc),
                                cudaMemcpyHostToDevice, c->stream));
    if (nk) {
        LGS_CUDA(c, cudaMemcpyAsync(b->dAngles.p, b->hStage.p, nk * sizeof(double),
                                    cudaMemcpyHostToDevice, c->stream));
        LGS_CUDA(c, cudaMemcpyAsync(b->dRanges.p, b->hStage.p + nk, nk * sizeof(double),
                                    cudaMemcpyHostToDevice, c->stream));
    }
    if (b->sweepSmem > 48 * 1024)
    {
        const int smem = (int)b->sweepSmem;
        if (w.rows) {
            LGS_CUDA(c, cudaFuncSetAttribute(csm_sweep_rows_kernel<kRowsUnroll, 5, kThetaGroup>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            LGS_CUDA(c, cudaFuncSetAttribute(csm_sweep_rows_kernel<kRowsUnroll, 4, kThetaGroup>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        } else {
            LGS_CUDA(c, cudaFuncSetAttribute(csm_sweep_kernel<kBeamPad, 1>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            LGS_CUDA(c, cudaFuncSetAttribute(csm_sweep_kernel<4, 4>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        }
    }
    if (w.rows) {
        // coarse kernel: one group's offsets per block, like the exhaustive sweep; tiles kernel: one per warp
        b->tilesSmem = (size_t)kTilesWarps * b->sweepSmem;
        if (b->sweepSmem > 48 * 1024)
            LGS_CUDA(c, cudaFuncSetAttribute(csm_coarse_kernel<kRowsUnroll, kThetaGroup>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->sweepSmem));
        const auto tilesKernel = w.rows == 5 ? csm_sweep_tiles_kernel<kRowsUnroll, 5, kThetaGroup>
                                             : csm_sweep_tiles_kernel<kRowsUnroll, 4, kThetaGroup>;
        if (b->tilesSmem > 48 * 1024)
            LGS_CUDA(c, cudaFuncSetAttribute(tilesKernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)b->tilesSmem));
        int perSm = 0;
        LGS_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, tilesKernel, kTilesWarps * 32,
                                                                  b->tilesSmem));
        if (perSm < 1)
            return lgs_fail(c, LGS_ERR_INVALID, "rtcsm: %d beams leave no room for the pruned sweep", b->maxKeptPad);
        b->tilesGrid = (int)std::min<long long>((long long)perSm * c->sm_count,
                                                (b->nTilesAll + kTilesWarps - 1) / kTilesWarps);
    }
    b->uploaded = true;
    return LGS_OK;
}

static int csm_launch_project(lgs_rtcsm_batch* b) {
    lgs_ctx* c = b->ctx;
    LGS_CUDA(c, cudaMemsetAsync(b->dNoBound.p, 0, b->nMatch * sizeof(int), c->stream));
    for (int m0 = 0; m0 < b->nMatch; m0 += 65535) {
        const int nm = std::min(65535, b->nMatch - m0);
        const long long per = (long long)b->maxNT * b->maxKeptPad;
        dim3 gridDim((unsigned)((per + 255) / 256), nm);
        csm_project_kernel<<<gridDim, 256, 0, c->stream>>>(b->dDescs.p + m0, b->dAngles.p,
                                                           b->dRanges.p, b->geom, b->win,
                                                           c->opt.edgeEps, b->dOffs.p, b->dCells.p, b->dFlags.p,
                                                           b->flagCap, b->dFlagCount.p, b->dNoBound.p + m0);
        LGS_LAUNCH_CHECK(c);
    }
    return LGS_OK;
}

static int csm_run_impl(lgs_rtcsm_batch* b, const lgs_grid* grid, const lgs_grid* coarse, float* ms) {
    if (!b || !grid || !coarse) return LGS_ERR_INVALID;
    lgs_ctx* c = b->ctx;
    if (!b->uploaded) return lgs_fail(c, LGS_ERR_INVALID, "rtcsm_batch_run before upload");
    if (coarse->nx != grid->nx || coarse->ny != grid->ny || coarse->pitch != grid->pitch ||
        grid->pitch != b->geom.pitch || grid->nx != b->geom.nx || grid->ny != b->geom.ny)
        return lgs_fail(c, LGS_ERR_INVALID, "rtcsm_batch_run: grid geometry mismatch");
    if (ms) ms[0] = ms[1] = ms[2] = 0.f;
    if (b->nMatch == 0) { b->ran = true; return LGS_OK; }
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, lgs_grid_acquire(c, grid));     // maps owned by another context (the builder's latest map)
    LGS_CUDA(c, lgs_grid_acquire(c, coarse));
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    if (ms) for (auto& e : ev) LGS_CUDA(c, cudaEventCreate(&e));
    LGS_CUDA(c, cudaMemsetAsync(b->dFlagCount.p, 0, sizeof(int), c->stream));
    if (ms) LGS_CUDA(c, cudaEventRecord(ev[0], c->stream));
    int rc = csm_launch_project(b);
    if (rc != LGS_OK) return rc;
    if (ms) LGS_CUDA(c, cudaEventRecord(ev[1], c->stream));
    b->lastGrid = grid; b->lastCoarse = coarse;
    rc = csm_launch_score(b, grid, coarse);
    if (rc != LGS_OK) return rc;
    if (ms) LGS_CUDA(c, cudaEventRecord(ev[2], c->stream));
    rc = csm_launch_select(b);
    if (rc != LGS_OK) return rc;
    if (ms) {
        LGS_CUDA(c, cudaEventRecord(ev[3], c->stream));
        LGS_CUDA(c, cudaEventSynchronize(ev[3]));
        for (int k = 0; k < 3; ++k) LGS_CUDA(c, cudaEventElapsedTime(&ms[k], ev[k], ev[k + 1]));
        for (auto& e : ev) cudaEventDestroy(e);
    }
    b->ran = true;
    return LGS_OK;
}

int lgs_rtcsm_batch_run(lgs_rtcsm_batch* b, const lgs_grid* grid, const lgs_grid* coarse) {
    return csm_run_impl(b, grid, coarse, nullptr);
}

int lgs_rtcsm_batch_run_timed(lgs_rtcsm_batch* b, const lgs_grid* grid, const lgs_grid* coarse,
                              float* ms) {
    if (!ms) return LGS_ERR_INVALID;
    return csm_run_impl(b, grid, coarse, ms);
}

int lgs_rtcsm_batch_results(lgs_rtcsm_batch* b, const lgs_grid* grid, const lgs_grid* coarse,
                            lgs_match_result* out) {
    if (!b || !grid || !coarse || (!out && b->nMatch > 0)) return LGS_ERR_INVALID;
    lgs_ctx* c = b->ctx;
    if (!b->ran) return lgs_fail(c, LGS_ERR_INVALID, "rtcsm_batch_results before run");
    if (b->nMatch == 0) return LGS_OK;
    LGS_CUDA(c, cudaSetDevice(c->device));
    const CsmWindow& w = b->win;
    LGS_CUDA(c, cudaMemcpyAsync(b->hFlagCount.p, b->dFlagCount.p, sizeof(int),
                                cudaMemcpyDeviceToHost, c->stream));
    LGS_CUDA(c, cudaMemcpyAsync(b->hResults.p, b->dResults.p, b->nMatch * sizeof(DevResult),
                                cudaMemcpyDeviceToHost, c->stream));
    LGS_CUDA(c, cudaStreamSynchronize(c->stream));
    int nFlag = *b->hFlagCount.p;
    std::fill(b->fixups.begin(), b->fixups.end(), 0);
    if (nFlag > b->flagCap) {
        // More near-edge points than the list holds (only with a widened guard band): grow the list
        // and project again -- the projection is deterministic, so it now records every one of them.
        b->flagCap = nFlag + nFlag / 8;
        LGS_CUDA(c, b->dFlags.reserve(b->flagCap));
        LGS_CUDA(c, cudaMemsetAsync(b->dFlagCount.p, 0, sizeof(int), c->stream));
        const int rcp = csm_launch_project(b);
        if (rcp != LGS_OK) return rcp;
        LGS_CUDA(c, cudaMemcpyAsync(b->hFlagCount.p, b->dFlagCount.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        LGS_CUDA(c, cudaStreamSynchronize(c->stream));
        nFlag = *b->hFlagCount.p;
        if (nFlag > b->flagCap)
            return lgs_fail(c, LGS_ERR_OVERFLOW, "rtcsm: %d near-edge points exceed the regrown fix-up list", nFlag);
    }
    if (nFlag > 0) {
        // Rare path: re-derive the flagged points with the host's libm (the reference's own
        // arithmetic, sensor_data.hpp:162-173 + grid_map.hpp:779-790), patch, and redo the sweep.
        std::vector<FlagEntry> fl(nFlag);
        LGS_CUDA(c, cudaMemcpy(fl.data(), b->dFlags.p, nFlag * sizeof(FlagEntry), cudaMemcpyDeviceToHost));
        std::vector<int> offVal(nFlag);
        std::vector<int2> cellVal(nFlag);
        std::vector<long long> where(2 * (size_t)nFlag);
        const int xLo = -w.winX, xHi = -w.winX + w.nxw - 1, yLo = -w.winY, yHi = -w.winY + w.nyw - 1;
        for (int k = 0; k < nFlag; ++k) {
            const CsmDesc& d = b->descs[fl[k].m];
            const int t = fl[k].t, i = fl[k].i;
            const double theta = d.st + d.stepT * static_cast<double>(t - d.winT);
            const double a = theta + b->hAngles[d.beamBegin + i];
            const double cosT = std::cos(a), sinT = std::sin(a);
            const double r = b->hRanges[d.beamBegin + i];
            const double hx = d.sx + r * cosT, hy = d.sy + r * sinT;
            const int cx = static_cast<int>(std::floor((hx - b->geom.minX) / b->geom.res));
            const int cy = static_cast<int>(std::floor((hy - b->geom.minY) / b->geom.res));
            const int ccx = std::min(std::max(cx, -xHi - 1), b->geom.nx - xLo);
            const int ccy = std::min(std::max(cy, -yHi - 1), b->geom.ny - yLo);
            offVal[k] = ccy * b->geom.pitch + ccx;
            cellVal[k] = make_int2(cx, cy);
            where[2 * k] = d.offBegin + (long long)t * d.nKeptPad + i;
            where[2 * k + 1] = d.cellBegin + (long long)t * d.nKept + i;
            b->fixups[fl[k].m]++;
        }
        LGS_CUDA(c, b->dFixOff.reserve(nFlag));
        LGS_CUDA(c, b->dFixCell.reserve(nFlag));
        LGS_CUDA(c, b->dFixWhere.reserve(2 * (size_t)nFlag));
        int* dOffVal = b->dFixOff.p; int2* dCellVal = b->dFixCell.p; long long* dWhere = b->dFixWhere.p;
        LGS_CUDA(c, cudaMemcpy(dOffVal, offVal.data(), nFlag * sizeof(int), cudaMemcpyHostToDevice));
        LGS_CUDA(c, cudaMemcpy(dCellVal, cellVal.data(), nFlag * sizeof(int2), cudaMemcpyHostToDevice));
        LGS_CUDA(c, cudaMemcpy(dWhere, where.data(), 2 * (size_t)nFlag * sizeof(long long), cudaMemcpyHostToDevice));
        csm_patch_kernel<<<(nFlag + 127) / 128, 128, 0, c->stream>>>(nullptr, dOffVal, dCellVal, dWhere,
                                                                     nFlag, b->dOffs.p, b->dCells.p);
        LGS_LAUNCH_CHECK(c);
        const int rc = csm_rescore_results(b, grid, coarse);
        if (rc != LGS_OK) return rc;
        // The patched offsets stay valid for a re-run of results(); a new run() re-projects.
        LGS_CUDA(c, cudaMemsetAsync(b->dFlagCount.p, 0, sizeof(int), c->stream));
    }
    bool needFull = false;
    for (int m = 0; m < b->nMatch; ++m) needFull |= b->hResults.p[m].needFull != 0;
    if (needFull) {   // the select flagged those matches: this pass scores all of their tiles
        const int rc = csm_rescore_results(b, grid, coarse);
        if (rc != LGS_OK) return rc;
    }
    for (int m = 0; m < b->nMatch; ++m) {
        const DevResult& r = b->hResults.p[m];
        const CsmDesc& d = b->descs[m];
        lgs_match_result& o = out[m];
        o.found = r.found; o.ix = r.ix; o.iy = r.iy; o.it = r.it;
        o.win_x = w.winX; o.win_y = w.winY; o.win_t = d.winT;
        o.n_fixups = b->fixups[m];
        o.step_x = b->geom.res; o.step_y = b->geom.res; o.step_t = d.stepT;
        o.score = r.score;
        o.n_scored = (long long)d.nT * ((long long)w.nxw * w.nyw + (long long)w.nbx * w.nby);
        o.exact_replay = r.exactReplay;
        o.reserved = 0;
    }
    return LGS_OK;
}

int lgs_rtcsm_batch_debug(lgs_rtcsm_batch* b, int m, int* dims, double* fine, double* coarse,
                          int* cells) {
    if (!b || m < 0 || m >= b->nMatch) return LGS_ERR_INVALID;
    lgs_ctx* c = b->ctx;
    if (!b->ran) return lgs_fail(c, LGS_ERR_INVALID, "rtcsm_batch_debug before run");
    LGS_CUDA(c, cudaSetDevice(c->device));
    if ((fine || coarse) && !b->tablesFull) {   // after a pruned run: fill both tables with the exhaustive sweep
        LGS_CUDA(c, lgs_grid_acquire(c, b->lastGrid));
        LGS_CUDA(c, lgs_grid_acquire(c, b->lastCoarse));
        const int rc = csm_launch_sweep(b, b->lastGrid, b->lastCoarse);
        if (rc != LGS_OK) return rc;
    }
    LGS_CUDA(c, cudaStreamSynchronize(c->stream));
    const CsmDesc& d = b->descs[m];
    const CsmWindow& w = b->win;
    if (dims) { dims[0] = d.nT; dims[1] = w.nxw; dims[2] = w.nyw; dims[3] = w.nbx; dims[4] = w.nby; dims[5] = d.nKept; }
    if (fine)
        LGS_CUDA(c, cudaMemcpy(fine, b->dFine.p + d.fineBegin,
                               (size_t)d.nT * w.nxw * w.nyw * sizeof(double), cudaMemcpyDeviceToHost));
    if (coarse)
        LGS_CUDA(c, cudaMemcpy(coarse, b->dCoarse.p + d.coarseBegin,
                               (size_t)d.nT * w.nbx * w.nby * sizeof(double), cudaMemcpyDeviceToHost));
    if (cells && d.nKept > 0)
        LGS_CUDA(c, cudaMemcpy(cells, b->dCells.p + d.cellBegin,
                               (size_t)d.nT * d.nKept * sizeof(int2), cudaMemcpyDeviceToHost));
    return LGS_OK;
}

int lgs_rtcsm_batch_work(const lgs_rtcsm_batch* b, long long* hyp, long long* gathers) {
    if (!b) return LGS_ERR_INVALID;
    if (hyp) *hyp = b->workHyp;
    if (gathers) *gathers = b->workGather;
    return LGS_OK;
}

int lgs_rtcsm_batch_fine_tiles(lgs_rtcsm_batch* b, long long* scored, long long* total) {
    if (!b) return LGS_ERR_INVALID;
    lgs_ctx* c = b->ctx;
    if (!b->ran) return lgs_fail(c, LGS_ERR_INVALID, "rtcsm_batch_fine_tiles before run");
    long long n = b->nTilesAll;
    if (b->win.rows && b->nMatch > 0) {
        LGS_CUDA(c, cudaSetDevice(c->device));
        int k = 0;
        LGS_CUDA(c, cudaMemcpyAsync(&k, b->dTileCount.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        LGS_CUDA(c, cudaStreamSynchronize(c->stream));
        n = k;
    }
    if (scored) *scored = n;
    if (total) *total = b->nTilesAll;
    return LGS_OK;
}

int lgs_rtcsm_match(lgs_ctx* ctx, const lgs_grid* grid, const lgs_grid* coarse,
                    const lgs_rtcsm_params* params, const lgs_scan_batch* scans,
                    const double* normThr, lgs_match_result* out) {
    lgs_rtcsm_batch* b = nullptr;
    int rc = lgs_rtcsm_batch_create(ctx, params, &b);
    if (rc != LGS_OK) return rc;
    rc = lgs_rtcsm_batch_upload(b, grid, scans, normThr);
    if (rc == LGS_OK) rc = lgs_rtcsm_batch_run(b, grid, coarse);
    if (rc == LGS_OK) rc = lgs_rtcsm_batch_results(b, grid, coarse, out);
    lgs_rtcsm_batch_destroy(b);
    return rc;
}

}  // extern "C"
