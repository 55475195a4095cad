// lgs_internal.cuh -- shared declarations of the sm_100a backend (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "lgs_b200.h"

struct lgs_grid {
    lgs_ctx* ctx = nullptr;
    int nx = 0, ny = 0, apron = 0;
    int pitch = 0;        // nx + 2 * apron (cells)
    int rows = 0;         // ny + 2 * apron
    double min_x = 0, min_y = 0, res = 0;
    // Window into a larger map (large-map row bands, SURVEY 8(e) C5): the grid stores cells
    // [off, off + n) of a map whose cell (0, 0) has its corner at (min_x, min_y); world -> cell
    // conversions stay global (bit-identical to the whole map) and subtract the offset.
    int off_x = 0, off_y = 0;
    bool owns = true;     // false for pyramid levels (views into the pyramid's slab)
    mutable bool foreign = false;   // a stream of ANOTHER context has read it (lgs_grid_acquire): destroy drains the device
    double* d = nullptr;  // rows * pitch doubles; cell (x, y) at d[(y + apron) * pitch + x + apron]
    __host__ __device__ const double* origin() const { return d + (size_t)apron * pitch + apron; }
    __host__ __device__ double* origin() { return d + (size_t)apron * pitch + apron; }
};

int lgs_fail(lgs_ctx* ctx, int code, const char* fmt, ...);

#define LGS_CUDA(ctx, call)                                                              \
    do {                                                                                 \
        cudaError_t e__ = (call);                                                        \
        if (e__ != cudaSuccess)                                                          \
            return lgs_fail((ctx), LGS_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__,   \
                            #call, cudaGetErrorString(e__));                             \
    } while (0)

#define LGS_LAUNCH_CHECK(ctx)                                                            \
    do {                                                                                 \
        (ctx)->launches++;                                                               \
        LGS_CUDA((ctx), cudaGetLastError());                                             \
    } while (0)

// Simple growable device / pinned-host buffers owned by batch objects.  Growth is geometric: a
// request a little above the capacity (scratch sizes follow the data, e.g. the ray lengths of a
// scan) must not cost a cudaFree + cudaMalloc pair -- milliseconds each -- call after call.
template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        size_t want = std::max(n, cap + cap / 2);
        cap = 0;
        cudaError_t e = cudaMalloc(&p, want * sizeof(T));
        if (e != cudaSuccess && want > n) {          // the head room is optional
            cudaGetLastError();
            want = n;
            e = cudaMalloc(&p, want * sizeof(T));
        }
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

template <typename T>
struct PinBuf {
    T* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        const size_t want = std::max(n, cap + cap / 2);
        cap = 0;
        cudaError_t e = cudaMallocHost(&p, want * sizeof(T));
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// Persistent scratch of lgs_grid_integrate_scans (grown on demand, freed with the context).
struct lgs_integ_ws {
    // Staging of one call (host inputs, pre-pass results, counters).  Two sets: an asynchronous caller
    // (lgs_grid_integrate_submit / _wait) stages call k + 1 on the copy stream while the chunks of call k
    // still read set k.
    struct Stage {
        DevBuf<double> sensor, hit;
        DevBuf<char> tab;                    // GridRef per map, hit offset per scan (+ end), map index per scan
        DevBuf<char> meta;                   // ScanMeta per scan
        DevBuf<int2> rel;                    // per beam: hit cell - sensor cell
        DevBuf<unsigned long long> counters;
        PinBuf<char> hMeta;
        PinBuf<unsigned long long> hCounters;
        cudaEvent_t evDone = nullptr;        // the call's counters are back and its last fold is done
        cudaEvent_t evCounters = nullptr;
        bool pending = false;                // submitted, not yet waited for
        void release() {
            sensor.release(); hit.release(); tab.release(); meta.release(); rel.release();
            counters.release(); hMeta.release(); hCounters.release();
            if (evDone) cudaEventDestroy(evDone);
            if (evCounters) cudaEventDestroy(evCounters);
            evDone = evCounters = nullptr; pending = false;
        }
    } stage[2];
    unsigned long long calls = 0;            // calls submitted so far (set = calls & 1)
    int nPending = 0;
    cudaStream_t copyStream = nullptr;       // staging + pre-pass of a call
    DevBuf<unsigned> kmin, kmax;             // per (tile, scan): beam index range [kmin, kmax)
    // Double buffered: the fold pass of chunk k (own stream) overlaps the mark / pairs / touch
    // passes of chunk k + 1 -- across calls too.
    DevBuf<uint2> tileInfo[2];               // per tile: {first pair, pairs}
    DevBuf<int4> pairs[2];                   // two int4 per (tile, scan) pair
    DevBuf<unsigned> records[2];             // per (pair, cell): encoded ordered touch sequence
    DevBuf<unsigned> side[2];                // raw touch / hit bitmap words of sequences no record holds
    cudaStream_t foldStream = nullptr;
    cudaEvent_t evTouch[2] = {nullptr, nullptr}, evFold[2] = {nullptr, nullptr};
    bool usedBuf[2] = {false, false};
    unsigned long long chunks = 0;           // chunks queued so far (buffer = chunks & 1)
    size_t cleanTiles = 0;                   // kmin / kmax are in their reset state up to here
    bool dirty = false;                      // a call failed between the mark and the pair pass
    long long fallbackCells = 0;
    DevBuf<char> regions;                    // region tables of the rounds with several chunks
    // per-scan update counts of a call that asks for each map's count (lgs_grid_integrate_many, synchronous)
    DevBuf<unsigned long long> touches;
    PinBuf<unsigned long long> hTouches;
    // Device projection of lgs_grid_construct_many (the projected hits themselves go into stage[].hit):
    // raw beams, per-scan inputs and hit counts / offsets, the upper interval ends and the beam of every hit,
    // per-map bbox keys and geometry, and the host fix-up lists (bbox candidates, near-edge hits).
    struct Construct {
        DevBuf<double> angles, ranges, hi, geo;
        DevBuf<char> scans;
        DevBuf<int> count, begin, beam, flags;
        DevBuf<unsigned long long> keys;
        DevBuf<int2> cand, edge;
        DevBuf<double> patch;
        PinBuf<int> hCount, hFlags;
        PinBuf<int2> hList;
        void release() {
            angles.release(); ranges.release(); hi.release(); geo.release(); scans.release(); count.release();
            begin.release(); beam.release(); flags.release(); keys.release(); cand.release(); edge.release();
            patch.release(); hCount.release(); hFlags.release(); hList.release();
        }
    } con;
    long long conBboxPoints = 0, conEdgePoints = 0;   // points re-derived on the host (lgs_ctx_construct_host_points)
    void release() {
        stage[0].release(); stage[1].release();
        kmin.release(); kmax.release();
        regions.release(); touches.release(); hTouches.release(); con.release();
        for (int b = 0; b < 2; ++b) {
            tileInfo[b].release(); pairs[b].release(); records[b].release(); side[b].release();
            if (evTouch[b]) cudaEventDestroy(evTouch[b]);
            if (evFold[b]) cudaEventDestroy(evFold[b]);
            evTouch[b] = evFold[b] = nullptr;
            usedBuf[b] = false;
        }
        if (foldStream) cudaStreamDestroy(foldStream);
        if (copyStream) cudaStreamDestroy(copyStream);
        foldStream = copyStream = nullptr;
        cleanTiles = 0; nPending = 0;
    }
};

// Scratch of the cost-function entry points (lgs_cost.cu).
struct lgs_cost_ws;
void lgs_cost_ws_destroy(lgs_cost_ws* ws);

// Tuning / diagnostic / test hooks of one context.  The LGS_* environment variables only supply the
// DEFAULTS, read once in lgs_ctx_create; afterwards lgs_ctx_set_option is the only way to change
// them, so no run path reads the environment or any process-global state.
struct lgs_opts {
    double edgeEps = 1e-9;      // "edge_eps"        fractional-cell guard band (see below)
    int csmFlat = 0;            // "csm_flat"        LGS_CSM_FLAT: flattened correlative sweep
    int bbSync = 0;             // "bb_sync"         LGS_BB_SYNC: level-synchronous B&B runs only
    int bbTable = 0;            // "bb_table"        LGS_BB_TABLE: level-synchronous runs through the full index table
    int bbWarpBelow = 8192;     // "bb_warp_below"   LGS_BB_WARP_BELOW: node count below which a level scores a warp per node
    int bbResolveUlps = 8;      // "bb_resolve_ulps" half width (ulps of cos / sin) of the on-device near-edge resolution
    int bbBlocksPerSm = 0;      // "bb_blocks_per_sm" persistent B&B kernel residency (0 = occupancy limit)
    double bbCost[4] = {100.0, 60.0, 36.0, 21.0};   // "bb_cost_g1/g4/g8/g32" per-pass cost (us) of the warp mappings
    int bbHostTiming = 0;       // "bb_host_timing"  LGS_BB_HOSTTIMING
    int bbCountNodes = 0;       // "bb_count_nodes": lgs_match_result::n_scored per query instead of per batch
    int bbEarlyReject = 1;      // "bb_early_reject" LGS_BB_EARLY_REJECT: device-only run stops hopeless sums early
    int integHostTiming = 0;    // "integ_host_timing" LGS_INTEG_HOSTTIMING
    double integHostTimingMinMs = 1.0;  // "integ_host_timing_min_ms" LGS_INTEG_HOSTTIMING_MIN_MS: report calls slower than this
    int integTiming = 0;        // "integ_timing"    LGS_INTEG_TIMING
    int integDiag = 0;          // "integ_diag"      LGS_INTEG_DIAG
    long long integSideWords = 0; // "integ_side_words" LGS_INTEG_SIDE_WORDS (0 = default size)
    double integResolveUlps = 8.0;  // "integ_resolve_ulps" half width (ulps of cos / sin) of lgs_grid_construct_many's intervals
    int gsTables = 0;           // "gs_tables"       LGS_GS_TABLES: grid search through the index tables
};

struct lgs_ctx {
    lgs_opts opt;
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaMemPool_t pool = nullptr;            // PRIVATE stream-ordered pool (grids, pyramid slabs, call scratch)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t evOrder = nullptr;           // cross-context ordering (lgs_grid_acquire)
    int sm_count = 148;
    int bbBlocks = 0;         // grid of the persistent branch-and-bound kernel (0: not yet sized)
    long long launches = 0;
    char err[512] = {0};
    DevBuf<double> scratch;   // reusable device scratch (precompute intermediate)
    lgs_integ_ws* integ = nullptr;
    lgs_cost_ws* cost = nullptr;
};

// Fractional-cell guard band (in cells): a projected coordinate closer than this to a cell
// edge is re-derived on the host with glibc sin/cos, because CUDA's double sin/cos may
// differ from glibc's in the last ulp (SURVEY.md H5).  Device-vs-host differences are
// below 1e-11 cells for |coordinates| < 1e4 m, so 1e-9 leaves two orders of magnitude.
#define LGS_EDGE_EPS_DEFAULT 1e-9

// ScanData::HitPoint with glibc cos / sin in the reference's operation order (lgs_host.cu): the host
// arithmetic every device projection is checked against.
void lgs_hit_point_host(const double* sensorPose, double angle, double r, double* hx, double* hy);

// Stream-ordered allocation from the context's private pool (freed with cudaFreeAsync).
inline cudaError_t lgs_alloc_async(lgs_ctx* c, void** p, size_t bytes) {
    return cudaMallocFromPoolAsync(p, bytes, c->pool, c->stream);
}
template <typename T>
inline cudaError_t lgs_alloc_async(lgs_ctx* c, T** p, size_t bytes) {
    return lgs_alloc_async(c, reinterpret_cast<void**>(p), bytes);
}
// Context `user` is about to read grid `g` on its stream.  If the grid belongs to another context
// (the builder's latest map read by the matcher's context), everything already queued on the owner's
// stream is ordered before the reader, and the grid remembers the foreign reader so that destroying
// it drains the device first (its buffer is freed stream-ordered on the OWNER's stream only).
cudaError_t lgs_grid_acquire(lgs_ctx* user, const lgs_grid* g);

// Pyramid levels are plain grids sharing the geometry of the map they were built from.
const lgs_grid* lgs_pyramid_level(const lgs_pyramid* p, int level);
// A matcher of context `user` is about to read the pyramid (its slab is freed stream-ordered on the
// owner's stream, so foreign readers make the destroy synchronise the device first).
void lgs_pyramid_note_user(const lgs_pyramid* p, const lgs_ctx* user);
