// lgs_integrate.cu -- occupancy-grid scan integration on sm_100a.
//
// Replaces the integration loops of GridMapBuilder::UpdateGridMap / ConstructMapFromScans
// (mapping/grid_map_builder.cpp:170-186, :311-328): for every beam that passed the range
// filter, the cells on Bresenham(sensorCell -> hitCell) (util.hpp:257-303) except the last get
// Update(pMiss), the last gets Update(pHit) (BinaryBayesGridCell::Update,
// grid_map/binary_bayes_grid_cell.hpp:75-119).
//
// The cell update is order dependent at the bit level (SURVEY.md H7): each cell must see its
// touches in (scan, beam) order, so updates cannot be scattered with atomics.  But WHICH touches a
// cell sees, and in which order, does not depend on the cell values.  The work is therefore split
// like a tiled rasteriser, over chunks of <= 64 scans:
//
//   1. mark   one thread per (scan, beam) walks the reference's Bresenham and, whenever the ray
//             enters another 16x16-cell tile, folds its beam index into the tile's [kmin, kmax)
//             range for that scan (idempotent atomics: min / max / or -- order free);
//   2. pairs  every tile turns its scan mask into a contiguous, scan-ordered run of
//             (tile, scan, kmin, kmax) pairs;
//   3. touch  fully parallel over the pairs: one block per pair drops the cells of the beams
//             kmin..kmax that fall into the tile into per-cell bitmaps in shared memory (bit = beam,
//             so ascending bits ARE the CPU's beam order), using the closed form of the
//             reference's Bresenham (step k of a ray is independent of step k - 1):
//                 x-major (|dx| > |dy|):  y_k = y0 + sy * floor((2|dy|k + |dx|) / (2|dx|)),  k = 0..|dx|
//                 y-major (otherwise)  :  x_k = x0 + sx * floor((2|dx|k + |dy|) / (2|dy|)),  k = 0..|dy|
//             (cells k < length are misses, k = length is the hit), then every cell packs its
//             ordered miss/hit sequence into one 32-bit record (raw bits up to 26 touches,
//             three run lengths beyond -- the near field is M^a H^b M^c);
//   4. fold   one thread OWNS one cell and applies the records of its tile in scan order with
//             exactly the CPU's IEEE sequence (div/mul/add intrinsics, no FMA), leaving a run early
//             once the value reaches its fixed point (the probability clamp makes runs idempotent).
//
// Nothing depends on beams being angularly sorted: an unsorted scan only widens [kmin, kmax).
// A record that fits neither format (alternating hits and misses in a cell crossed by > 26 beams)
// is marked, and the owner re-derives that (cell, scan) by testing the beams kmin..kmax itself.
#include <cmath>

#include <chrono>

#include "lgs_internal.cuh"

namespace {

constexpr int kTile = 16;                      // tile side (cells)
constexpr int kTileShift = 4;
constexpr int kTileCells = kTile * kTile;      // = threads per block of the touch / fold passes
constexpr int kChunk = 64;                     // scans per chunk (one mask bit each)
constexpr int kSeg = 128;                      // beams per shared-memory bitmap segment
constexpr int kSegWords = kSeg / 32;
constexpr unsigned kRawMax = 26;               // touches a raw record holds
constexpr unsigned kRecOverflow = 0xFFFFFFFFu;
constexpr unsigned kRecSide = 31u << 26;
constexpr int kFoldBatch = 8;                  // records a fold thread keeps in flight
constexpr size_t kRecordBudget = (size_t)1 << 30;   // bytes of records per chunk before it is split

struct ScanMeta {
    int sx, sy;          // sensor cell
    int beamBegin, n;    // beams of this scan
    int maxLen;          // max Chebyshev ray length in cells
    int bad;             // a touched cell lies outside the grid
};

struct GridRef {
    double* origin;
    int nx, ny, pitch;
    double minX, minY, res;
};

GridRef gridRef(lgs_grid* g) { return GridRef{g->origin(), g->nx, g->ny, g->pitch, g->min_x, g->min_y, g->res}; }

// A chunk's tile region (x0, y0, tw) inside a ROUND, the set of chunks -- of different maps -- that one
// launch of each pass covers: the round's regions share one tile index space and one mark-pass grid.
struct Region {
    GridRef g;
    int x0, y0, tw;      // tile-aligned origin (cells), tiles per region row
    int tileBase;        // first tile of the region in the round's tile index space
    int scanBase;        // first scan of the chunk (index into the call's ScanMeta)
    int rowBase;         // first mark-pass row (blockIdx.y) of the chunk
};

// Region source of a round with one chunk (every round of a one-map call): nothing to look up.
struct OneRegion {
    Region r;            // tileBase == rowBase == 0
    __device__ __forceinline__ Region byTile(int) const { return r; }
    __device__ __forceinline__ Region byRow(int) const { return r; }
};
// Region source of a round with several chunks: the last region whose base is <= the index (bases ascend).
struct RegionTable {
    const Region* __restrict__ r;
    int n;
    __device__ __forceinline__ Region byTile(int t) const {
        int lo = 0, hi = n - 1;
        while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (r[mid].tileBase <= t) lo = mid; else hi = mid - 1; }
        return r[lo];
    }
    __device__ __forceinline__ Region byRow(int y) const {
        int lo = 0, hi = n - 1;
        while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (r[mid].rowBase <= y) lo = mid; else hi = mid - 1; }
        return r[lo];
    }
};

__device__ __forceinline__ double clampProb(double v) {
    // std::clamp(v, ProbabilityMin, ProbabilityMax)  (binary_bayes_grid_cell.hpp:50-52, :97-101)
    const double lo = 1e-3, hi = 1.0 - 1e-3;
    return v < lo ? lo : (hi < v ? hi : v);
}

// BinaryBayesGridCell<double>::Update (binary_bayes_grid_cell.hpp:75-92); oddsP = ValueToOdds(p).
__device__ __forceinline__ double bayesUpdate(double v, double p, double oddsP) {
    if (v == 0.0) return clampProb(p);
    const double cv = clampProb(v);
    const double oldOdds = __ddiv_rn(cv, __dsub_rn(1.0, cv));           // ValueToOdds
    const double o = __dmul_rn(oldOdds, oddsP);
    const double nv = clampProb(__ddiv_rn(o, __dadd_rn(1.0, o)));       // OddsToValue
    return clampProb(nv);
}

// 0 = not on the ray, 1 = miss cell, 2 = hit cell.  (rx, ry) = cell - sensorCell, (ex, ey) = hitCell - sensorCell.
// Division free: with k the step along the major axis, the reference's minor coordinate is
// floor((2|minor| k + |major|) / (2|major|)) (util.hpp:276-299), i.e. the cell is on the ray iff
//     2|major| t <= 2|minor| k + |major| < 2|major| (t + 1),   t = signed minor offset >= 0.
__device__ __forceinline__ int rayTouch(int rx, int ry, int ex, int ey) {
    const int ax = abs(ex), ay = abs(ey);
    int k, t, amaj, amin;
    if (ax > ay) {                                   // x-major (util.hpp:276-287)
        k = ex < 0 ? -rx : rx; t = ey < 0 ? -ry : ry; amaj = ax; amin = ay;
    } else {                                         // y-major (util.hpp:288-299), also dx == dy == 0
        k = ey < 0 ? -ry : ry; t = ex < 0 ? -rx : rx; amaj = ay; amin = ax;
    }
    if (k < 0 || k > amaj || t < 0) return 0;
    const int lhs = 2 * amin * k + amaj;             // < 2^31 for maps below 16k cells per side
    const int m2 = 2 * amaj;
    if (amaj == 0) return (t == 0) ? 2 : 0;          // zero-length ray: the sensor cell is the hit
    if (m2 * t > lhs || lhs >= m2 * (t + 1)) return 0;
    return k == amaj ? 2 : 1;
}

// Minor-axis offset of step k of a ray: floor((2 amin k + amaj) / (2 amaj)) (util.hpp:276-299), amaj > 0.
// For rays up to 2047 cells the dividend is below 2^24, i.e. exact in float: one reciprocal, one
// multiply and an integer correction replace the 32-bit division; longer rays divide.
__device__ __forceinline__ int minorAt(int amin, int amaj, int k) {
    const int lhs = 2 * amin * k + amaj, m2 = 2 * amaj;
    if (amaj > 2047) return (int)((unsigned)lhs / (unsigned)m2);
    int q = __float2int_rz(__fmul_rn((float)lhs, __frcp_rn((float)m2)));
    const int r = lhs - q * m2;
    if (r < 0) --q; else if (r >= m2) ++q;
    return q;
}

// ---- pre-pass A: sensor cells ---------------------------------------------------------------------
// Scan s belongs to grids[mapOf[s]].
__global__ void integ_sensor_kernel(const double* __restrict__ sensorXY, const int* __restrict__ hitBegin,
                                    int nScans, const GridRef* __restrict__ grids, const int* __restrict__ mapOf,
                                    ScanMeta* __restrict__ meta) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nScans) return;
    const GridRef g = grids[mapOf[s]];
    ScanMeta m;
    // WorldCoordinateToGridCellIndex (grid_map.hpp:779-790)
    m.sx = __double2int_rd(__ddiv_rn(__dsub_rn(sensorXY[2 * s], g.minX), g.res));
    m.sy = __double2int_rd(__ddiv_rn(__dsub_rn(sensorXY[2 * s + 1], g.minY), g.res));
    m.beamBegin = hitBegin[s];
    m.n = hitBegin[s + 1] - hitBegin[s];
    m.maxLen = 0;
    m.bad = (m.sx < 0 || m.sx >= g.nx || m.sy < 0 || m.sy >= g.ny) ? 1 : 0;
    meta[s] = m;
}

// ---- pre-pass B: per beam end cell relative to the sensor cell ---------------------------------------
// touches (NULL = not wanted): per scan, the Update calls of the CPU, one per cell of each ray.
__global__ void integ_beam_kernel(const double* __restrict__ hitXY, const GridRef* __restrict__ grids,
                                  const int* __restrict__ mapOf, ScanMeta* __restrict__ meta,
                                  int2* __restrict__ rel, unsigned long long* __restrict__ touches) {
    const int s = blockIdx.y;
    const GridRef g = grids[mapOf[s]];
    const int n = meta[s].n, beamBegin = meta[s].beamBegin, sx = meta[s].sx, sy = meta[s].sy;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int len = 0;
    if (i < n) {
        const size_t b = (size_t)beamBegin + i;
        const double2 h = reinterpret_cast<const double2*>(hitXY)[b];
        const int ex = __double2int_rd(__ddiv_rn(__dsub_rn(h.x, g.minX), g.res));
        const int ey = __double2int_rd(__ddiv_rn(__dsub_rn(h.y, g.minY), g.res));
        if (ex < 0 || ex >= g.nx || ey < 0 || ey >= g.ny) atomicOr(&meta[s].bad, 1);
        const int dx = ex - sx, dy = ey - sy;
        rel[b] = make_int2(dx, dy);
        len = max(abs(dx), abs(dy));
    }
    if (touches) {
        unsigned cells = i < n ? (unsigned)len + 1u : 0u;
        for (int o = 16; o > 0; o >>= 1) cells += __shfl_xor_sync(0xffffffffu, cells, o);
        if ((threadIdx.x & 31) == 0 && cells) atomicAdd(touches + s, (unsigned long long)cells);
    }
    for (int o = 16; o > 0; o >>= 1) len = max(len, __shfl_xor_sync(0xffffffffu, len, o));
    if ((threadIdx.x & 31) == 0 && len > 0) atomicMax(&meta[s].maxLen, len);
}

// ---- 1. mark: beam index range per (tile, scan) ------------------------------------------------------
// One thread per (scan, beam, 16-step piece of the ray); a warp = 32 consecutive beams at the same
// distance from the sensor, which mostly cross the same tiles.  A 16-step piece of a (monotone)
// Bresenham path visits at most 3 tiles; for each of them the warp groups the lanes that share the
// tile and issues ONE atomicMin (lowest beam of the group) and ONE atomicMax (highest beam).
// Row blockIdx.y = scan s of the chunk of region R; its tiles are R.tileBase + the tile in R's region.
template <class Regions>
__global__ void __launch_bounds__(128)
integ_mark_kernel(const ScanMeta* __restrict__ meta, const int2* __restrict__ rel, Regions regions,
                  int beamsPad, unsigned* __restrict__ kmin, unsigned* __restrict__ kmax) {
    const Region R = regions.byRow(blockIdx.y);
    const int s = blockIdx.y - R.rowBase;
    const ScanMeta m = meta[R.scanBase + s];
    const int t = blockIdx.x * blockDim.x + threadIdx.x;        // beamsPad is a multiple of 32:
    const int i = t % beamsPad, piece = t / beamsPad;           // a warp never straddles two pieces
    const int lane = threadIdx.x & 31;
    int tiles[3] = {-1, -1, -1};
    if (i < m.n) {
        const int2 e = __ldg(rel + m.beamBegin + i);
        const int ax = abs(e.x), ay = abs(e.y);
        const bool xMajor = ax > ay;                            // util.hpp:276 vs :288
        const int amaj = xMajor ? ax : ay, amin = xMajor ? ay : ax;
        const int kBegin = piece * kTile;
        if (kBegin <= amaj) {
            const int kEnd = min(kBegin + kTile - 1, amaj);
            const int sMaj = (xMajor ? e.x : e.y) < 0 ? -1 : 1, sMin = (xMajor ? e.y : e.x) < 0 ? -1 : 1;
            const int bx = m.sx - R.x0, by = m.sy - R.y0;
            const int m2 = 2 * amaj, d2 = 2 * amin;
            int minor = amaj ? minorAt(amin, amaj, kBegin) : 0;
            int rem = d2 * kBegin + amaj - minor * m2;
            int nt = 0, last = -1;
            for (int k = kBegin; k <= kEnd; ++k) {
                const int x = bx + (xMajor ? sMaj * k : sMin * minor);
                const int y = by + (xMajor ? sMin * minor : sMaj * k);
                const int tile = R.tileBase + (y >> kTileShift) * R.tw + (x >> kTileShift);
                if (tile != last) {
                    last = tile;
                    if (nt == 0) tiles[0] = tile; else if (nt == 1) tiles[1] = tile; else tiles[2] = tile;
                    ++nt;
                }
                rem += d2;
                if (rem >= m2) { rem -= m2; ++minor; }
            }
        }
    }
#pragma unroll
    for (int u = 0; u < 3; ++u) {
        const int mine = tiles[u];
        unsigned pending = __ballot_sync(0xffffffffu, mine >= 0);
        while (pending) {
            const int leader = __ffs(pending) - 1;
            const int tl = __shfl_sync(0xffffffffu, mine, leader);
            const unsigned grp = __ballot_sync(0xffffffffu, mine == tl);
            if (lane == leader) {
                const size_t idx = (size_t)tl * kChunk + s;
                atomicMin(kmin + idx, (unsigned)i);                             // lowest lane = lowest beam
                atomicMax(kmax + idx, (unsigned)(i + (31 - __clz(grp)) - lane) + 1u);
            }
            pending &= ~grp;
        }
    }
}

// ---- 2. pairs: scan-ordered pair descriptors per tile; resets the mark buffers --------------------------
// Descriptor = two int4: {ox, oy, k0, k1} (tile origin relative to the scan's sensor cell, beam range)
// and {beamBegin, tile, scan, 0}, so the touch pass needs no further dependent look-ups.
// One warp per tile: lanes read the tile's 64 kmax entries (non-zero = the scan touches the tile).
template <class Regions>
__global__ void __launch_bounds__(128)
integ_pairs_kernel(int nTiles, const ScanMeta* __restrict__ meta, Regions regions,
                   unsigned* __restrict__ kmin, unsigned* __restrict__ kmax,
                   uint2* __restrict__ tileInfo, int4* __restrict__ pairs, unsigned* __restrict__ nPairs) {
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (t >= nTiles) return;
    const Region R = regions.byTile(t);
    const int lt = t - R.tileBase;
    const size_t idx = (size_t)t * kChunk + lane;
    const unsigned hiA = kmax[idx], hiB = kmax[idx + 32];
    const unsigned mA = __ballot_sync(0xffffffffu, hiA != 0u), mB = __ballot_sync(0xffffffffu, hiB != 0u);
    const unsigned cnt = (unsigned)(__popc(mA) + __popc(mB));
    unsigned base = 0;
    if (cnt && lane == 0) base = atomicAdd(nPairs, cnt);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (lane == 0) tileInfo[t] = make_uint2(base, cnt);
    const unsigned below = (1u << lane) - 1u;
    const int tx = R.x0 + (lt % R.tw) * kTile, ty = R.y0 + (lt / R.tw) * kTile;
    auto emit = [&](unsigned slot, int s, unsigned lo, unsigned hi) {
        const ScanMeta m = meta[R.scanBase + s];
        pairs[2 * (size_t)slot] = make_int4(tx - m.sx, ty - m.sy, (int)lo, (int)hi);
        pairs[2 * (size_t)slot + 1] = make_int4(m.beamBegin, t, s, 0);
    };
    if (hiA) {
        emit(base + __popc(mA & below), lane, kmin[idx], hiA);
        kmin[idx] = 0xFFFFFFFFu; kmax[idx] = 0u;
    }
    if (hiB) {
        emit(base + __popc(mA) + __popc(mB & below), lane + 32, kmin[idx + 32], hiB);
        kmin[idx + 32] = 0xFFFFFFFFu; kmax[idx + 32] = 0u;
    }
}

// ---- 3. touch: ordered miss/hit sequence of every cell of a (tile, scan) pair ----------------------------
// Record formats (32 bit):   0                      no touch
//   raw  [31] = 0, [30:26] = count (1..26), [25:0] = types in order (1 = hit)
//   runs [31] = 1, [30] = type of the first run, [29:20] [19:10] [9:0] = three alternating run lengths
//   side [31] = 0, [30:26] = 31, [25:0] = offset (units of 8 words) of the cell's non-empty raw
//        touch / hit bitmap words in the side buffer: sequences that fit neither format (a near cell whose
//        beams alternate between ending in it and passing through)
//   0xFFFFFFFF               side buffer exhausted: the owner re-derives the sequence from the beams
struct TouchSeq {
    unsigned cnt = 0, raw = 0, r0 = 0, r1 = 0, r2 = 0;
    int nrun = 0, cur = -1, first = 0;
    __device__ __forceinline__ void append(int type, unsigned n) {
        if (cnt < kRawMax && type) raw |= (n >= 32u ? 0xFFFFFFFFu : ((1u << n) - 1u)) << cnt;
        cnt += n;
        if (type != cur) { cur = type; if (++nrun == 1) first = type; }
        if (nrun == 1) r0 += n; else if (nrun == 2) r1 += n; else if (nrun == 3) r2 += n;
    }
    __device__ __forceinline__ unsigned record() const {
        if (cnt == 0) return 0u;
        if (cnt <= kRawMax) return (cnt << 26) | (raw & ((1u << 26) - 1u));
        if (nrun <= 3 && r0 < 1023u && r1 < 1023u && r2 < 1023u)
            return 0x80000000u | ((unsigned)first << 30) | (r0 << 20) | (r1 << 10) | r2;
        return kRecOverflow;
    }
};

__global__ void __launch_bounds__(kTileCells, 4)
integ_touch_kernel(const int2* __restrict__ rel, const int4* __restrict__ pairs,
                   const unsigned* __restrict__ nPairs, unsigned* __restrict__ records, unsigned* __restrict__ side,
                   unsigned* __restrict__ sideCursor, unsigned sideCap,
                   unsigned long long* __restrict__ counters) {
    __shared__ unsigned sBits[2][2 * kSegWords * kTileCells];   // double buffered; [touch | hit][word][cell]
    int buf = 0;
    __shared__ unsigned sSum[kTileCells / 32];
    const int tid = threadIdx.x;
    const unsigned nP = *nPairs;
    unsigned total = 0, overflow = 0;
    int4 nextA = make_int4(0, 0, 0, 0), nextB = nextA;
    // Threads per beam in the scatter step: 4 (4 steps each) for segments of <= 64 beams, else 2.
    auto lanesPerBeam = [](int nb) { return nb <= kTileCells / 4 ? 4 : 2; };
    int2 eNext = make_int2(0, 0);                            // this thread's beam of the next pair's first segment
    if (blockIdx.x < nP) {
        nextA = pairs[2 * (size_t)blockIdx.x]; nextB = pairs[2 * (size_t)blockIdx.x + 1];
        const int nb = min(kSeg, nextA.w - nextA.z), b = tid / lanesPerBeam(nb);
        if (b < nb) eNext = __ldg(rel + nextB.x + nextA.z + b);
    }
    for (unsigned p = blockIdx.x; p < nP; p += gridDim.x) {
        const int4 pr = nextA;                              // .x/.y tile origin - sensor cell, .z/.w beams
        const int2* __restrict__ E = rel + nextB.x;
        const int2 eFirst = eNext;
        const bool more = p + gridDim.x < nP;
        if (more) {                                         // the next descriptor is in flight meanwhile
            nextA = pairs[2 * (size_t)(p + gridDim.x)];
            nextB = pairs[2 * (size_t)(p + gridDim.x) + 1];
        }
        bool fetched = false;
        const int ox = pr.x, oy = pr.y;
        TouchSeq seq;
        unsigned rec = 0u, sideOff = 0u;
        int wFirst = 0x7fffffff, wLast = -1;                   // non-empty bitmap words of this cell
        // pass 0 builds the records; pass 1 (only if a cell of this pair fits no record format)
        // repeats the bitmaps and streams the raw words of those cells to the side buffer
        for (int pass = 0; pass < 2; ++pass) {
            for (int seg = pr.z; seg < pr.w; seg += kSeg) {
                // Two barriers per segment: the buffer cleared here was last read two segments ago.
                buf ^= 1;
                unsigned* sTouch = sBits[buf];
                unsigned* sHit = sBits[buf] + kSegWords * kTileCells;
                const int nW = (min(kSeg, pr.w - seg) + 31) >> 5;
                for (int w = 0; w < nW; ++w) { sTouch[w * kTileCells + tid] = 0u; sHit[w * kTileCells + tid] = 0u; }
                __syncthreads();
                const int nb = min(kSeg, pr.w - seg);
                const int per = lanesPerBeam(nb), b = tid / per;
                if (b < nb) {
                    // `per` threads per beam share the <= 16 steps whose major coordinate lies inside
                    // the tile; the minor coordinate floor((2 amin k + amaj) / (2 amaj)) is divided
                    // out once per thread and then carried with its remainder (2 amin <= 2 amaj: at
                    // most one increment a step)
                    const int2 e = (pass == 0 && seg == pr.z) ? eFirst : __ldg(E + seg + b);
                    const int ax = abs(e.x), ay = abs(e.y);
                    const bool xMajor = ax > ay;
                    const int amaj = xMajor ? ax : ay, amin = xMajor ? ay : ax;
                    const int eMaj = xMajor ? e.x : e.y, eMin = xMajor ? e.y : e.x;
                    const int oMaj = xMajor ? ox : oy, oMin = xMajor ? oy : ox;
                    const int steps = kTile / per, sub = tid - b * per;
                    const int kBase = (eMaj >= 0 ? oMaj : -oMaj - (kTile - 1)) + sub * steps;
                    const int kLo = max(kBase, 0);
                    const int kHi = min(kBase + steps - 1, amaj);
                    if (kLo <= kHi) {
                        const int m2 = 2 * amaj, d2 = 2 * amin;
                        int minor = amaj ? minorAt(amin, amaj, kLo) : 0;
                        int rem = d2 * kLo + amaj - minor * m2;
                        const unsigned bitb = 1u << (b & 31);
                        unsigned* tw_ = sTouch + (b >> 5) * kTileCells;
                        unsigned* hw_ = sHit + (b >> 5) * kTileCells;
                        for (int k = kLo; k <= kHi; ++k) {
                            const int j = eMaj >= 0 ? k - oMaj : -k - oMaj;              // column (row) in the tile
                            const int lMin = (eMin < 0 ? -minor : minor) - oMin;
                            if ((unsigned)lMin < (unsigned)kTile) {
                                const int cell = xMajor ? (lMin * kTile + j) : (j * kTile + lMin);
                                atomicOr(tw_ + cell, bitb);
                                if (k == amaj) atomicOr(hw_ + cell, bitb);
                            }
                            rem += d2;
                            if (rem >= m2) { rem -= m2; ++minor; }
                        }
                    }
                }
                if (more && !fetched) {                     // next pair's beams: in flight during the extraction
                    fetched = true;
                    const int nbN = min(kSeg, nextA.w - nextA.z), bN = tid / lanesPerBeam(nbN);
                    if (bN < nbN) eNext = __ldg(rel + nextB.x + nextA.z + bN);
                }
                __syncthreads();
                if (pass == 0) {
                    for (int w = 0; w < nW; ++w) {
                        unsigned t = sTouch[w * kTileCells + tid];
                        if (t == 0u) continue;
                        const int gw = ((seg - pr.z) / kSeg) * kSegWords + w;
                        wFirst = min(wFirst, gw); wLast = gw;
                        const unsigned h = sHit[w * kTileCells + tid];
                        while (t) {                              // maximal runs of equal type, ascending beams
                            const int type = (h >> (__ffs(t) - 1)) & 1;
                            const unsigned same = type ? (t & h) : (t & ~h);
                            const unsigned other = t & ~same;
                            const unsigned upto = other ? ((1u << (__ffs(other) - 1)) - 1u) : 0xFFFFFFFFu;
                            const unsigned run = same & upto;
                            seq.append(type, (unsigned)__popc(run));
                            t &= ~run;
                        }
                    }
                } else if ((rec >> 26) == 31u) {
                    unsigned* out = side + (size_t)sideOff + 2;
                    for (int w = 0; w < nW; ++w) {
                        const int gw = ((seg - pr.z) / kSeg) * kSegWords + w;
                        if (gw < wFirst || gw > wLast) continue;
                        out[2 * (gw - wFirst)] = sTouch[w * kTileCells + tid];
                        out[2 * (gw - wFirst) + 1] = sHit[w * kTileCells + tid];
                    }
                }
            }
            if (pass == 0) {
                rec = seq.record();
                if (rec == kRecOverflow) {
                    // header {first word | words << 16, -} + (touch, hit) word pairs, in units of 8 words
                    const unsigned nWords = (unsigned)(wLast - wFirst + 1);
                    const unsigned words = (2u + 2u * nWords + 7u) & ~7u;
                    sideOff = atomicAdd(sideCursor, words);
                    if (sideOff + words <= sideCap && nWords < 65536u) {
                        rec = kRecSide | (sideOff >> 3);
                        side[sideOff] = (unsigned)wFirst | (nWords << 16);
                    }
                }
                if (!__syncthreads_or((rec >> 26) == 31u)) break;
            }
        }
        records[(size_t)p * kTileCells + tid] = rec;
        total += seq.cnt;
        overflow += rec == kRecOverflow ? 1u : 0u;
    }
    // one atomic per block: touches (= Update calls of the CPU) and overflowed records
    unsigned v = total | 0u;
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    unsigned ov = overflow;
    for (int o = 16; o > 0; o >>= 1) ov += __shfl_down_sync(0xffffffffu, ov, o);
    if ((tid & 31) == 0) sSum[tid >> 5] = v;
    __syncthreads();
    if (tid == 0) {
        unsigned long long tot = 0;
        for (int k = 0; k < kTileCells / 32; ++k) tot += sSum[k];
        if (tot) atomicAdd(counters, tot);
    }
    if ((tid & 31) == 0 && ov) atomicAdd(counters + 1, (unsigned long long)ov);
}

// ---- 4. fold: one thread owns one cell ---------------------------------------------------------------
struct FoldArgs {
    const int2* rel;
    const uint2* tileInfo;
    const int4* pairs;
    const unsigned* records;
    const unsigned* side;
    unsigned long long* diag;      // LGS_INTEG_TIMING: [2] max / [3] sum of computed updates per thread
    double pHit, pMiss, oddsHit, oddsMiss;
};

// One thread owns one cell.  Raw records (the common case) are queued per lane and applied only when
// some lane of the warp is about to overflow its 64-touch queue: neighbouring cells see similar
// numbers of touches over a chunk, so the lanes of a warp then have similar amounts of work, while
// applying every record at once would run the ~100-instruction update under heavy divergence.
// A touch that cannot change the value (cell already at the clamp the observation pushes towards:
// the clamp makes the update idempotent there) is skipped without arithmetic.
struct Folder {
    const FoldArgs& a;
    double v;
    unsigned long long q = 0ull;
    int qn = 0;
    bool missSat, hitSat;
    unsigned computed = 0;
    __device__ __forceinline__ Folder(const FoldArgs& args, double v0) : a(args), v(v0) {
        const double lo = 1e-3, hi = 1.0 - 1e-3;
        missSat = bayesUpdate(lo, a.pMiss, a.oddsMiss) == lo;
        hitSat = bayesUpdate(hi, a.pHit, a.oddsHit) == hi;
    }
    __device__ __forceinline__ bool saturated(bool hit) const {
        return hit ? (hitSat && v == 1.0 - 1e-3) : (missSat && v == 1e-3);
    }
    __device__ __forceinline__ void touch(bool hit) {
        if (!saturated(hit)) { v = bayesUpdate(v, hit ? a.pHit : a.pMiss, hit ? a.oddsHit : a.oddsMiss); ++computed; }
    }
    // Every iteration performs exactly one COMPUTED update per lane: a lane first drops, without
    // iterating, the leading touches that cannot change a value sitting on a clamp, so a warp
    // iterates max-over-lanes(computed updates) times, not max-over-lanes(queue length) times.
    __device__ __forceinline__ void drain() {
        while (qn) {
            const bool atLo = missSat && v == 1e-3, atHi = hitSat && v == 1.0 - 1e-3;
            if (atLo || atHi) {
                const unsigned long long x = atLo ? q : ~q;            // first touch of the other type
                const int n = min(qn, x ? __ffsll((long long)x) - 1 : 64);
                q = n >= 64 ? 0ull : q >> n;
                qn -= n;
                if (!qn) break;
            }
            const bool hit = q & 1ull;
            v = bayesUpdate(v, hit ? a.pHit : a.pMiss, hit ? a.oddsHit : a.oddsMiss);
            ++computed;
            q >>= 1; --qn;
        }
    }
    __device__ __forceinline__ void run(bool hit, unsigned n) {
        for (unsigned j = 0; j < n; ++j) {
            if (saturated(hit)) break;
            const double nv = bayesUpdate(v, hit ? a.pHit : a.pMiss, hit ? a.oddsHit : a.oddsMiss);
            ++computed;
            if (nv == v) break;            // fixed point: the rest of the run is a no-op
            v = nv;
        }
    }
};

template <class Regions>
__global__ void __launch_bounds__(kTileCells)
integ_fold_kernel(FoldArgs a, Regions regions) {
    const uint2 info = a.tileInfo[blockIdx.x];
    if (info.y == 0u) return;
    const Region reg = regions.byTile(blockIdx.x);
    const GridRef& g = reg.g;
    const int lt = blockIdx.x - reg.tileBase;
    const int tid = threadIdx.x;
    const int cx = reg.x0 + (lt % reg.tw) * kTile + (tid & (kTile - 1));
    const int cy = reg.y0 + (lt / reg.tw) * kTile + (tid >> kTileShift);
    const bool inside = cx < g.nx && cy < g.ny;
    double* cell = g.origin + (size_t)cy * g.pitch + cx;
    const double v0 = inside ? *cell : 0.0;
    Folder f(a, v0);
    // Records are prefetched kFoldBatch pairs at a time (they do not depend on the cell value): the
    // loads of the next batch are in flight while this thread's own column of the shared staging
    // buffer is consumed, so a tile touched by all 64 scans pays 8 memory round trips, not 64.
    __shared__ unsigned sRec[kFoldBatch * kTileCells];
    const unsigned* __restrict__ R = a.records + (size_t)info.x * kTileCells + tid;
    unsigned pre[kFoldBatch];
#pragma unroll
    for (int u = 0; u < kFoldBatch; ++u) pre[u] = (unsigned)u < info.y ? __ldcs(R + (size_t)u * kTileCells) : 0u;
    for (unsigned j = 0; j < info.y; ++j) {
        const unsigned u0 = j % kFoldBatch;
        if (u0 == 0u) {
#pragma unroll
            for (int u = 0; u < kFoldBatch; ++u) sRec[u * kTileCells + tid] = pre[u];
#pragma unroll
            for (int u = 0; u < kFoldBatch; ++u) {
                const unsigned jj = j + kFoldBatch + u;
                pre[u] = jj < info.y ? __ldcs(R + (size_t)jj * kTileCells) : 0u;
            }
        }
        const unsigned rec = sRec[u0 * kTileCells + tid];
        if (__any_sync(0xffffffffu, f.qn > 64 - (int)kRawMax)) f.drain();
        const unsigned cnt = rec >> 26;
        if (cnt <= kRawMax) {                                   // raw (or empty): queue
            f.q |= (unsigned long long)(rec & ((1u << 26) - 1u)) << f.qn;
            f.qn += (int)cnt;
            continue;
        }
        f.drain();
        if (rec == kRecOverflow) {
            const int4 pr = a.pairs[2 * (size_t)(info.x + j)];
            const int2* __restrict__ E = a.rel + a.pairs[2 * (size_t)(info.x + j) + 1].x;
            const int rx = pr.x + (tid & (kTile - 1)), ry = pr.y + (tid >> kTileShift);
            for (int i = pr.z; i < pr.w; ++i) {
                const int2 e = __ldg(E + i);
                const int ty = rayTouch(rx, ry, e.x, e.y);
                if (ty) f.touch(ty == 2);
            }
        } else if (cnt == 31u) {
            const unsigned* __restrict__ S = a.side + (size_t)(rec & ((1u << 26) - 1u)) * 8u;
            const unsigned nWords = S[0] >> 16;
            const uint2* __restrict__ W = reinterpret_cast<const uint2*>(S + 2);
            uint2 nx = W[0];
            for (unsigned w = 0; w < nWords; ++w) {
                unsigned t = nx.x;
                const unsigned h = nx.y;
                if (w + 1 < nWords) nx = W[w + 1];
                while (t) {
                    const bool hit = (h >> (__ffs(t) - 1)) & 1u;
                    const unsigned same = hit ? (t & h) : (t & ~h);
                    const unsigned other = t & ~same;
                    const unsigned upto = other ? ((1u << (__ffs(other) - 1)) - 1u) : 0xFFFFFFFFu;
                    const unsigned run = same & upto;
                    f.run(hit, (unsigned)__popc(run));
                    t &= ~run;
                }
            }
        } else {                                                // three alternating runs
            const bool first = (rec >> 30) & 1u;
            f.run(first, (rec >> 20) & 1023u);
            f.run(!first, (rec >> 10) & 1023u);
            f.run(first, rec & 1023u);
        }
    }
    f.drain();
    if (a.diag) { atomicMax(a.diag + 2, (unsigned long long)f.computed); atomicAdd(a.diag + 3, (unsigned long long)f.computed); }
    if (inside && f.v != v0) *cell = f.v;
}

__global__ void grid_shift_copy_kernel(const double* __restrict__ src, int srcNx, int srcNy, int srcPitch,
                                       double* __restrict__ dst, int dstNx, int dstNy, int dstPitch,
                                       int shiftX, int shiftY) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (x >= dstNx || y >= dstNy) return;
    const int ox = x + shiftX, oy = y + shiftY;
    double v = 0.0;
    if (ox >= 0 && ox < srcNx && oy >= 0 && oy < srcNy) v = src[(size_t)oy * srcPitch + ox];
    dst[(size_t)y * dstPitch + x] = v;
}

// ---- lgs_grid_construct_many: projection of raw scans ------------------------------------------------
// ConstructMapFromScans (grid_map_builder.cpp:227-332) projects every beam with glibc cos / sin.  The device's
// sincos may differ from glibc in the last ulps, so every hit is carried as an interval [lo, hi] that contains
// glibc's value: the CPU's expression sx + r * cos(st + a) evaluated, in its operation order, at cos +- U ulps
// (every operation is monotone; r may have either sign, so lo / hi are the smaller / larger end).  A cell whose
// floor is equal at both ends is the CPU's cell; the bbox extremes and the near-edge hits are settled on the host
// with glibc (DESIGN.md section 3.4).
struct ConScan {
    double sx, sy, st;          // sensor pose
    double rmin, rmax;          // usable range window: a beam is used unless r >= rmax || r <= rmin
    int beamBegin, n;           // beams [beamBegin, beamBegin + n) of the call
    int map;
};
constexpr int kConThreads = 256;                 // one block per scan
enum { kConBad = 0, kConCand = 1, kConEdge = 2 };   // ConFlags: first bad scan, bbox candidates, near-edge hits

// Unsigned keys that order like the doubles they encode (no NaN): per-map bbox bounds by integer atomics.
__host__ __device__ inline unsigned long long conKey(unsigned long long bits) {
    return (bits >> 63) ? ~bits : (bits | 0x8000000000000000ull);
}

__device__ __forceinline__ bool conUsed(double r, const ConScan& q) { return !(r >= q.rmax || r <= q.rmin); }   // :365-366

// Sum over the block of one int per thread.
__device__ __forceinline__ int conBlockSum(int v, int* sh) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    int t = 0;
    for (int w = 0; w < kConThreads / 32; ++w) t += sh[w];
    __syncthreads();
    return t;
}

// Used beams per scan; the first scan with a non-finite angle or range on a used beam.
__global__ void __launch_bounds__(kConThreads)
con_count_kernel(const ConScan* __restrict__ scans, const double* __restrict__ angles, const double* __restrict__ ranges,
                 int* __restrict__ count, int* __restrict__ flags) {
    __shared__ int sh[kConThreads / 32];
    const int s = blockIdx.x;
    const ConScan q = scans[s];
    int k = 0;
    bool bad = false;
    for (int i = threadIdx.x; i < q.n; i += kConThreads) {
        const double r = ranges[q.beamBegin + i];
        if (!conUsed(r, q)) continue;
        ++k;
        bad |= !isfinite(r) || !isfinite(angles[q.beamBegin + i]);
    }
    if (bad) atomicMin(flags + kConBad, s);
    k = conBlockSum(k, sh);
    if (threadIdx.x == 0) count[s] = k;
}

// begin[s] = hits of the scans before s (one block; begin[n] = all hits).
__global__ void __launch_bounds__(1024) con_offsets_kernel(const int* __restrict__ count, int n, int* __restrict__ begin) {
    __shared__ int sh[1024];
    const int per = (n + 1023) / 1024, s0 = min(n, (int)threadIdx.x * per), s1 = min(n, s0 + per);
    int sum = 0;
    for (int s = s0; s < s1; ++s) sum += count[s];
    sh[threadIdx.x] = sum;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {                 // inclusive scan of the segment sums
        const int v = threadIdx.x >= (unsigned)o ? sh[threadIdx.x - o] : 0;
        __syncthreads();
        sh[threadIdx.x] += v;
        __syncthreads();
    }
    int run = sh[threadIdx.x] - sum;
    for (int s = s0; s < s1; ++s) { begin[s] = run; run += count[s]; }
    if (threadIdx.x == 1023) begin[n] = sh[1023];
}

// Hits of scan s in beam order at begin[s]: lo -> hit (the staging buffer of the integration), hi -> hi, the
// call's beam index -> beam.  A non-finite end makes the interval (-inf, inf).  Per map, keys[4 m + ..] take
// the bbox bounds the device can prove: [0] / [1] min over hits of hi.x / hi.y (min sides), [2] / [3] max of
// lo.x / lo.y (max sides); the host seeds them with the sensor positions and the reference's initial values.
__global__ void __launch_bounds__(kConThreads)
con_project_kernel(const ConScan* __restrict__ scans, const double* __restrict__ angles,
                   const double* __restrict__ ranges, const int* __restrict__ begin, double ulps,
                   double2* __restrict__ lo, double2* __restrict__ hi, int* __restrict__ beam,
                   unsigned long long* __restrict__ keys) {
    __shared__ int sh[kConThreads / 32];
    __shared__ double sr[4][kConThreads / 32];
    const int s = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const ConScan q = scans[s];
    const double k = ulps * 2.220446049250313e-16, inf = __longlong_as_double(0x7ff0000000000000ll);
    double bnd[4] = {inf, inf, -inf, -inf};
    int base = begin[s];
    for (int c0 = 0; c0 < q.n; c0 += kConThreads) {
        const int i = c0 + threadIdx.x;
        const double r = i < q.n ? ranges[q.beamBegin + i] : 0.0;
        const bool used = i < q.n && conUsed(r, q);
        const unsigned m = __ballot_sync(0xffffffffu, used);
        if (lane == 0) sh[warp] = __popc(m);
        __syncthreads();
        int off = base, tot = 0;
        for (int w = 0; w < kConThreads / 32; ++w) { off += w < warp ? sh[w] : 0; tot += sh[w]; }
        __syncthreads();
        base += tot;
        if (!used) continue;
        off += __popc(m & ((1u << lane) - 1u));
        double sn, cs;
        sincos(__dadd_rn(q.st, angles[q.beamBegin + i]), &sn, &cs);            // sensor_data.hpp:168-169
        const double wc = __dadd_rn(__dmul_rn(fabs(cs), k), 4.9406564584124654e-324);
        const double ws = __dadd_rn(__dmul_rn(fabs(sn), k), 4.9406564584124654e-324);
        const double x0 = __dadd_rn(q.sx, __dmul_rn(r, __dsub_rn(cs, wc))), x1 = __dadd_rn(q.sx, __dmul_rn(r, __dadd_rn(cs, wc)));
        const double y0 = __dadd_rn(q.sy, __dmul_rn(r, __dsub_rn(sn, ws))), y1 = __dadd_rn(q.sy, __dmul_rn(r, __dadd_rn(sn, ws)));
        const bool fx = isfinite(x0) && isfinite(x1), fy = isfinite(y0) && isfinite(y1);
        const double2 l = make_double2(fx ? fmin(x0, x1) : -inf, fy ? fmin(y0, y1) : -inf);
        const double2 h = make_double2(fx ? fmax(x0, x1) : inf, fy ? fmax(y0, y1) : inf);
        lo[off] = l;
        hi[off] = h;
        beam[off] = q.beamBegin + i;
        bnd[0] = fmin(bnd[0], h.x); bnd[1] = fmin(bnd[1], h.y);
        bnd[2] = fmax(bnd[2], l.x); bnd[3] = fmax(bnd[3], l.y);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        double v = bnd[j];
        for (int o = 16; o > 0; o >>= 1) {
            const double u = __shfl_xor_sync(0xffffffffu, v, o);
            v = j < 2 ? fmin(v, u) : fmax(v, u);
        }
        if (lane == 0) sr[j][warp] = v;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        const int j = threadIdx.x;
        double v = sr[j][0];
        for (int w = 1; w < kConThreads / 32; ++w) v = j < 2 ? fmin(v, sr[j][w]) : fmax(v, sr[j][w]);
        const unsigned long long key = conKey((unsigned long long)__double_as_longlong(v));
        if (j < 2) atomicMin(keys + 4 * q.map + j, key); else atomicMax(keys + 4 * q.map + j, key);
    }
}

// Hits that may hold a bbox extreme (hi >= the max side's bound, lo <= the min side's): {call beam, sides}
// into cand[0 .. cap), every one counted in flags[kConCand].
__global__ void __launch_bounds__(kConThreads)
con_candidates_kernel(const ConScan* __restrict__ scans, const int* __restrict__ begin, const double2* __restrict__ lo,
                      const double2* __restrict__ hi, const int* __restrict__ beam,
                      const unsigned long long* __restrict__ keys, int2* __restrict__ cand, int cap, int* __restrict__ flags) {
    const int s = blockIdx.x;
    const unsigned long long* K = keys + 4 * scans[s].map;
    const unsigned long long k0 = K[0], k1 = K[1], k2 = K[2], k3 = K[3];
    for (int b = begin[s] + threadIdx.x; b < begin[s + 1]; b += kConThreads) {
        const double2 l = lo[b], h = hi[b];
        const int sides = (conKey((unsigned long long)__double_as_longlong(l.x)) <= k0 ? 1 : 0) |
                          (conKey((unsigned long long)__double_as_longlong(l.y)) <= k1 ? 2 : 0) |
                          (conKey((unsigned long long)__double_as_longlong(h.x)) >= k2 ? 4 : 0) |
                          (conKey((unsigned long long)__double_as_longlong(h.y)) >= k3 ? 8 : 0);
        if (!sides) continue;
        const int slot = atomicAdd(flags + kConCand, 1);
        if (slot < cap) cand[slot] = make_int2(beam[b], sides);
    }
}

// Hits whose interval ends fall into different cells of their map's new geometry (geo[3 m ..] = min_x, min_y,
// res): {hit, call beam} into edge[0 .. cap), every one counted in flags[kConEdge].  The cells are the
// integration's (integ_beam_kernel), so a hit that is not listed keeps lo, which lies in the CPU's cell.
__global__ void __launch_bounds__(kConThreads)
con_edge_kernel(const ConScan* __restrict__ scans, const int* __restrict__ begin, const double2* __restrict__ lo,
                const double2* __restrict__ hi, const int* __restrict__ beam, const double* __restrict__ geo,
                int2* __restrict__ edge, int cap, int* __restrict__ flags) {
    const int s = blockIdx.x;
    const double* G = geo + 3 * scans[s].map;
    const double minX = G[0], minY = G[1], res = G[2];
    auto cell = [&](double p, double mn) { return __double2int_rd(__ddiv_rn(__dsub_rn(p, mn), res)); };
    for (int b = begin[s] + threadIdx.x; b < begin[s + 1]; b += kConThreads) {
        const double2 l = lo[b], h = hi[b];
        if (cell(l.x, minX) == cell(h.x, minX) && cell(l.y, minY) == cell(h.y, minY)) continue;
        const int slot = atomicAdd(flags + kConEdge, 1);
        if (slot < cap) edge[slot] = make_int2(b, beam[b]);
    }
}

// The host's glibc hit of every near-edge hit, in the order of the edge list.
__global__ void con_patch_kernel(const int2* __restrict__ edge, const double2* __restrict__ val, int n,
                                 double2* __restrict__ hit) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) hit[edge[k].x] = val[k];
}

}  // namespace

extern "C" {

}  // extern "C"

namespace {

// The grid takes nx x ny cells at (minX, minY) in a fresh buffer, on its own context's stream; with `copy`, new
// cell (x, y) takes old cell (x + shiftX, y + shiftY) (one launch), otherwise every cell is unknown.
int grid_replace(lgs_grid* g, int nx, int ny, double minX, double minY, bool copy, int shiftX, int shiftY);

// Completion of the OLDEST submitted call: its update count, the fallback statistics, its staging set.
int integ_wait(lgs_ctx* c, long long* nUpdatesOut) {
    if (nUpdatesOut) *nUpdatesOut = 0;
    if (!c->integ || c->integ->nPending == 0) return LGS_OK;
    lgs_integ_ws& w = *c->integ;
    lgs_integ_ws::Stage& st = w.stage[(w.calls - (unsigned long long)w.nPending) & 1];
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, cudaEventSynchronize(st.evDone));
    st.pending = false;
    --w.nPending;
    if (nUpdatesOut) *nUpdatesOut = (long long)st.hCounters.p[0];
    w.fallbackCells += (long long)st.hCounters.p[1];
    return LGS_OK;
}

// The checks of one (grid, scan batch) pair of a call; map = its index in the call.  b == NULL: the grid only
// (lgs_grid_construct_many checks its raw scans itself).
int integ_check(lgs_ctx* c, int map, const lgs_grid* g, const lgs_hit_batch* b) {
    if (!g) return lgs_fail(c, LGS_ERR_INVALID, "integrate: grid of map %d is NULL", map);
    if (b && (b->n_scans < 0 || (b->n_scans > 0 && (!b->sensor_xy || !b->hit_begin))))
        return lgs_fail(c, LGS_ERR_INVALID, "integrate: bad scan batch of map %d", map);
    if (b && b->n_scans > 0 && b->hit_begin[b->n_scans] > 0 && !b->hit_xy)
        return lgs_fail(c, LGS_ERR_INVALID, "integrate: hit_xy of map %d is NULL", map);
    if (g->off_x || g->off_y)
        return lgs_fail(c, LGS_ERR_INVALID, "integrate: grid of map %d is windowed (lgs_grid_set_window), not supported", map);
    if (g->ctx->device != c->device)
        return lgs_fail(c, LGS_ERR_INVALID, "integrate: grid of map %d lives on device %d, the context on %d", map,
                        g->ctx->device, c->device);
    return LGS_OK;
}

// The checks of a synchronous many-map call (`who` names it in the messages): nothing submitted in flight,
// every (grid, batch) pair, no grid twice.  batches == NULL: grids only.
int integ_check_many(lgs_ctx* c, const char* who, int nMaps, lgs_grid* const* grids, const lgs_hit_batch* batches) {
    if (c->integ && c->integ->nPending > 0)
        return lgs_fail(c, LGS_ERR_INVALID, "%s: an lgs_grid_integrate_submit call is in flight, wait for it first", who);
    for (int i = 0; i < nMaps; ++i) {
        const int rc = integ_check(c, i, grids[i], batches ? &batches[i] : nullptr);
        if (rc != LGS_OK) return rc;
    }
    std::vector<const lgs_grid*> sorted(grids, grids + nMaps);
    std::sort(sorted.begin(), sorted.end());
    if (std::adjacent_find(sorted.begin(), sorted.end()) != sorted.end())
        return lgs_fail(c, LGS_ERR_INVALID, "%s: the same grid appears twice", who);
    return LGS_OK;
}

// The integration workspace of a context, with its copy stream.
int integ_workspace(lgs_ctx* c) {
    if (!c->integ) c->integ = new lgs_integ_ws();
    if (!c->integ->copyStream) LGS_CUDA(c, cudaStreamCreateWithFlags(&c->integ->copyStream, cudaStreamNonBlocking));
    return LGS_OK;
}

// Everything of a call up to the last enqueue; the host waits only for the pre-pass (scan bounds).
// A call integrates batches[i] into grids[i], i < nMaps (checked by the caller): every map is staged into
// one blob behind a device table of grids, and the next chunk of every map goes into one round of
// launches.  perMap (NULL = not wanted) receives each map's update count.  hitsOnDevice: the hits are
// already in the staging set's hit buffer, at the call's hit offsets (lgs_grid_construct_many's device
// projection, queued on the copy stream), and batches[].hit_xy is not read.
int integ_submit(lgs_ctx* c, int nMaps, lgs_grid* const* grids, const lgs_hit_batch* batches, double pHit,
                 double pMiss, long long* perMap, bool hitsOnDevice = false) {
    // scans of map i are scans [scanBase[i], scanBase[i + 1]) of the call, their hits start at hitBase[i]
    std::vector<int> scanBase(nMaps + 1, 0);
    std::vector<long long> hitBase(nMaps + 1, 0);
    for (int i = 0; i < nMaps; ++i) {
        scanBase[i + 1] = scanBase[i] + batches[i].n_scans;
        hitBase[i + 1] = hitBase[i] + (batches[i].n_scans > 0 ? batches[i].hit_begin[batches[i].n_scans] : 0);
    }
    const int n = scanBase[nMaps];
    const long long total = hitBase[nMaps];
    if (n == 0) return LGS_OK;
    if (total > 0x7fffffffLL) return lgs_fail(c, LGS_ERR_INVALID, "integrate: %lld hits in one call (at most 2^31 - 1)", total);
    LGS_CUDA(c, cudaSetDevice(c->device));
    for (int i = 0; i < nMaps; ++i) LGS_CUDA(c, lgs_grid_acquire(c, grids[i]));
    const int rcWs = integ_workspace(c);
    if (rcWs != LGS_OK) return rcWs;
    lgs_integ_ws& ws = *c->integ;
    if (ws.nPending >= 2 || ws.stage[ws.calls & 1].pending)
        return lgs_fail(c, LGS_ERR_INVALID, "integrate: two calls are in flight, wait for the older one first");
    lgs_integ_ws::Stage& w0 = ws.stage[ws.calls & 1];
    if (!w0.evDone) {
        LGS_CUDA(c, cudaEventCreateWithFlags(&w0.evDone, cudaEventDisableTiming));
        LGS_CUDA(c, cudaEventCreateWithFlags(&w0.evCounters, cudaEventDisableTiming));
    }
    // `w` = the shared workspace with this call's staging set in front of it
    struct View {
        DevBuf<double>& sensor; DevBuf<double>& hit; DevBuf<char>& tab; DevBuf<char>& meta; DevBuf<int2>& rel;
        DevBuf<unsigned long long>& counters; PinBuf<char>& hMeta; PinBuf<unsigned long long>& hCounters;
        DevBuf<unsigned>& kmin; DevBuf<unsigned>& kmax;
        DevBuf<uint2>* tileInfo; DevBuf<int4>* pairs; DevBuf<unsigned>* records; DevBuf<unsigned>* side;
        cudaStream_t& foldStream; cudaEvent_t* evTouch; cudaEvent_t* evFold;
        size_t& cleanTiles; bool& dirty;
    } w{w0.sensor, w0.hit, w0.tab, w0.meta, w0.rel, w0.counters, w0.hMeta, w0.hCounters, ws.kmin, ws.kmax,
        ws.tileInfo, ws.pairs, ws.records, ws.side, ws.foldStream, ws.evTouch, ws.evFold, ws.cleanTiles, ws.dirty};
    cudaStream_t cs0 = ws.copyStream;
    // LGS_INTEG_HOSTTIMING=1 (diagnostic): host wall time of the call's phases to stderr when a call
    // takes longer than a millisecond.
    const bool hostTiming = c->opt.integHostTiming != 0;
    const auto tStart = std::chrono::steady_clock::now();
    auto msSince = [](std::chrono::steady_clock::time_point t) {
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t).count(); };
    double tStage = 0.0, tPre = 0.0, tLoop = 0.0;

    // Stage the whole batch once, on the copy stream (under the chunks of an earlier call that is still
    // running); the passes then run over chunks of <= 64 scans (one mask bit each).  The pre-pass finds the
    // grid of scan s as grids[mapOf[s]]: the grid table, the hit offsets rebased into the blob and mapOf
    // go in one copy (pageable host vector: the copy has taken it when cudaMemcpyAsync returns).
    const size_t tabBytes = (size_t)nMaps * sizeof(GridRef) + (size_t)(2 * n + 1) * sizeof(int);
    LGS_CUDA(c, w.sensor.reserve((size_t)n * 2));
    LGS_CUDA(c, w.hit.reserve(std::max<size_t>((size_t)total, 1) * 2));
    LGS_CUDA(c, w.tab.reserve(tabBytes));
    LGS_CUDA(c, w.meta.reserve((size_t)n * sizeof(ScanMeta)));
    LGS_CUDA(c, w.rel.reserve(std::max<size_t>((size_t)total, 1)));
    LGS_CUDA(c, w.counters.reserve(8));
    LGS_CUDA(c, w.hMeta.reserve((size_t)n * sizeof(ScanMeta)));
    LGS_CUDA(c, w.hCounters.reserve(8));
    std::vector<char> hTab(tabBytes);
    GridRef* tg = reinterpret_cast<GridRef*>(hTab.data());
    int* hBegin = reinterpret_cast<int*>(tg + nMaps);
    int* hMapOf = hBegin + n + 1;
    for (int i = 0; i < nMaps; ++i) {
        tg[i] = gridRef(grids[i]);
        for (int s = 0; s < batches[i].n_scans; ++s) {
            hBegin[scanBase[i] + s] = (int)(hitBase[i] + batches[i].hit_begin[s]);
            hMapOf[scanBase[i] + s] = i;
        }
    }
    hBegin[n] = (int)total;
    for (int i = 0; i < nMaps; ++i) {
        const lgs_hit_batch& b = batches[i];
        if (b.n_scans == 0) continue;
        LGS_CUDA(c, cudaMemcpyAsync(w.sensor.p + 2 * (size_t)scanBase[i], b.sensor_xy,
                                    (size_t)b.n_scans * 2 * sizeof(double), cudaMemcpyHostToDevice, cs0));
        if (!hitsOnDevice && hitBase[i + 1] > hitBase[i])
            LGS_CUDA(c, cudaMemcpyAsync(w.hit.p + 2 * (size_t)hitBase[i], b.hit_xy,
                                        (size_t)(hitBase[i + 1] - hitBase[i]) * 2 * sizeof(double),
                                        cudaMemcpyHostToDevice, cs0));
    }
    LGS_CUDA(c, cudaMemcpyAsync(w.tab.p, hTab.data(), tabBytes, cudaMemcpyHostToDevice, cs0));
    const GridRef* dGrids = reinterpret_cast<const GridRef*>(w.tab.p);
    const int* dBegin = reinterpret_cast<const int*>(dGrids + nMaps);
    const int* dMapOf = dBegin + n + 1;
    // per-scan update counts, only for perMap (the call's total is counters[0] of the touch pass)
    unsigned long long* dTouches = nullptr;
    if (perMap) {
        LGS_CUDA(c, ws.touches.reserve((size_t)n));
        LGS_CUDA(c, ws.hTouches.reserve((size_t)n));
        dTouches = ws.touches.p;
        LGS_CUDA(c, cudaMemsetAsync(dTouches, 0, (size_t)n * sizeof(unsigned long long), cs0));
    }
    LGS_CUDA(c, cudaMemsetAsync(w.counters.p, 0, 8 * sizeof(unsigned long long), cs0));
    tStage = msSince(tStart);

    int maxBeams = 0;
    for (int i = 0; i < nMaps; ++i)
        for (int s = 0; s < batches[i].n_scans; ++s)
            maxBeams = std::max(maxBeams, batches[i].hit_begin[s + 1] - batches[i].hit_begin[s]);
    ScanMeta* dMeta = reinterpret_cast<ScanMeta*>(w.meta.p);
    ScanMeta* hMeta = reinterpret_cast<ScanMeta*>(w.hMeta.p);
    // Pre-pass over the whole batch: sensor cells, relative end cells, ray lengths, bounds check.
    integ_sensor_kernel<<<(n + 127) / 128, 128, 0, cs0>>>(w.sensor.p, dBegin, n, dGrids, dMapOf, dMeta);
    LGS_LAUNCH_CHECK(c);
    for (int s0 = 0; maxBeams > 0 && s0 < n; s0 += 65535) {       // grid rows: at most 65535 scans a launch
        dim3 gb((maxBeams + 127) / 128, std::min(n - s0, 65535));
        integ_beam_kernel<<<gb, 128, 0, cs0>>>(w.hit.p, dGrids, dMapOf + s0, dMeta + s0, w.rel.p,
                                               dTouches ? dTouches + s0 : nullptr);
        LGS_LAUNCH_CHECK(c);
    }
    if (dTouches)
        LGS_CUDA(c, cudaMemcpyAsync(ws.hTouches.p, dTouches, (size_t)n * sizeof(unsigned long long),
                                    cudaMemcpyDeviceToHost, cs0));
    LGS_CUDA(c, cudaMemcpyAsync(hMeta, dMeta, (size_t)n * sizeof(ScanMeta), cudaMemcpyDeviceToHost, cs0));
    LGS_CUDA(c, cudaStreamSynchronize(cs0));
    tPre = msSince(tStart);
    for (int i = 0; i < nMaps; ++i)
        for (int s = scanBase[i]; s < scanBase[i + 1]; ++s)
            if (hMeta[s].bad)
                return lgs_fail(c, LGS_ERR_INVALID, "integrate: map %d, scan %d touches cells outside the %dx%d grid "
                                "(expand the map first, as GridMap::Expand does)", i, s - scanBase[i],
                                grids[i]->nx, grids[i]->ny);

    // ValueToOdds(prob) for the two observations (binary_bayes_grid_cell.hpp:104-113), host IEEE.
    auto clampP = [](double v) { const double lo = 1e-3, hi = 1.0 - 1e-3; return v < lo ? lo : (hi < v ? hi : v); };
    const double oddsHit = clampP(pHit) / (1.0 - clampP(pHit));
    const double oddsMiss = clampP(pMiss) / (1.0 - clampP(pMiss));

    // Side buffer for touch sequences that fit no record format (words; LGS_INTEG_SIDE_WORDS is a test
    // hook that shrinks it to exercise the exhaustive fallback).
    size_t sideCap = (size_t)8 << 20;
    if (c->opt.integSideWords > 0) sideCap = (size_t)std::max<long long>(8, c->opt.integSideWords);
    // tiles of scan s's reach: the square of half side maxLen around the sensor cell
    auto tileSpan = [](int lo, int hi) { return (hi >> kTileShift) - (lo >> kTileShift) + 1; };

    // LGS_INTEG_TIMING=1 (diagnostic): CUDA-event time of every pass, summed over the call, to stderr.
    const bool timing = c->opt.integTiming != 0;
    const bool diag = timing && c->opt.integDiag != 0;   // + per-cell update counts (slows the fold)
    std::vector<cudaEvent_t> evs;
    auto stamp = [&]() { if (timing) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, c->stream); evs.push_back(e); } };
    // The fold pass runs on a second stream so that it overlaps the next round's touch passes
    // (LGS_INTEG_TIMING serialises everything on the context stream to time the passes).
    const bool overlap = !timing;
    if (!w.foldStream) {
        LGS_CUDA(c, cudaStreamCreateWithFlags(&w.foldStream, cudaStreamNonBlocking));
        for (int b = 0; b < 2; ++b) {
            LGS_CUDA(c, cudaEventCreateWithFlags(&w.evTouch[b], cudaEventDisableTiming));
            LGS_CUDA(c, cudaEventCreateWithFlags(&w.evFold[b], cudaEventDisableTiming));
        }
    }
    // Rounds: consecutive chunks (below) share one launch of each pass while the round holds at most one chunk
    // per map (the fold owns the map's cells), and its records, tile index space and mark-pass rows stay within
    // the limits of one chunk.  A round is launched as soon as it is closed; one with several chunks takes its
    // regions from a table at its own place in ws.regions.  A one-chunk round (every round of a one-map call)
    // copies no table: that copy would run on the context stream while the fold of a call submitted before
    // this one may still be reading the table on the fold stream.
    struct Round { int first, count, rows, beams, len; size_t tiles, pairBound; };
    std::vector<Region> regions;
    LGS_CUDA(c, ws.regions.reserve((size_t)n * sizeof(Region)));   // a chunk holds >= 1 scan
    int lastBuf = -1;
    auto launchRound = [&](const Round& rd) -> int {
        const size_t nTiles = rd.tiles, pairBound = rd.pairBound;
        const OneRegion one{regions[rd.first]};
        RegionTable table{nullptr, rd.count};
        if (rd.count > 1) {
            Region* dst = reinterpret_cast<Region*>(ws.regions.p) + rd.first;
            LGS_CUDA(c, cudaMemcpyAsync(dst, regions.data() + rd.first, (size_t)rd.count * sizeof(Region),
                                        cudaMemcpyHostToDevice, c->stream));
            table.r = dst;
        }

        // mark buffers: kept in their reset state by the pair pass; (re)initialise what is new
        if (w.dirty) { w.cleanTiles = 0; w.dirty = false; }
        if (nTiles * kChunk > w.kmin.cap) w.cleanTiles = 0;           // reserve() reallocates
        LGS_CUDA(c, w.kmin.reserve(nTiles * kChunk));
        LGS_CUDA(c, w.kmax.reserve(nTiles * kChunk));
        const int buf = (int)(ws.chunks & 1);
        ++ws.chunks;
        // this buffer's previous fold (round k - 2, possibly of the previous call) must be done before it is
        // overwritten: the context stream waits for it; only a buffer that has to grow makes the host wait
        // (reallocation frees)
        if (ws.usedBuf[buf]) {
            const bool grows = nTiles > w.tileInfo[buf].cap || 2 * pairBound > w.pairs[buf].cap ||
                               pairBound * kTileCells > w.records[buf].cap || sideCap > w.side[buf].cap;
            if (grows) LGS_CUDA(c, cudaEventSynchronize(w.evFold[buf]));
            else LGS_CUDA(c, cudaStreamWaitEvent(c->stream, w.evFold[buf], 0));
        }
        LGS_CUDA(c, w.tileInfo[buf].reserve(nTiles));
        LGS_CUDA(c, w.pairs[buf].reserve(2 * pairBound));
        LGS_CUDA(c, w.records[buf].reserve(pairBound * kTileCells));
        LGS_CUDA(c, w.side[buf].reserve(sideCap));
        if (nTiles > w.cleanTiles) {
            const size_t a0 = w.cleanTiles, cnt = w.kmin.cap / kChunk - a0;   // initialise up to the capacity
            LGS_CUDA(c, cudaMemsetAsync(w.kmin.p + a0 * kChunk, 0xFF, cnt * kChunk * sizeof(unsigned), c->stream));
            LGS_CUDA(c, cudaMemsetAsync(w.kmax.p + a0 * kChunk, 0, cnt * kChunk * sizeof(unsigned), c->stream));
            w.cleanTiles = w.kmin.cap / kChunk;
        }
        unsigned* nPairs = reinterpret_cast<unsigned*>(w.counters.p + 4 + buf);   // [0] pairs, [1] side-buffer cursor
        LGS_CUDA(c, cudaMemsetAsync(nPairs, 0, 2 * sizeof(unsigned), c->stream));

        w.dirty = true;
        stamp();
        const int beamsPad = (rd.beams + 31) & ~31, pieces = rd.len / kTile + 1;
        dim3 gm((unsigned)(((size_t)beamsPad * pieces + 127) / 128), rd.rows);
        if (rd.count == 1) integ_mark_kernel<<<gm, 128, 0, c->stream>>>(dMeta, w.rel.p, one, beamsPad, w.kmin.p, w.kmax.p);
        else integ_mark_kernel<<<gm, 128, 0, c->stream>>>(dMeta, w.rel.p, table, beamsPad, w.kmin.p, w.kmax.p);
        LGS_LAUNCH_CHECK(c);
        stamp();
        const unsigned pairBlocks = (unsigned)((nTiles * 32 + 127) / 128);
        if (rd.count == 1)
            integ_pairs_kernel<<<pairBlocks, 128, 0, c->stream>>>((int)nTiles, dMeta, one, w.kmin.p, w.kmax.p,
                                                                  w.tileInfo[buf].p, w.pairs[buf].p, nPairs);
        else
            integ_pairs_kernel<<<pairBlocks, 128, 0, c->stream>>>((int)nTiles, dMeta, table, w.kmin.p, w.kmax.p,
                                                                  w.tileInfo[buf].p, w.pairs[buf].p, nPairs);
        LGS_LAUNCH_CHECK(c);
        stamp();
        w.dirty = false;
        const unsigned touchBlocks = (unsigned)std::min<size_t>(pairBound, (size_t)c->sm_count * 4);
        integ_touch_kernel<<<touchBlocks, kTileCells, 0, c->stream>>>(w.rel.p, w.pairs[buf].p, nPairs, w.records[buf].p,
                                                                      w.side[buf].p, nPairs + 1, (unsigned)sideCap,
                                                                      w.counters.p);
        LGS_LAUNCH_CHECK(c);
        stamp();
        // fold on its own stream: it only has to follow this round's touch pass and the previous fold
        LGS_CUDA(c, cudaEventRecord(w.evTouch[buf], c->stream));
        cudaStream_t fs = overlap ? w.foldStream : c->stream;
        if (overlap) LGS_CUDA(c, cudaStreamWaitEvent(fs, w.evTouch[buf], 0));
        FoldArgs a{w.rel.p, w.tileInfo[buf].p, w.pairs[buf].p, w.records[buf].p, w.side[buf].p,
                   diag ? w.counters.p : nullptr, pHit, pMiss, oddsHit, oddsMiss};
        if (rd.count == 1) integ_fold_kernel<<<(unsigned)nTiles, kTileCells, 0, fs>>>(a, one);
        else integ_fold_kernel<<<(unsigned)nTiles, kTileCells, 0, fs>>>(a, table);
        LGS_LAUNCH_CHECK(c);
        LGS_CUDA(c, cudaEventRecord(w.evFold[buf], fs));
        ws.usedBuf[buf] = true;
        lastBuf = buf;
        stamp();
        return LGS_OK;
    };

    // Chunks: each map's scans in order, a chunk grows while it stays within 64 scans and the record budget;
    // chunks without hits are dropped.  Pass p takes chunk p of every map that has one.
    Round rd{0, 0, 0, 0, 0, 0, 0};
    std::vector<int> next(scanBase.begin(), scanBase.end() - 1), inRound(nMaps, -1);
    int nRounds = 0;
    for (bool more = true; more;) {
        more = false;
        for (int i = 0; i < nMaps; ++i) {
            const int end = scanBase[i + 1];
            if (next[i] >= end) continue;
            more = true;
            const lgs_grid* grid = grids[i];
            int x0 = grid->nx, y0 = grid->ny, x1 = -1, y1 = -1, subBeams = 0, subLen = 0, ns = 0;
            size_t pairBound = 0;
            while (next[i] + ns < end && ns < kChunk) {
                const ScanMeta& m = hMeta[next[i] + ns];
                if (m.n > 0) {
                    const int lx = std::max(m.sx - m.maxLen, 0), hx = std::min(m.sx + m.maxLen, grid->nx - 1);
                    const int ly = std::max(m.sy - m.maxLen, 0), hy = std::min(m.sy + m.maxLen, grid->ny - 1);
                    const size_t pb = (size_t)tileSpan(lx, hx) * tileSpan(ly, hy);
                    if (ns > 0 && (pairBound + pb) * kTileCells * sizeof(unsigned) > kRecordBudget) break;
                    pairBound += pb;
                    x0 = std::min(x0, lx); x1 = std::max(x1, hx);
                    y0 = std::min(y0, ly); y1 = std::max(y1, hy);
                    subBeams = std::max(subBeams, m.n);
                    subLen = std::max(subLen, m.maxLen);
                }
                ++ns;
            }
            const int cs = next[i];
            next[i] += ns;
            if (subBeams == 0 || x1 < x0 || y1 < y0) continue;
            x0 &= ~(kTile - 1); y0 &= ~(kTile - 1);                   // tile-aligned region origin
            const int tw = tileSpan(x0, x1), th = tileSpan(y0, y1);
            const size_t nTiles = (size_t)tw * th;
            if (nTiles * kChunk >= ((size_t)1 << 31)) return lgs_fail(c, LGS_ERR_INVALID, "integrate: region of %dx%d tiles is too large", tw, th);
            pairBound = std::min(pairBound, nTiles * ns);
            if (rd.count > 0 && (inRound[i] == nRounds || (rd.pairBound + pairBound) * kTileCells * sizeof(unsigned) > kRecordBudget ||
                                 (rd.tiles + nTiles) * kChunk >= ((size_t)1 << 31) || rd.rows + ns > 65535)) {
                const int rc = launchRound(rd);
                if (rc != LGS_OK) return rc;
                rd = Round{(int)regions.size(), 0, 0, 0, 0, 0, 0};
                ++nRounds;
            }
            regions.push_back(Region{gridRef(grids[i]), x0, y0, tw, (int)rd.tiles, cs, rd.rows});
            ++rd.count;
            rd.rows += ns;
            rd.beams = std::max(rd.beams, subBeams);
            rd.len = std::max(rd.len, subLen);
            rd.tiles += nTiles;
            rd.pairBound += pairBound;
            inRound[i] = nRounds;
        }
    }
    if (rd.count > 0) {
        const int rc = launchRound(rd);
        if (rc != LGS_OK) return rc;
        ++nRounds;
    }
    tLoop = msSince(tStart);
    // The call is complete when its counters are back AND its last fold is done.  The context stream does
    // not wait for that fold: the next call's first chunk starts under it (the record buffers and the
    // fold stream's own order keep the cells right); lgs_grid_integrate_wait is what orders everything
    // else behind the call.
    LGS_CUDA(c, cudaMemcpyAsync(w.hCounters.p, w.counters.p, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    if (overlap && lastBuf >= 0) {
        LGS_CUDA(c, cudaEventRecord(w0.evCounters, c->stream));
        LGS_CUDA(c, cudaStreamWaitEvent(w.foldStream, w0.evCounters, 0));
        LGS_CUDA(c, cudaEventRecord(w0.evDone, w.foldStream));
    } else {
        LGS_CUDA(c, cudaEventRecord(w0.evDone, c->stream));
    }
    w0.pending = true;
    ++ws.calls;
    ++ws.nPending;
    if (perMap)
        for (int i = 0; i < nMaps; ++i) {
            unsigned long long u = 0;
            for (int s = scanBase[i]; s < scanBase[i + 1]; ++s) u += ws.hTouches.p[s];
            perMap[i] = (long long)u;
        }
    if (hostTiming && msSince(tStart) > c->opt.integHostTimingMinMs)
        fprintf(stderr, "[lgs integrate host] %d scans into %d maps, %d rounds: staged %.3f ms, pre-pass synced "
                "%.3f ms, rounds queued %.3f ms\n", n, nMaps, nRounds, tStage, tPre, tLoop);
    if (timing) {
        LGS_CUDA(c, cudaStreamSynchronize(c->stream));
        float t[4] = {0, 0, 0, 0};
        for (size_t k = 0; k + 5 <= evs.size(); k += 5)      // 5 stamps per round
            for (int j = 0; j < 4; ++j) { float ms = 0; cudaEventElapsedTime(&ms, evs[k + j], evs[k + j + 1]); t[j] += ms; }
        fprintf(stderr, "[lgs integrate] %d scans: mark %.3f ms, pairs %.3f ms, touch %.3f ms, fold %.3f ms; computed updates: "
                "max per cell and call %llu, total %llu of %llu touches\n", n, t[0], t[1], t[2], t[3],
                w.hCounters.p[2], w.hCounters.p[3], w.hCounters.p[0]);
        for (cudaEvent_t e : evs) cudaEventDestroy(e);
    }
    return LGS_OK;
}

}  // namespace

extern "C" {

int lgs_grid_integrate_scans(lgs_ctx* c, lgs_grid* grid, const lgs_hit_batch* scans, double pHit,
                             double pMiss, long long* nUpdatesOut) {
    if (!c || !grid || !scans) return LGS_ERR_INVALID;
    if (nUpdatesOut) *nUpdatesOut = 0;
    // calls submitted asynchronously before this one finish first (their counts are dropped)
    while (c->integ && c->integ->nPending > 0) { const int rc = integ_wait(c, nullptr); if (rc != LGS_OK) return rc; }
    const int rc = lgs_grid_integrate_submit(c, grid, scans, pHit, pMiss);
    if (rc != LGS_OK) return rc;
    return integ_wait(c, nUpdatesOut);
}

int lgs_grid_integrate_submit(lgs_ctx* c, lgs_grid* grid, const lgs_hit_batch* scans, double pHit, double pMiss) {
    if (!c || !grid || !scans) return LGS_ERR_INVALID;
    if (scans->n_scans == 0) return LGS_OK;          // nothing in flight: the matching wait reports 0 updates
    const int rc = integ_check(c, 0, grid, scans);
    if (rc != LGS_OK) return rc;
    return integ_submit(c, 1, &grid, scans, pHit, pMiss, nullptr);
}

int lgs_grid_integrate_wait(lgs_ctx* c, long long* nUpdatesOut) {
    if (!c) return LGS_ERR_INVALID;
    return integ_wait(c, nUpdatesOut);
}

int lgs_grid_integrate_many(lgs_ctx* c, int nMaps, lgs_grid* const* grids, const lgs_hit_batch* scans,
                            double pHit, double pMiss, long long* nUpdates) {
    if (!c) return LGS_ERR_INVALID;
    if (nMaps < 0 || (nMaps > 0 && (!grids || !scans)))
        return lgs_fail(c, LGS_ERR_INVALID, "integrate_many: %d maps, grids %p, scans %p", nMaps, (const void*)grids,
                        (const void*)scans);
    if (nUpdates) std::fill(nUpdates, nUpdates + nMaps, 0LL);
    // every argument is checked before anything is staged: a refused call leaves every grid as it was
    int rc = integ_check_many(c, "integrate_many", nMaps, grids, scans);
    if (rc != LGS_OK) return rc;
    rc = integ_submit(c, nMaps, grids, scans, pHit, pMiss, nUpdates);
    if (rc != LGS_OK) return rc;
    return integ_wait(c, nullptr);
}

int lgs_grid_construct_many(lgs_ctx* c, int nMaps, lgs_grid* const* grids, const lgs_scan_batch* scans,
                            const lgs_geometry* cur, double pHit, double pMiss, lgs_geometry* geoOut,
                            double* bboxOut, long long* nUpdates) {
    if (!c) return LGS_ERR_INVALID;
    if (nMaps < 0 || (nMaps > 0 && (!grids || !scans || !cur || !geoOut)))
        return lgs_fail(c, LGS_ERR_INVALID, "construct_many: %d maps, grids %p, scans %p, cur %p, geometry_out %p", nMaps,
                        (const void*)grids, (const void*)scans, (const void*)cur, (const void*)geoOut);
    if (nUpdates) std::fill(nUpdates, nUpdates + nMaps, 0LL);
    // every argument is checked before any grid changes: a refused call leaves every grid as it was
    int rc = integ_check_many(c, "construct_many", nMaps, grids, nullptr);
    if (rc != LGS_OK) return rc;
    std::vector<ConScan> hs;
    std::vector<int> scanBase(nMaps + 1, 0);
    std::vector<long long> beamBase(nMaps + 1, 0);
    for (int i = 0; i < nMaps; ++i) {
        const lgs_scan_batch& b = scans[i];
        if (b.n_scans < 1) return lgs_fail(c, LGS_ERR_INVALID, "construct_many: map %d has no scans", i);
        if (!b.beam_begin || !b.sensor_pose || !b.range_min || !b.range_max)
            return lgs_fail(c, LGS_ERR_INVALID, "construct_many: map %d: beam_begin, sensor_pose, range_min and range_max "
                            "are required", i);
        const lgs_geometry& g = cur[i];
        if (g.patch <= 0 || !(g.res > 0.0) || !std::isfinite(g.res) || !std::isfinite(g.min_x) || !std::isfinite(g.min_y))
            return lgs_fail(c, LGS_ERR_INVALID, "construct_many: bad current geometry of map %d", i);
        for (int s = 0; s < b.n_scans; ++s) {
            const double* p = b.sensor_pose + 3 * s;
            if (b.beam_begin[s + 1] < b.beam_begin[s])
                return lgs_fail(c, LGS_ERR_INVALID, "construct_many: map %d, scan %d: beam_begin decreases", i, s);
            if (!std::isfinite(p[0]) || !std::isfinite(p[1]) || !std::isfinite(p[2]) ||
                !std::isfinite(b.range_min[s]) || !std::isfinite(b.range_max[s]))
                return lgs_fail(c, LGS_ERR_INVALID, "construct_many: map %d, scan %d: non-finite sensor pose or range window", i, s);
            hs.push_back(ConScan{p[0], p[1], p[2], b.range_min[s], b.range_max[s],
                                 (int)(beamBase[i] + b.beam_begin[s] - b.beam_begin[0]), b.beam_begin[s + 1] - b.beam_begin[s], i});
        }
        const long long nb = b.beam_begin[b.n_scans] - b.beam_begin[0];
        if (nb > 0 && (!b.angles || !b.ranges)) return lgs_fail(c, LGS_ERR_INVALID, "construct_many: map %d: angles / ranges NULL", i);
        scanBase[i + 1] = scanBase[i] + b.n_scans;
        beamBase[i + 1] = beamBase[i] + nb;
        if (beamBase[i + 1] > 0x7fffffffLL)
            return lgs_fail(c, LGS_ERR_INVALID, "construct_many: more than 2^31 - 1 beams in one call");
    }
    if (nMaps == 0) return LGS_OK;
    const int n = scanBase[nMaps];
    const long long beams = beamBase[nMaps];
    LGS_CUDA(c, cudaSetDevice(c->device));
    rc = integ_workspace(c);
    if (rc != LGS_OK) return rc;
    lgs_integ_ws& ws = *c->integ;
    lgs_integ_ws::Construct& w = ws.con;
    DevBuf<double>& hit = ws.stage[ws.calls & 1].hit;          // the staging set integ_submit uses next
    cudaStream_t cs = ws.copyStream;                            // integ_submit's pre-pass follows on it

    // Stage: raw beams, the scan table, the bbox seeds (DBL_MAX / DBL_MIN as ConstructMapFromScans starts them,
    // :236-237, and every sensor position), the flags.
    const double kTiny = 2.2250738585072014e-308, kMax = 1.7976931348623157e308;
    std::vector<unsigned long long> keys(4 * (size_t)nMaps);
    auto key = [](double v) { unsigned long long u; memcpy(&u, &v, 8); return conKey(u); };
    for (int i = 0; i < nMaps; ++i) {
        double bx0 = kMax, by0 = kMax, bx1 = kTiny, by1 = kTiny;
        for (int s = scanBase[i]; s < scanBase[i + 1]; ++s) {
            bx0 = std::min(bx0, hs[s].sx); by0 = std::min(by0, hs[s].sy);
            bx1 = std::max(bx1, hs[s].sx); by1 = std::max(by1, hs[s].sy);
        }
        keys[4 * i] = key(bx0); keys[4 * i + 1] = key(by0); keys[4 * i + 2] = key(bx1); keys[4 * i + 3] = key(by1);
    }
    const size_t nbAlloc = std::max<size_t>((size_t)beams, 1);
    LGS_CUDA(c, w.angles.reserve(nbAlloc));
    LGS_CUDA(c, w.ranges.reserve(nbAlloc));
    LGS_CUDA(c, hit.reserve(2 * nbAlloc));
    LGS_CUDA(c, w.hi.reserve(2 * nbAlloc));
    LGS_CUDA(c, w.beam.reserve(nbAlloc));
    LGS_CUDA(c, w.scans.reserve((size_t)n * sizeof(ConScan)));
    LGS_CUDA(c, w.count.reserve((size_t)n));
    LGS_CUDA(c, w.begin.reserve((size_t)n + 1));
    LGS_CUDA(c, w.keys.reserve(4 * (size_t)nMaps));
    LGS_CUDA(c, w.geo.reserve(3 * (size_t)nMaps));
    LGS_CUDA(c, w.flags.reserve(4));
    LGS_CUDA(c, w.hFlags.reserve(4));
    LGS_CUDA(c, w.hCount.reserve((size_t)n));
    if (w.cand.cap == 0) LGS_CUDA(c, w.cand.reserve(4096));
    if (w.edge.cap == 0) LGS_CUDA(c, w.edge.reserve(4096));
    for (int i = 0; i < nMaps; ++i) {
        const lgs_scan_batch& b = scans[i];
        const size_t nb = (size_t)(beamBase[i + 1] - beamBase[i]);
        if (nb == 0) continue;
        LGS_CUDA(c, cudaMemcpyAsync(w.angles.p + beamBase[i], b.angles + b.beam_begin[0], nb * sizeof(double),
                                    cudaMemcpyHostToDevice, cs));
        LGS_CUDA(c, cudaMemcpyAsync(w.ranges.p + beamBase[i], b.ranges + b.beam_begin[0], nb * sizeof(double),
                                    cudaMemcpyHostToDevice, cs));
    }
    LGS_CUDA(c, cudaMemcpyAsync(w.scans.p, hs.data(), (size_t)n * sizeof(ConScan), cudaMemcpyHostToDevice, cs));
    LGS_CUDA(c, cudaMemcpyAsync(w.keys.p, keys.data(), keys.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, cs));
    const int flags0[4] = {0x7fffffff, 0, 0, 0};
    LGS_CUDA(c, cudaMemcpyAsync(w.flags.p, flags0, sizeof(flags0), cudaMemcpyHostToDevice, cs));
    const ConScan* dScans = reinterpret_cast<const ConScan*>(w.scans.p);
    double2* lo = reinterpret_cast<double2*>(hit.p);
    const double2* hi = reinterpret_cast<const double2*>(w.hi.p);

    // Projection, bbox bounds and candidates; the host reads the hit counts and the candidates back.
    con_count_kernel<<<n, kConThreads, 0, cs>>>(dScans, w.angles.p, w.ranges.p, w.count.p, w.flags.p);
    LGS_LAUNCH_CHECK(c);
    con_offsets_kernel<<<1, 1024, 0, cs>>>(w.count.p, n, w.begin.p);
    LGS_LAUNCH_CHECK(c);
    con_project_kernel<<<n, kConThreads, 0, cs>>>(dScans, w.angles.p, w.ranges.p, w.begin.p,
                                                  std::max(c->opt.integResolveUlps, 0.0), lo,
                                                  reinterpret_cast<double2*>(w.hi.p), w.beam.p, w.keys.p);
    LGS_LAUNCH_CHECK(c);
    // A fix-up list comes back with its count; a list longer than its buffer is listed again into a grown one.
    auto fetchList = [&](DevBuf<int2>& list, int which, auto launch) -> int {
        LGS_CUDA(c, cudaMemsetAsync(w.flags.p + which, 0, sizeof(int), cs));
        launch();
        LGS_LAUNCH_CHECK(c);
        LGS_CUDA(c, cudaMemcpyAsync(w.hFlags.p, w.flags.p, 4 * sizeof(int), cudaMemcpyDeviceToHost, cs));
        LGS_CUDA(c, cudaStreamSynchronize(cs));
        const int cnt = w.hFlags.p[which];
        if ((size_t)cnt > list.cap) {
            LGS_CUDA(c, list.reserve((size_t)cnt));
            LGS_CUDA(c, cudaMemsetAsync(w.flags.p + which, 0, sizeof(int), cs));
            launch();
            LGS_LAUNCH_CHECK(c);
        }
        LGS_CUDA(c, w.hList.reserve(std::max(cnt, 1)));
        LGS_CUDA(c, cudaMemcpyAsync(w.hList.p, list.p, (size_t)cnt * sizeof(int2), cudaMemcpyDeviceToHost, cs));
        LGS_CUDA(c, cudaStreamSynchronize(cs));
        return LGS_OK;
    };
    LGS_CUDA(c, cudaMemcpyAsync(w.hCount.p, w.count.p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, cs));
    rc = fetchList(w.cand, kConCand, [&]() {
        con_candidates_kernel<<<n, kConThreads, 0, cs>>>(dScans, w.begin.p, lo, hi, w.beam.p, w.keys.p, w.cand.p,
                                                         (int)std::min<size_t>(w.cand.cap, 0x7fffffff), w.flags.p);
    });
    if (rc != LGS_OK) return rc;
    if (w.hFlags.p[kConBad] != 0x7fffffff) {
        const int s = w.hFlags.p[kConBad];
        const int i = (int)(std::upper_bound(scanBase.begin(), scanBase.end(), s) - scanBase.begin()) - 1;
        return lgs_fail(c, LGS_ERR_INVALID, "construct_many: map %d, scan %d: a beam that passes the range filter has a "
                        "non-finite angle or range", i, s - scanBase[i]);
    }
    const int nCand = w.hFlags.p[kConCand];
    ws.conBboxPoints += nCand;

    // The scan and beam of a call beam, and glibc's hit of it.
    auto hostHit = [&](int callBeam, double* hx, double* hy) {
        const int i = (int)(std::upper_bound(beamBase.begin(), beamBase.end(), (long long)callBeam) - beamBase.begin()) - 1;
        const lgs_scan_batch& b = scans[i];
        const int j = b.beam_begin[0] + (int)(callBeam - beamBase[i]);                 // beam of the batch
        const int s = (int)(std::upper_bound(b.beam_begin, b.beam_begin + b.n_scans + 1, j) - b.beam_begin) - 1;
        lgs_hit_point_host(b.sensor_pose + 3 * s, b.angles[j], b.ranges[j], hx, hy);
    };
    // Exact bbox: the seeds, every sensor position and the candidates' glibc hits, in (scan, beam) order like
    // the reference (no other hit can be an extreme).  Then GridMap::Resize's geometry and the size check.
    std::vector<int2> cands(w.hList.p, w.hList.p + nCand);
    std::vector<int> order(nCand);
    for (int k = 0; k < nCand; ++k) order[k] = k;
    std::sort(order.begin(), order.end(), [&](int a, int b) { return cands[a].x < cands[b].x; });
    std::vector<lgs_geometry> geo(nMaps);
    std::vector<double> bbox(4 * (size_t)nMaps), geoTab(3 * (size_t)nMaps);
    for (int i = 0, k = 0; i < nMaps; ++i) {
        double bx0 = kMax, by0 = kMax, bx1 = kTiny, by1 = kTiny;
        for (int s = scanBase[i]; s < scanBase[i + 1]; ++s) {
            bx0 = std::min(bx0, hs[s].sx); by0 = std::min(by0, hs[s].sy);
            bx1 = std::max(bx1, hs[s].sx); by1 = std::max(by1, hs[s].sy);
            for (; k < nCand && cands[order[k]].x < hs[s].beamBegin + hs[s].n; ++k) {
                double hx, hy;
                hostHit(cands[order[k]].x, &hx, &hy);
                bx0 = std::min(bx0, hx); by0 = std::min(by0, hy);
                bx1 = std::max(bx1, hx); by1 = std::max(by1, hy);
            }
        }
        bbox[4 * i] = bx0; bbox[4 * i + 1] = by0; bbox[4 * i + 2] = bx1; bbox[4 * i + 3] = by1;
        if (lgs_geometry_resize(&cur[i], bx0, by0, bx1, by1, &geo[i], nullptr, nullptr) != LGS_OK)
            return lgs_fail(c, LGS_ERR_INVALID, "construct_many: map %d: no geometry for bbox [%g, %g] x [%g, %g]", i, bx0, bx1, by0, by1);
        const long long a = grids[i]->apron;
        if (((long long)geo[i].nx + 2 * a) * ((long long)geo[i].ny + 2 * a) >= (1LL << 31))
            return lgs_fail(c, LGS_ERR_INVALID, "construct_many: map %d: %dx%d cells are too many", i, geo[i].nx, geo[i].ny);
        geoTab[3 * i] = geo[i].min_x; geoTab[3 * i + 1] = geo[i].min_y; geoTab[3 * i + 2] = geo[i].res;
    }

    // GridMap::Resize + Reset: every grid takes its new geometry with every cell unknown, on its own stream.
    for (int i = 0; i < nMaps; ++i) {
        lgs_grid* g = grids[i];
        g->res = geo[i].res;
        if (g->nx == geo[i].nx && g->ny == geo[i].ny) {
            g->min_x = geo[i].min_x; g->min_y = geo[i].min_y;
            rc = lgs_grid_clear(g);
        } else {
            rc = grid_replace(g, geo[i].nx, geo[i].ny, geo[i].min_x, geo[i].min_y, false, 0, 0);
        }
        if (rc != LGS_OK) {
            const std::string why = g->ctx->err;
            return lgs_fail(c, rc, "construct_many: map %d: %s", i, why.c_str());
        }
        geoOut[i] = geo[i];
        if (bboxOut) std::copy(&bbox[4 * i], &bbox[4 * i + 4], bboxOut + 4 * i);
    }

    // Near-edge hits: glibc's hit replaces the interval end in the staging buffer.
    LGS_CUDA(c, cudaMemcpyAsync(w.geo.p, geoTab.data(), geoTab.size() * sizeof(double), cudaMemcpyHostToDevice, cs));
    rc = fetchList(w.edge, kConEdge, [&]() {
        con_edge_kernel<<<n, kConThreads, 0, cs>>>(dScans, w.begin.p, lo, hi, w.beam.p, w.geo.p, w.edge.p,
                                                   (int)std::min<size_t>(w.edge.cap, 0x7fffffff), w.flags.p);
    });
    if (rc != LGS_OK) return rc;
    const int nEdge = w.hFlags.p[kConEdge];
    ws.conEdgePoints += nEdge;
    std::vector<double> patch(2 * (size_t)std::max(nEdge, 1));
    for (int k = 0; k < nEdge; ++k) hostHit(w.hList.p[k].y, &patch[2 * k], &patch[2 * k + 1]);
    LGS_CUDA(c, w.patch.reserve(patch.size()));
    LGS_CUDA(c, cudaMemcpyAsync(w.patch.p, patch.data(), patch.size() * sizeof(double), cudaMemcpyHostToDevice, cs));
    con_patch_kernel<<<std::max((nEdge + 255) / 256, 1), 256, 0, cs>>>(w.edge.p, reinterpret_cast<const double2*>(w.patch.p),
                                                                      nEdge, lo);
    LGS_LAUNCH_CHECK(c);

    // From here on the integration of lgs_grid_integrate_many, its hits already staged.
    std::vector<double> sensorXY(2 * (size_t)n);
    std::vector<int> hitBegin((size_t)n + nMaps);
    std::vector<lgs_hit_batch> batches(nMaps);
    for (int i = 0; i < nMaps; ++i) {
        int* hb = hitBegin.data() + scanBase[i] + i;
        hb[0] = 0;
        for (int s = scanBase[i]; s < scanBase[i + 1]; ++s) {
            sensorXY[2 * s] = hs[s].sx; sensorXY[2 * s + 1] = hs[s].sy;
            hb[s - scanBase[i] + 1] = hb[s - scanBase[i]] + w.hCount.p[s];
        }
        batches[i] = lgs_hit_batch{scans[i].n_scans, sensorXY.data() + 2 * scanBase[i], hb, nullptr};
    }
    rc = integ_submit(c, nMaps, grids, batches.data(), pHit, pMiss, nUpdates, true);
    if (rc != LGS_OK) return rc;
    return integ_wait(c, nullptr);
}

int lgs_ctx_construct_host_points(const lgs_ctx* c, long long* bboxPoints, long long* edgePoints) {
    if (!c) return LGS_ERR_INVALID;
    if (bboxPoints) *bboxPoints = c->integ ? c->integ->conBboxPoints : 0;
    if (edgePoints) *edgePoints = c->integ ? c->integ->conEdgePoints : 0;
    return LGS_OK;
}

long long lgs_ctx_integrate_fallback_cells(const lgs_ctx* c) { return (c && c->integ) ? c->integ->fallbackCells : 0; }

int lgs_grid_resize(lgs_grid* g, int nx, int ny, double minX, double minY, int shiftX, int shiftY) {
    return g ? grid_replace(g, nx, ny, minX, minY, true, shiftX, shiftY) : LGS_ERR_INVALID;
}

int lgs_grid_clear(lgs_grid* g) {
    if (!g) return LGS_ERR_INVALID;
    lgs_ctx* c = g->ctx;
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, cudaMemsetAsync(g->d, 0, (size_t)g->pitch * g->rows * sizeof(double), c->stream));
    return LGS_OK;
}

}  // extern "C"

namespace {

int grid_replace(lgs_grid* g, int nx, int ny, double minX, double minY, bool copy, int shiftX, int shiftY) {
    lgs_ctx* c = g->ctx;
    if (nx < 0 || ny < 0) return lgs_fail(c, LGS_ERR_INVALID, "grid_resize: %dx%d", nx, ny);
    const long long pitch = (long long)nx + 2LL * g->apron, rows = (long long)ny + 2LL * g->apron;
    if (pitch * rows >= (1LL << 31)) return lgs_fail(c, LGS_ERR_INVALID, "grid_resize: too many cells");
    LGS_CUDA(c, cudaSetDevice(c->device));
    double* nd = nullptr;
    const size_t bytes = (size_t)pitch * rows * sizeof(double);
    // stream-ordered: the new buffer comes from the pool and the old one returns to it after the
    // copy, without synchronising the device (a map that grows every few frames pays microseconds)
    cudaError_t e = lgs_alloc_async(c, &nd, std::max<size_t>(bytes, 8));
    if (e != cudaSuccess) return lgs_fail(c, LGS_ERR_NOMEM, "grid_resize: cudaMallocAsync(%zu) -> %s", bytes, cudaGetErrorString(e));
    LGS_CUDA(c, cudaMemsetAsync(nd, 0, bytes, c->stream));
    if (copy && nx > 0 && ny > 0) {
        dim3 gridDim((nx + 255) / 256, ny);
        grid_shift_copy_kernel<<<gridDim, 256, 0, c->stream>>>(g->origin(), g->nx, g->ny, g->pitch,
                                                               nd + (size_t)g->apron * pitch + g->apron,
                                                               nx, ny, (int)pitch, shiftX, shiftY);
        LGS_LAUNCH_CHECK(c);
    }
    LGS_CUDA(c, cudaFreeAsync(g->d, c->stream));
    g->d = nd; g->nx = nx; g->ny = ny; g->pitch = (int)pitch; g->rows = (int)rows;
    g->min_x = minX; g->min_y = minY;
    return LGS_OK;
}

}  // namespace
