// lgs_precompute.cu -- sliding-window-max maps on sm_100a.
//
// Replaces PrecomputeGridMap / PrecomputeGridMaps / SlidingWindowMaxRow / SlidingWindowMaxCol
// (mapping/grid_map_builder.cpp:403-536) and SlidingWindowMax (util.hpp:199-253).
//
// The reference's deque algorithm emits, for a line of n cells and window w,
//     out[i] = max(in[s .. s+w)),  s = min(i, max(n - w, 0))
// (the last full window is repeated at the tail, util.hpp:250-252; reads past the end of a
// line shorter than w return the unknown value 0.0).  Max is exact, so any evaluation order
// gives bit-identical cells; two passes (y then x, grid_map_builder.cpp:510-512) equal the 2-D
// window maximum.
//
//  * generic window (the correlative matcher's lowRes, e.g. 5): two separable passes, each
//    thread scanning w cached neighbours, lanes along x so every access is coalesced;
//  * pyramid (windows 1, 2, 4, ..., 2^H): level h is built from level h-1 with four reads,
//        out_2w(i) = max(out_w(s), out_w(s + w)),  s = min(i, n - 2w)      when n >= 2w
//        out_2w(i) = max(out_w(0), out_w(n - 1))                            otherwise,
//    applied per axis, so a level costs one read-mostly-from-L2 pass + one write
//    (16 B of HBM traffic per cell per level).
#include "lgs_internal.cuh"

namespace {

// Vertical pass: tmp(x, y) = max_{dy<w} in(x, ys + dy), ys = min(y, max(ny - w, 0)).
__global__ void __launch_bounds__(256)
winmax_y_kernel(const double* __restrict__ in, double* __restrict__ out, int nx, int ny, int pitchIn,
                int pitchOut, int w) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (x >= nx) return;
    const int ys = min(y, max(ny - w, 0));
    const int ye = min(ys + w, ny);   // cells past the last row read as 0.0 <= every value
    double m = 0.0;
    for (int yy = ys; yy < ye; ++yy) m = fmax(m, __ldg(in + (size_t)yy * pitchIn + x));
    out[(size_t)y * pitchOut + x] = m;
}

// Horizontal pass: out(x, y) = max_{dx<w} tmp(xs + dx, y), xs = min(x, max(nx - w, 0)).
__global__ void __launch_bounds__(256)
winmax_x_kernel(const double* __restrict__ in, double* __restrict__ out, int nx, int ny, int pitchIn,
                int pitchOut, int w) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (x >= nx) return;
    const int xs = min(x, max(nx - w, 0));
    const int xe = min(xs + w, nx);
    const double* row = in + (size_t)y * pitchIn;
    double m = 0.0;
    for (int xx = xs; xx < xe; ++xx) m = fmax(m, __ldg(row + xx));
    out[(size_t)y * pitchOut + x] = m;
}

// ---- pyramids: every pass is one launch over all pyramids of a call ----------------------------------
// One entry per pyramid; a launch's flat index (thread of the apron clear, block of the row passes) finds
// its pyramid by the base of its range.
struct PyrBuild {
    const double* src;        // the grid's cell (0, 0)
    double* slab;             // level h's cell (0, 0) is at level0 + h * levelCells
    double* level0;
    size_t levelCells;
    int nx, ny, pitch, rows, apron, xBlocks;
    long long apronBase;      // first apron work item
    long long blockBase;      // first block of the row passes: ny * xBlocks blocks of kPyrCells * 256 cells
};
constexpr int kPyrCells = 4;

template <long long PyrBuild::*Base>
__device__ __forceinline__ const PyrBuild& findBuild(const PyrBuild* __restrict__ builds, int n, long long v) {
    int lo = 0, hi = n - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (builds[mid].*Base <= v) lo = mid; else hi = mid - 1; }
    return builds[lo];
}

// Zero the apron of every level of a pyramid slab (the interior is fully written by the level
// kernels, so clearing the whole slab would double the write traffic of a build).
// Work item r < (H + 1) * per of a slab's apron clear, per = apron cells of one level.
__global__ void __launch_bounds__(256)
zero_apron_kernel(const PyrBuild* __restrict__ builds, int n, long long items) {
    const long long t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t0 >= items) return;
    const PyrBuild& j = findBuild<&PyrBuild::apronBase>(builds, n, t0);
    const long long t = t0 - j.apronBase;
    const int pitch = j.pitch, rows = j.rows, apron = j.apron;
    const long long band = (long long)apron * pitch;                       // full rows at the bottom / top
    const long long side = (long long)(rows - 2 * apron) * (2 * apron);     // left + right columns
    const long long per = 2 * band + side;
    const int lvl = (int)(t / per);
    const long long r = t - (long long)lvl * per;
    size_t cell;
    if (r < band) cell = (size_t)r;
    else if (r < 2 * band) cell = (size_t)(rows - apron) * pitch + (size_t)(r - band);
    else {
        const long long q = r - 2 * band;
        const int row = apron + (int)(q / (2 * apron)), k = (int)(q % (2 * apron));
        cell = (size_t)row * pitch + (k < apron ? k : pitch - 2 * apron + k);
    }
    j.slab[j.levelCells * lvl + cell] = 0.0;
}

// Level 0: window 1 = the grid itself (grid_map_builder.cpp:485-487 with winSize 1).
__global__ void __launch_bounds__(256)
pyr_copy_kernel(const PyrBuild* __restrict__ builds, int n) {
    const PyrBuild& j = findBuild<&PyrBuild::blockBase>(builds, n, blockIdx.x);
    const long long b = (long long)blockIdx.x - j.blockBase;
    const int y = (int)(b / j.xBlocks), xb = (int)(b % j.xBlocks) * (kPyrCells * 256) + threadIdx.x;
    const double* in = j.src + (size_t)y * j.pitch;
    double* o = j.level0 + (size_t)y * j.pitch;
#pragma unroll
    for (int k = 0; k < kPyrCells; ++k)
        if (xb + k * 256 < j.nx) o[xb + k * 256] = __ldg(in + xb + k * 256);
}

// Pyramid doubling step: level h (window 2w) from level h - 1 (window w), both axes at once.  A block
// covers kPyrCells * 256 consecutive cells of one row; thread t owns cells t, t + 256, ... so every load
// and store is coalesced and kPyrCells * 4 independent loads are in flight per thread.  The output level
// is larger than L2 on big maps and is next read by a later launch: streaming stores.
__global__ void __launch_bounds__(256)
winmax_double_kernel(const PyrBuild* __restrict__ builds, int n, int h) {
    const PyrBuild& j = findBuild<&PyrBuild::blockBase>(builds, n, blockIdx.x);
    const long long b = (long long)blockIdx.x - j.blockBase;
    const int y = (int)(b / j.xBlocks), nx = j.nx, ny = j.ny, pitch = j.pitch, w = 1 << (h - 1);
    const double* in = j.level0 + j.levelCells * (h - 1);
    int y0, y1;
    if (ny >= 2 * w) { y0 = min(y, ny - 2 * w); y1 = y0 + w; } else { y0 = 0; y1 = ny - 1; }
    const double* r0 = in + (size_t)y0 * pitch;
    const double* r1 = in + (size_t)y1 * pitch;
    double* o = j.level0 + j.levelCells * h + (size_t)y * pitch;
    const int xb = (int)(b % j.xBlocks) * (kPyrCells * 256) + threadIdx.x;
    double m[kPyrCells];
#pragma unroll
    for (int k = 0; k < kPyrCells; ++k) {
        const int x = min(xb + k * 256, nx - 1);
        int x0, x1;
        if (nx >= 2 * w) { x0 = min(x, nx - 2 * w); x1 = x0 + w; } else { x0 = 0; x1 = nx - 1; }
        m[k] = fmax(fmax(__ldg(r0 + x0), __ldg(r0 + x1)), fmax(__ldg(r1 + x0), __ldg(r1 + x1)));
    }
#pragma unroll
    for (int k = 0; k < kPyrCells; ++k) {
        const int x = xb + k * 256;
        if (x < nx) __stcs(o + x, m[k]);
    }
}

bool same_geometry(const lgs_grid* a, const lgs_grid* b) {
    return a->nx == b->nx && a->ny == b->ny && a->min_x == b->min_x && a->min_y == b->min_y &&
           a->res == b->res && a->off_x == b->off_x && a->off_y == b->off_y;
}

}  // namespace

struct lgs_pyramid {
    lgs_ctx* ctx = nullptr;
    double* slab = nullptr;             // all levels, contiguous
    std::vector<lgs_grid*> levels;      // headers into the slab (owns == false)
    bool foreign = false;               // read by a context other than the owner (another stream)
    const lgs_ctx* lastUser = nullptr;  // the foreign context already ordered after the build
};

void lgs_pyramid_note_user(const lgs_pyramid* p, const lgs_ctx* user) {
    if (!p || user == p->ctx || user == p->lastUser) return;   // the levels never change after the build
    const_cast<lgs_pyramid*>(p)->foreign = true;
    const_cast<lgs_pyramid*>(p)->lastUser = user;
    // the build queued on the owner's stream is ordered before the foreign reader
    lgs_ctx* u = const_cast<lgs_ctx*>(user);
    if (cudaEventRecord(u->evOrder, p->ctx->stream) == cudaSuccess) cudaStreamWaitEvent(u->stream, u->evOrder, 0);
}

const lgs_grid* lgs_pyramid_level(const lgs_pyramid* p, int level) {
    return (p && level >= 0 && level < (int)p->levels.size()) ? p->levels[level] : nullptr;
}

extern "C" {

int lgs_precompute(lgs_ctx* c, const lgs_grid* in, int win, lgs_grid* out) {
    if (!c || !in || !out) return LGS_ERR_INVALID;
    if (win < 1) return lgs_fail(c, LGS_ERR_INVALID, "precompute: window %d", win);
    if (!same_geometry(in, out) || in == out)
        return lgs_fail(c, LGS_ERR_INVALID, "precompute: output must be a distinct grid of equal geometry");
    if (in->nx == 0 || in->ny == 0) return LGS_OK;
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, lgs_grid_acquire(c, in));      // pending integration / resize work of another context
    LGS_CUDA(c, lgs_grid_acquire(c, out));
    LGS_CUDA(c, c->scratch.reserve((size_t)in->nx * in->ny));
    dim3 block(256), gridDim((in->nx + 255) / 256, in->ny);
    winmax_y_kernel<<<gridDim, block, 0, c->stream>>>(in->origin(), c->scratch.p, in->nx, in->ny,
                                                      in->pitch, in->nx, win);
    LGS_LAUNCH_CHECK(c);
    winmax_x_kernel<<<gridDim, block, 0, c->stream>>>(c->scratch.p, out->origin(), in->nx, in->ny,
                                                      in->nx, out->pitch, win);
    LGS_LAUNCH_CHECK(c);
    return LGS_OK;
}

int lgs_pyramid_create(lgs_ctx* c, const lgs_grid* in, int heightMax, lgs_pyramid** outp) {
    if (!c || !in || !outp) return LGS_ERR_INVALID;
    return lgs_pyramid_create_many(c, 1, &in, heightMax, outp);
}

int lgs_pyramid_create_many(lgs_ctx* c, int n, const lgs_grid* const* grids, int heightMax, lgs_pyramid** out) {
    if (!c) return LGS_ERR_INVALID;
    if (n < 0 || (n > 0 && (!grids || !out)))
        return lgs_fail(c, LGS_ERR_INVALID, "pyramid_create_many: %d grids, grids %p, out %p", n, (const void*)grids,
                        (const void*)out);
    std::fill(out, out + n, nullptr);
    if (heightMax < 0 || heightMax > 20) return lgs_fail(c, LGS_ERR_INVALID, "pyramid: height %d", heightMax);
    for (int i = 0; i < n; ++i) {
        if (!grids[i]) return lgs_fail(c, LGS_ERR_INVALID, "pyramid: grid %d is NULL", i);
        if (grids[i]->ctx->device != c->device)
            return lgs_fail(c, LGS_ERR_INVALID, "pyramid: grid %d lives on device %d, the context on %d", i,
                            grids[i]->ctx->device, c->device);
    }
    if (n == 0) return LGS_OK;
    LGS_CUDA(c, cudaSetDevice(c->device));
    for (int i = 0; i < n; ++i) LGS_CUDA(c, lgs_grid_acquire(c, grids[i]));   // pending work of other contexts
    // Every pyramid keeps a slab of its own (lgs_pyramid_destroy frees them one by one): all its levels,
    // each a grid header pointing into it with the input's geometry and zero apron.  Stream-ordered
    // allocation from the device pool (kept warm by lgs_ctx_create's release threshold): a rebuild does not
    // pay a synchronous cudaMalloc of the whole slab.
    std::vector<PyrBuild> builds(n);
    long long items = 0, blocks = 0;
    auto release = [&]() {
        for (int i = 0; i < n; ++i) if (out[i]) { lgs_pyramid_destroy(out[i]); out[i] = nullptr; }
    };
    for (int i = 0; i < n; ++i) {
        const lgs_grid* in = grids[i];
        lgs_pyramid* p = new lgs_pyramid();
        p->ctx = c;
        const size_t levelCells = (size_t)in->pitch * in->rows;
        const size_t bytes = levelCells * (size_t)(heightMax + 1) * sizeof(double);
        const cudaError_t me = lgs_alloc_async(c, &p->slab, std::max<size_t>(bytes, 8));
        if (me != cudaSuccess) {
            delete p;
            release();
            return lgs_fail(c, LGS_ERR_NOMEM, "pyramid: grid %d: cudaMallocAsync(%zu) -> %s", i, bytes,
                            cudaGetErrorString(me));
        }
        for (int h = 0; h <= heightMax; ++h) {
            lgs_grid* g = new lgs_grid(*in);
            g->ctx = c;
            g->d = p->slab + levelCells * h;
            g->owns = false;
            p->levels.push_back(g);
        }
        out[i] = p;
        const int xBlocks = (in->nx + kPyrCells * 256 - 1) / (kPyrCells * 256);
        builds[i] = PyrBuild{in->origin(), p->slab, p->levels[0]->origin(), levelCells, in->nx, in->ny, in->pitch,
                             in->rows, in->apron, xBlocks, items, blocks};
        // the apron of every level, the whole slab when the grid is empty (all of it is apron then)
        if (in->apron > 0)
            items += (2LL * in->apron * in->pitch + (long long)(in->rows - 2 * in->apron) * 2 * in->apron) * (heightMax + 1);
        if (in->nx > 0 && in->ny > 0) blocks += (long long)in->ny * xBlocks;
    }
    if (blocks > 0x7fffffffLL) {
        release();
        return lgs_fail(c, LGS_ERR_INVALID, "pyramid: %lld row blocks in one launch", blocks);
    }
    PyrBuild* dBuilds = nullptr;
    cudaError_t e = lgs_alloc_async(c, &dBuilds, (size_t)n * sizeof(PyrBuild));
    if (e != cudaSuccess) {
        release();
        return lgs_fail(c, LGS_ERR_NOMEM, "pyramid: build table -> %s", cudaGetErrorString(e));
    }
    // pageable source: the copy has taken it when cudaMemcpyAsync returns
    e = cudaMemcpyAsync(dBuilds, builds.data(), (size_t)n * sizeof(PyrBuild), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess && items > 0) {
        zero_apron_kernel<<<(unsigned)((items + 255) / 256), 256, 0, c->stream>>>(dBuilds, n, items);
        c->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess && blocks > 0) {
        pyr_copy_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(dBuilds, n);
        c->launches++;
        e = cudaGetLastError();
        for (int h = 1; e == cudaSuccess && h <= heightMax; ++h) {
            winmax_double_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(dBuilds, n, h);
            c->launches++;
            e = cudaGetLastError();
        }
    }
    cudaFreeAsync(dBuilds, c->stream);
    if (e != cudaSuccess) {
        release();
        return lgs_fail(c, LGS_ERR_CUDA, "pyramid: %s", cudaGetErrorString(e));
    }
    return LGS_OK;
}

int lgs_pyramid_destroy(lgs_pyramid* p) {
    if (!p) return LGS_OK;
    cudaSetDevice(p->ctx->device);
    for (lgs_grid* g : p->levels) delete g;
    if (p->foreign) cudaDeviceSynchronize();               // another context's stream may still read it
    if (p->slab) cudaFreeAsync(p->slab, p->ctx->stream);   // ordered after every use on the context stream
    delete p;
    return LGS_OK;
}

int lgs_pyramid_levels(const lgs_pyramid* p) { return p ? (int)p->levels.size() : 0; }

int lgs_pyramid_download(const lgs_pyramid* p, int level, double* dense) {
    if (!p || level < 0 || level >= (int)p->levels.size()) return LGS_ERR_INVALID;
    return lgs_grid_download(p->levels[level], dense);
}

}  // extern "C"
