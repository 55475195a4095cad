// lgs_core.cu -- context and dense device grid of the sm_100a backend.
//
// The device grid replaces GridMap<T>'s patch-tiled storage (grid_map/grid_map.hpp:22-318,
// grid_map_patch.hpp:15-75) on the hot path.  Reads of unallocated patches and of cells
// outside the map both return the unknown value 0.0 through Value(x, y, unknown)
// (grid_map.hpp:859-873), so a dense row-major array whose unknown cells hold 0.0 and which
// is surrounded by a zero apron is value-equivalent for every reader on the path.
#include <cstddef>

#include "lgs_internal.cuh"

cudaError_t lgs_grid_acquire(lgs_ctx* user, const lgs_grid* g) {
    if (!g || g->ctx == user) return cudaSuccess;
    g->foreign = true;
    cudaError_t e = cudaEventRecord(user->evOrder, g->ctx->stream);
    if (e != cudaSuccess) return e;
    return cudaStreamWaitEvent(user->stream, user->evOrder, 0);
}

int lgs_fail(lgs_ctx* ctx, int code, const char* fmt, ...) {
    if (ctx) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(ctx->err, sizeof(ctx->err), fmt, ap);
        va_end(ap);
    }
    return code;
}

namespace {

struct OptField { const char* name; const char* env; int kind; size_t off; };   // kind 0 int, 1 double, 2 long long
#define LGS_OPT(name, env, kind, field) {name, env, kind, offsetof(lgs_opts, field)}
const OptField kOptFields[] = {
    LGS_OPT("edge_eps", nullptr, 1, edgeEps),
    LGS_OPT("csm_flat", "LGS_CSM_FLAT", 0, csmFlat),
    LGS_OPT("bb_sync", "LGS_BB_SYNC", 0, bbSync),
    LGS_OPT("bb_table", "LGS_BB_TABLE", 0, bbTable),
    LGS_OPT("bb_warp_below", "LGS_BB_WARP_BELOW", 0, bbWarpBelow),
    LGS_OPT("bb_resolve_ulps", "LGS_BB_RESOLVE_ULPS", 0, bbResolveUlps),
    LGS_OPT("bb_blocks_per_sm", "LGS_BB_BLOCKS_PER_SM", 0, bbBlocksPerSm),
    LGS_OPT("bb_cost_g1", nullptr, 1, bbCost[0]),
    LGS_OPT("bb_cost_g4", nullptr, 1, bbCost[1]),
    LGS_OPT("bb_cost_g8", nullptr, 1, bbCost[2]),
    LGS_OPT("bb_cost_g32", nullptr, 1, bbCost[3]),
    LGS_OPT("bb_host_timing", "LGS_BB_HOSTTIMING", 0, bbHostTiming),
    LGS_OPT("bb_count_nodes", nullptr, 0, bbCountNodes),
    LGS_OPT("bb_early_reject", "LGS_BB_EARLY_REJECT", 0, bbEarlyReject),
    LGS_OPT("integ_host_timing", "LGS_INTEG_HOSTTIMING", 0, integHostTiming),
    LGS_OPT("integ_host_timing_min_ms", "LGS_INTEG_HOSTTIMING_MIN_MS", 1, integHostTimingMinMs),
    LGS_OPT("integ_timing", "LGS_INTEG_TIMING", 0, integTiming),
    LGS_OPT("integ_diag", "LGS_INTEG_DIAG", 0, integDiag),
    LGS_OPT("integ_side_words", "LGS_INTEG_SIDE_WORDS", 2, integSideWords),
    LGS_OPT("integ_resolve_ulps", nullptr, 1, integResolveUlps),
    LGS_OPT("gs_tables", "LGS_GS_TABLES", 0, gsTables),
};
#undef LGS_OPT

void opt_store(lgs_opts* o, const OptField& f, double v) {
    char* base = reinterpret_cast<char*>(o) + f.off;
    if (f.kind == 0) *reinterpret_cast<int*>(base) = (int)v;
    else if (f.kind == 1) *reinterpret_cast<double*>(base) = v;
    else *reinterpret_cast<long long*>(base) = (long long)v;
}

double opt_load(const lgs_opts* o, const OptField& f) {
    const char* base = reinterpret_cast<const char*>(o) + f.off;
    if (f.kind == 0) return *reinterpret_cast<const int*>(base);
    if (f.kind == 1) return *reinterpret_cast<const double*>(base);
    return (double)*reinterpret_cast<const long long*>(base);
}

// The one place the environment is read: defaults of a NEW context.
void opts_from_env(lgs_opts* o) {
    for (const OptField& f : kOptFields) {
        if (!f.env) continue;
        const char* e = getenv(f.env);
        if (!e) continue;
        char* end = nullptr;
        const double v = strtod(e, &end);
        opt_store(o, f, end != e ? v : 1.0);      // "LGS_X=" or a non-number means "on"
    }
}

}  // namespace

extern "C" {

int lgs_ctx_set_option(lgs_ctx* c, const char* name, double value) {
    if (!c || !name) return LGS_ERR_INVALID;
    for (const OptField& f : kOptFields)
        if (strcmp(f.name, name) == 0) {
            if (strcmp(name, "edge_eps") == 0 && !(value > 0.0 && value < 0.5)) value = LGS_EDGE_EPS_DEFAULT;
            opt_store(&c->opt, f, value);
            if (strncmp(name, "bb_", 3) == 0) c->bbBlocks = 0;   // re-size the persistent grid
            return LGS_OK;
        }
    return lgs_fail(c, LGS_ERR_INVALID, "ctx_set_option: unknown option '%s'", name);
}

int lgs_ctx_get_option(const lgs_ctx* c, const char* name, double* value) {
    if (!c || !name || !value) return LGS_ERR_INVALID;
    for (const OptField& f : kOptFields)
        if (strcmp(f.name, name) == 0) { *value = opt_load(&c->opt, f); return LGS_OK; }
    return LGS_ERR_INVALID;
}

const char* lgs_version(void) { return "lgs_b200 0.1 (sm_100a)"; }

int lgs_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int lgs_ctx_create(int device, lgs_ctx** out) {
    if (!out) return LGS_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n)
        return LGS_ERR_CUDA;   // no CPU fallback: the caller must fail loudly
    lgs_ctx* c = new lgs_ctx();
    opts_from_env(&c->opt);
    c->device = device;
    cudaDeviceProp prop;
    if (cudaSetDevice(device) != cudaSuccess ||
        cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete c; return LGS_ERR_CUDA; }
    if (prop.major < 10) { delete c; return LGS_ERR_CUDA; }   // sm_100a code only
    c->sm_count = prop.multiProcessorCount;
    {   // A PRIVATE pool that keeps freed stream-ordered allocations (pyramid slabs, grids): the device's
        // default pool is process-global, so raising ITS release threshold would change the memory
        // behaviour of every other user of the process (e.g. PyTorch's async allocations).
        cudaMemPoolProps props{};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        if (cudaMemPoolCreate(&c->pool, &props) != cudaSuccess) { delete c; return LGS_ERR_CUDA; }
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(c->pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->evOrder, cudaEventDisableTiming) != cudaSuccess) {
        if (c->stream) cudaStreamDestroy(c->stream);
        if (c->ev0) cudaEventDestroy(c->ev0);
        if (c->ev1) cudaEventDestroy(c->ev1);
        cudaMemPoolDestroy(c->pool);
        delete c;
        return LGS_ERR_CUDA;
    }
    *out = c;
    return LGS_OK;
}

int lgs_ctx_destroy(lgs_ctx* c) {
    if (!c) return LGS_OK;
    cudaSetDevice(c->device);
    if (c->stream) { cudaStreamSynchronize(c->stream); cudaStreamDestroy(c->stream); }
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->evOrder) cudaEventDestroy(c->evOrder);
    c->scratch.release();
    if (c->integ) { c->integ->release(); delete c->integ; }
    lgs_cost_ws_destroy(c->cost);
    if (c->pool) cudaMemPoolDestroy(c->pool);   // grids / pyramids still alive keep their memory until freed
    delete c;
    return LGS_OK;
}

const char* lgs_ctx_last_error(const lgs_ctx* c) { return c ? c->err : "null context"; }

int lgs_ctx_synchronize(lgs_ctx* c) {
    if (!c) return LGS_ERR_INVALID;
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, cudaStreamSynchronize(c->stream));
    return LGS_OK;
}

int lgs_ctx_wait_ctx(lgs_ctx* c, lgs_ctx* other) {
    if (!c || !other) return LGS_ERR_INVALID;
    if (c == other) return LGS_OK;
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, cudaEventRecord(c->evOrder, other->stream));
    LGS_CUDA(c, cudaStreamWaitEvent(c->stream, c->evOrder, 0));
    return LGS_OK;
}

int lgs_host_pin(lgs_ctx* c, void* ptr, unsigned long long bytes) {
    if (!c || !ptr || bytes == 0) return LGS_ERR_INVALID;
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterDefault));
    return LGS_OK;
}

int lgs_host_unpin(lgs_ctx* c, void* ptr) {
    if (!c || !ptr) return LGS_ERR_INVALID;
    LGS_CUDA(c, cudaHostUnregister(ptr));
    return LGS_OK;
}

int lgs_device_alloc(lgs_ctx* c, unsigned long long bytes, void** out) {
    if (!c || !out || bytes == 0) return LGS_ERR_INVALID;
    *out = nullptr;
    LGS_CUDA(c, cudaSetDevice(c->device));
    cudaError_t e = cudaMalloc(out, (size_t)bytes);
    if (e != cudaSuccess) return lgs_fail(c, LGS_ERR_NOMEM, "device_alloc(%llu) -> %s", bytes, cudaGetErrorString(e));
    LGS_CUDA(c, cudaMemsetAsync(*out, 0, (size_t)bytes, c->stream));
    return LGS_OK;
}

int lgs_device_free(lgs_ctx* c, void* ptr) {
    if (!c) return LGS_ERR_INVALID;
    if (!ptr) return LGS_OK;
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, cudaStreamSynchronize(c->stream));
    LGS_CUDA(c, cudaFree(ptr));
    return LGS_OK;
}

int lgs_device_download(lgs_ctx* c, const void* devicePtr, void* host, unsigned long long bytes) {
    if (!c || (bytes > 0 && (!devicePtr || !host))) return LGS_ERR_INVALID;
    if (bytes == 0) return LGS_OK;
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, cudaMemcpyAsync(host, devicePtr, (size_t)bytes, cudaMemcpyDeviceToHost, c->stream));
    LGS_CUDA(c, cudaStreamSynchronize(c->stream));
    return LGS_OK;
}

void* lgs_ctx_stream(lgs_ctx* c) { return c ? (void*)c->stream : nullptr; }

int lgs_ctx_timer_start(lgs_ctx* c) {
    if (!c) return LGS_ERR_INVALID;
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, cudaEventRecord(c->ev0, c->stream));
    return LGS_OK;
}

int lgs_ctx_timer_stop(lgs_ctx* c, float* ms) {
    if (!c || !ms) return LGS_ERR_INVALID;
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, cudaEventRecord(c->ev1, c->stream));
    LGS_CUDA(c, cudaEventSynchronize(c->ev1));
    LGS_CUDA(c, cudaEventElapsedTime(ms, c->ev0, c->ev1));
    return LGS_OK;
}

long long lgs_ctx_launch_count(const lgs_ctx* c) { return c ? c->launches : 0; }

int lgs_grid_create(lgs_ctx* c, int nx, int ny, double min_x, double min_y, double res,
                    int apron, lgs_grid** out) {
    if (!c || !out) return LGS_ERR_INVALID;
    *out = nullptr;
    if (nx < 0 || ny < 0 || apron < 1 || !(res > 0.0))
        return lgs_fail(c, LGS_ERR_INVALID, "grid_create: nx=%d ny=%d apron=%d res=%g", nx, ny,
                        apron, res);
    const long long pitch = (long long)nx + 2LL * apron, rows = (long long)ny + 2LL * apron;
    if (pitch * rows >= (1LL << 31))
        return lgs_fail(c, LGS_ERR_INVALID, "grid_create: %lld cells exceed int32 indexing",
                        pitch * rows);
    LGS_CUDA(c, cudaSetDevice(c->device));
    lgs_grid* g = new lgs_grid();
    g->ctx = c; g->nx = nx; g->ny = ny; g->apron = apron;
    g->pitch = (int)pitch; g->rows = (int)rows;
    g->min_x = min_x; g->min_y = min_y; g->res = res;
    const size_t bytes = (size_t)pitch * rows * sizeof(double);
    // stream-ordered pool allocation: lgs_grid_resize can then swap buffers without a device sync
    cudaError_t e = lgs_alloc_async(c, &g->d, std::max<size_t>(bytes, 8));
    if (e != cudaSuccess) {
        delete g;
        return lgs_fail(c, LGS_ERR_NOMEM, "grid_create: cudaMallocAsync(%zu) -> %s", bytes,
                        cudaGetErrorString(e));
    }
    e = cudaMemsetAsync(g->d, 0, bytes, c->stream);
    if (e != cudaSuccess) {
        cudaFree(g->d); delete g;
        return lgs_fail(c, LGS_ERR_CUDA, "grid_create: memset -> %s", cudaGetErrorString(e));
    }
    *out = g;
    return LGS_OK;
}

int lgs_grid_destroy(lgs_grid* g) {
    if (!g) return LGS_OK;
    cudaSetDevice(g->ctx->device);
    if (g->d && g->owns) {
        if (g->foreign) cudaDeviceSynchronize();   // another context's stream may still read it
        cudaFreeAsync(g->d, g->ctx->stream);        // ordered after every use on the owner's stream
    }
    delete g;
    return LGS_OK;
}

int lgs_grid_upload(lgs_grid* g, const double* dense) {
    if (!g || !dense) return LGS_ERR_INVALID;
    lgs_ctx* c = g->ctx;
    if (g->nx == 0 || g->ny == 0) return LGS_OK;
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, cudaMemcpy2DAsync(g->origin(), (size_t)g->pitch * sizeof(double), dense,
                                  (size_t)g->nx * sizeof(double), (size_t)g->nx * sizeof(double),
                                  g->ny, cudaMemcpyHostToDevice, c->stream));
    LGS_CUDA(c, cudaStreamSynchronize(c->stream));
    return LGS_OK;
}

int lgs_grid_download(const lgs_grid* g, double* dense) {
    if (!g || !dense) return LGS_ERR_INVALID;
    lgs_ctx* c = g->ctx;
    if (g->nx == 0 || g->ny == 0) return LGS_OK;
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, cudaMemcpy2DAsync(dense, (size_t)g->nx * sizeof(double), g->origin(),
                                  (size_t)g->pitch * sizeof(double),
                                  (size_t)g->nx * sizeof(double), g->ny, cudaMemcpyDeviceToHost,
                                  c->stream));
    LGS_CUDA(c, cudaStreamSynchronize(c->stream));
    return LGS_OK;
}

int lgs_grid_download_region(const lgs_grid* g, int x0, int y0, int w, int h, double* dst, long long dstPitch) {
    if (!g || !dst) return LGS_ERR_INVALID;
    lgs_ctx* c = g->ctx;
    if (w == 0 || h == 0) return LGS_OK;
    if (x0 < 0 || y0 < 0 || w < 0 || h < 0 || x0 + (long long)w > g->nx || y0 + (long long)h > g->ny || dstPitch < w)
        return lgs_fail(c, LGS_ERR_INVALID, "grid_download_region: [%d, %d) x [%d, %d) of a %dx%d grid, pitch %lld",
                        x0, x0 + w, y0, y0 + h, g->nx, g->ny, dstPitch);
    LGS_CUDA(c, cudaSetDevice(c->device));
    LGS_CUDA(c, cudaMemcpy2DAsync(dst, (size_t)dstPitch * sizeof(double), g->origin() + (size_t)y0 * g->pitch + x0,
                                  (size_t)g->pitch * sizeof(double), (size_t)w * sizeof(double), h,
                                  cudaMemcpyDeviceToHost, c->stream));
    LGS_CUDA(c, cudaStreamSynchronize(c->stream));
    return LGS_OK;
}

int lgs_grid_copy(const lgs_grid* src, lgs_grid* dst) {
    if (!src || !dst || src == dst) return LGS_ERR_INVALID;
    lgs_ctx* c = dst->ctx;
    if (src->ctx->device != c->device)
        return lgs_fail(c, LGS_ERR_INVALID, "grid_copy: grids live on devices %d and %d", src->ctx->device, c->device);
    if (src->res != dst->res)
        return lgs_fail(c, LGS_ERR_INVALID, "grid_copy: resolutions %g and %g differ", src->res, dst->res);
    LGS_CUDA(c, cudaSetDevice(c->device));
    if (dst->nx != src->nx || dst->ny != src->ny) {
        // new placement, everything unknown (shifts beyond any map size)
        const int rc = lgs_grid_resize(dst, src->nx, src->ny, src->min_x, src->min_y, 1 << 30, 1 << 30);
        if (rc != LGS_OK) return rc;
    }
    dst->min_x = src->min_x; dst->min_y = src->min_y;
    dst->off_x = src->off_x; dst->off_y = src->off_y;
    // everything queued on the source's stream (its last integration) is ordered before the copy
    LGS_CUDA(c, lgs_grid_acquire(c, src));
    if (src->nx > 0 && src->ny > 0)
        LGS_CUDA(c, cudaMemcpy2DAsync(dst->origin(), (size_t)dst->pitch * sizeof(double), src->origin(),
                                      (size_t)src->pitch * sizeof(double), (size_t)src->nx * sizeof(double),
                                      src->ny, cudaMemcpyDeviceToDevice, c->stream));
    return LGS_OK;
}

int lgs_grid_set_window(lgs_grid* g, int off_x, int off_y) {
    if (!g) return LGS_ERR_INVALID;
    if (off_x < 0 || off_y < 0) return lgs_fail(g->ctx, LGS_ERR_INVALID, "grid_set_window: negative offset");
    g->off_x = off_x; g->off_y = off_y;
    return LGS_OK;
}

int lgs_grid_info(const lgs_grid* g, int* nx, int* ny, double* min_x, double* min_y, double* res,
                  int* apron) {
    if (!g) return LGS_ERR_INVALID;
    if (nx) *nx = g->nx;
    if (ny) *ny = g->ny;
    if (min_x) *min_x = g->min_x;
    if (min_y) *min_y = g->min_y;
    if (res) *res = g->res;
    if (apron) *apron = g->apron;
    return LGS_OK;
}

}  // extern "C"
