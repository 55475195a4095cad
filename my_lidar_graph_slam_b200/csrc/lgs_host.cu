// lgs_host.cu -- host-side helpers of the C ABI (no device code).
//
// These restate, with the CPU's own arithmetic (glibc sin/cos, no FMA contraction), the small
// pieces of reference logic a caller needs around the device kernels when it does not link the
// reference itself: the range filter + HitPoint of one scan (grid_map_builder.cpp:335-380,
// sensor_data.hpp:162-173) and the patch-aligned map geometry of GridMap::Resize / Expand
// (grid_map/grid_map.hpp:652-736, :907-916).  The C++ adapters use the reference's own
// GridMap / ScanData for the same purpose; tests check both against the oracle.
#include <cmath>

#include "lgs_internal.cuh"

namespace {

// GridMap::GridCellIndexToPatchIndex (grid_map.hpp:907-916): note idx/size - 1 for idx < 0.
inline int cellToPatch(int idx, int patch) { return idx < 0 ? idx / patch - 1 : idx / patch; }

inline int worldToCell(double p, double minP, double res) {
    return static_cast<int>(std::floor((p - minP) / res));   // grid_map.hpp:779-790
}

}  // namespace

void lgs_hit_point_host(const double* sensorPose, double angle, double r, double* hx, double* hy) {
    const double cosT = std::cos(sensorPose[2] + angle);              // sensor_data.hpp:168-169
    const double sinT = std::sin(sensorPose[2] + angle);
    *hx = sensorPose[0] + r * cosT;
    *hy = sensorPose[1] + r * sinT;
}

extern "C" {

int lgs_scan_hit_points(const double* sensorPose, int n, const double* angles, const double* ranges,
                        double rangeMin, double rangeMax, double* hitXY, int* nHit, double* bbox) {
    if (!sensorPose || n < 0 || (n > 0 && (!angles || !ranges)) || !hitXY || !nHit) return LGS_ERR_INVALID;
    double minX = sensorPose[0], minY = sensorPose[1], maxX = sensorPose[0], maxY = sensorPose[1];
    int k = 0;
    for (int i = 0; i < n; ++i) {
        const double r = ranges[i];
        if (r >= rangeMax || r <= rangeMin) continue;                 // grid_map_builder.cpp:365-366
        double hx, hy;
        lgs_hit_point_host(sensorPose, angles[i], r, &hx, &hy);
        hitXY[2 * k] = hx; hitXY[2 * k + 1] = hy; ++k;
        minX = std::min(minX, hx); minY = std::min(minY, hy);         // :373-377
        maxX = std::max(maxX, hx); maxY = std::max(maxY, hy);
    }
    *nHit = k;
    if (bbox) { bbox[0] = minX; bbox[1] = minY; bbox[2] = maxX; bbox[3] = maxY; }
    return LGS_OK;
}

int lgs_geometry_resize(const lgs_geometry* cur, double minX, double minY, double maxX, double maxY,
                        lgs_geometry* out, int* shiftX, int* shiftY) {
    if (!cur || !out || cur->patch <= 0 || !(cur->res > 0.0) || !(minX <= maxX) || !(minY <= maxY))
        return LGS_ERR_INVALID;
    const int p = cur->patch;
    const int cx0 = worldToCell(minX, cur->min_x, cur->res), cy0 = worldToCell(minY, cur->min_y, cur->res);
    const int cx1 = worldToCell(maxX, cur->min_x, cur->res), cy1 = worldToCell(maxY, cur->min_y, cur->res);
    const int px0 = cellToPatch(cx0, p), py0 = cellToPatch(cy0, p);
    const int px1 = cellToPatch(cx1, p), py1 = cellToPatch(cy1, p);
    const int npx = std::max(0, px1 - px0 + 1), npy = std::max(0, py1 - py0 + 1);      // :670-672
    *out = *cur;
    out->nx = npx * p; out->ny = npy * p;
    out->min_x = cur->min_x + (px0 * p) * cur->res;                                      // :707-710
    out->min_y = cur->min_y + (py0 * p) * cur->res;
    if (shiftX) *shiftX = px0 * p;
    if (shiftY) *shiftY = py0 * p;
    return LGS_OK;
}

int lgs_geometry_expand(const lgs_geometry* cur, double minX, double minY, double maxX, double maxY,
                        double enlargeStep, lgs_geometry* out, int* shiftX, int* shiftY, int* changed) {
    if (!cur || !out) return LGS_ERR_INVALID;
    auto inside = [&](double x, double y) {
        const int ix = worldToCell(x, cur->min_x, cur->res), iy = worldToCell(y, cur->min_y, cur->res);
        return ix >= 0 && ix < cur->nx && iy >= 0 && iy < cur->ny;
    };
    if (inside(minX, minY) && inside(maxX, maxY)) {                                      // :723-724
        *out = *cur;
        if (shiftX) *shiftX = 0;
        if (shiftY) *shiftY = 0;
        if (changed) *changed = 0;
        return LGS_OK;
    }
    double loX = cur->min_x + cur->res * 0, loY = cur->min_y + cur->res * 0;             // :726
    double hiX = cur->min_x + cur->res * cur->nx, hiY = cur->min_y + cur->res * cur->ny; // :727-728
    loX = (minX < loX) ? minX - enlargeStep : loX;                                       // :730-733
    loY = (minY < loY) ? minY - enlargeStep : loY;
    hiX = (maxX > hiX) ? maxX + enlargeStep : hiX;
    hiY = (maxY > hiY) ? maxY + enlargeStep : hiY;
    if (changed) *changed = 1;
    return lgs_geometry_resize(cur, loX, loY, hiX, hiY, out, shiftX, shiftY);
}

}  // extern "C"
