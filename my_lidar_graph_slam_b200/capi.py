"""ctypes binding to liblgs_b200.so, the C-ABI of the sm_100a backend (include/lgs_b200.h).

This is plumbing for tests and bench.py: every compute call goes through the C ABI exactly
as the C++ adapters (adapters/) do.  There is NO fallback: if the shared library is missing
or no B200-class GPU is usable, the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblgs_b200.so")

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int)
vp = C.c_void_p

ERRORS = {1: "LGS_ERR_INVALID", 2: "LGS_ERR_CUDA", 3: "LGS_ERR_NOMEM", 4: "LGS_ERR_APRON",
          5: "LGS_ERR_OVERFLOW"}


class LgsError(RuntimeError):
    pass


class ScanBatch(C.Structure):
    _fields_ = [("n_scans", C.c_int), ("beam_begin", c_ip), ("angles", c_dp), ("ranges", c_dp),
                ("sensor_pose", c_dp), ("range_min", c_dp), ("range_max", c_dp)]


class MatchResult(C.Structure):
    _fields_ = [("found", C.c_int), ("ix", C.c_int), ("iy", C.c_int), ("it", C.c_int),
                ("win_x", C.c_int), ("win_y", C.c_int), ("win_t", C.c_int),
                ("n_fixups", C.c_int), ("step_x", C.c_double), ("step_y", C.c_double),
                ("step_t", C.c_double), ("score", C.c_double), ("n_scored", C.c_longlong),
                ("exact_replay", C.c_int), ("reserved", C.c_int)]


MATCH_DTYPE = np.dtype([("found", np.int32), ("ix", np.int32), ("iy", np.int32), ("it", np.int32),
                        ("win_x", np.int32), ("win_y", np.int32), ("win_t", np.int32), ("n_fixups", np.int32),
                        ("step_x", np.float64), ("step_y", np.float64), ("step_t", np.float64),
                        ("score", np.float64), ("n_scored", np.int64), ("exact_replay", np.int32),
                        ("reserved", np.int32)])
assert MATCH_DTYPE.itemsize == C.sizeof(MatchResult)


class LoopRecord(C.Structure):
    _fields_ = [("found", C.c_int), ("ix", C.c_int), ("iy", C.c_int), ("it", C.c_int),
                ("score", C.c_double), ("id", C.c_longlong)]


# the 32-byte exchange record of loop detection (lgs_loop_record); "submap" = the caller's pair id
RECORD_DTYPE = np.dtype([("found", np.int32), ("ix", np.int32), ("iy", np.int32), ("it", np.int32),
                         ("score", np.float64), ("submap", np.int64)])
assert RECORD_DTYPE.itemsize == C.sizeof(LoopRecord) == 32


class BbParams(C.Structure):
    _fields_ = [("node_height_max", C.c_int), ("range_x", C.c_double), ("range_y", C.c_double),
                ("range_theta", C.c_double), ("scan_range_max", C.c_double),
                ("score_range_min", C.c_double), ("score_range_max", C.c_double)]


class RtcsmParams(C.Structure):
    _fields_ = [("low_res", C.c_int), ("range_x", C.c_double), ("range_y", C.c_double),
                ("range_theta", C.c_double), ("scan_range_max", C.c_double)]


# name -> (restype, argtypes); also the list tests use to check the exported symbols.
SIGNATURES = {
    "lgs_version": (C.c_char_p, []),
    "lgs_host_pin": (C.c_int, [vp, vp, C.c_ulonglong]),
    "lgs_host_unpin": (C.c_int, [vp, vp]),
    "lgs_measure_gather_peak": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.POINTER(C.c_double)]),
    "lgs_device_alloc": (C.c_int, [vp, C.c_ulonglong, C.POINTER(vp)]),
    "lgs_device_free": (C.c_int, [vp, vp]),
    "lgs_device_download": (C.c_int, [vp, vp, vp, C.c_ulonglong]),
    "lgs_ctx_set_option": (C.c_int, [vp, C.c_char_p, C.c_double]),
    "lgs_ctx_get_option": (C.c_int, [vp, C.c_char_p, C.POINTER(C.c_double)]),
    "lgs_device_count": (C.c_int, []),
    "lgs_ctx_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
    "lgs_ctx_destroy": (C.c_int, [vp]),
    "lgs_ctx_last_error": (C.c_char_p, [vp]),
    "lgs_ctx_synchronize": (C.c_int, [vp]),
    "lgs_ctx_wait_ctx": (C.c_int, [vp, vp]),
    "lgs_ctx_stream": (vp, [vp]),
    "lgs_ctx_timer_start": (C.c_int, [vp]),
    "lgs_ctx_timer_stop": (C.c_int, [vp, C.POINTER(C.c_float)]),
    "lgs_ctx_launch_count": (C.c_longlong, [vp]),
    "lgs_grid_create": (C.c_int, [vp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double,
                                  C.c_int, C.POINTER(vp)]),
    "lgs_grid_destroy": (C.c_int, [vp]),
    "lgs_grid_upload": (C.c_int, [vp, c_dp]),
    "lgs_grid_download": (C.c_int, [vp, c_dp]),
    "lgs_grid_set_window": (C.c_int, [vp, C.c_int, C.c_int]),
    "lgs_grid_info": (C.c_int, [vp, c_ip, c_ip, c_dp, c_dp, c_dp, c_ip]),
    "lgs_precompute": (C.c_int, [vp, vp, C.c_int, vp]),
    "lgs_pyramid_create": (C.c_int, [vp, vp, C.c_int, C.POINTER(vp)]),
    "lgs_pyramid_destroy": (C.c_int, [vp]),
    "lgs_pyramid_download": (C.c_int, [vp, C.c_int, c_dp]),
    "lgs_pyramid_levels": (C.c_int, [vp]),
    "lgs_rtcsm_batch_create": (C.c_int, [vp, C.POINTER(RtcsmParams), C.POINTER(vp)]),
    "lgs_rtcsm_batch_destroy": (C.c_int, [vp]),
    "lgs_rtcsm_batch_upload": (C.c_int, [vp, vp, C.POINTER(ScanBatch), c_dp]),
    "lgs_rtcsm_batch_run": (C.c_int, [vp, vp, vp]),
    "lgs_rtcsm_batch_run_timed": (C.c_int, [vp, vp, vp, C.POINTER(C.c_float)]),
    "lgs_rtcsm_batch_results": (C.c_int, [vp, vp, vp, C.POINTER(MatchResult)]),
    "lgs_rtcsm_batch_debug": (C.c_int, [vp, C.c_int, c_ip, c_dp, c_dp, c_ip]),
    "lgs_rtcsm_batch_work": (C.c_int, [vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
    "lgs_rtcsm_batch_fine_tiles": (C.c_int, [vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
    "lgs_rtcsm_match": (C.c_int, [vp, vp, vp, C.POINTER(RtcsmParams), C.POINTER(ScanBatch), c_dp,
                                  C.POINTER(MatchResult)]),
    "lgs_bb_batch_create": (C.c_int, [vp, C.POINTER(BbParams), C.POINTER(vp)]),
    "lgs_bb_batch_destroy": (C.c_int, [vp]),
    "lgs_bb_batch_upload": (C.c_int, [vp, C.POINTER(ScanBatch), C.POINTER(vp), c_dp]),
    "lgs_bb_batch_upload_pairs": (C.c_int, [vp, C.POINTER(ScanBatch), C.c_int, c_ip, C.POINTER(vp), c_dp]),
    "lgs_bb_batch_run": (C.c_int, [vp]),
    "lgs_bb_batch_results": (C.c_int, [vp, C.POINTER(MatchResult)]),
    "lgs_bb_batch_work": (C.c_int, [vp, C.POINTER(C.c_longlong), C.c_int,
                                    C.POINTER(C.c_longlong)]),
    "lgs_bb_batch_force_replay": (C.c_int, [vp, C.c_int]),
    "lgs_bb_batch_set_record_ids": (C.c_int, [vp, C.POINTER(C.c_longlong), C.c_int]),
    "lgs_bb_batch_set_record_sink": (C.c_int, [vp, vp, C.c_longlong]),
    "lgs_bb_batch_records": (C.c_int, [vp, C.POINTER(LoopRecord)]),
    "lgs_bb_batch_settle": (C.c_int, [vp]),
    "lgs_bb_batch_device_records": (vp, [vp]),
    "lgs_bb_batch_phase_times": (C.c_int, [vp, c_dp, c_ip, C.c_int]),
    "lgs_bb_batch_query_nodes": (C.c_int, [vp, C.POINTER(C.c_longlong), C.c_int]),
    "lgs_bb_batch_skipped_gathers": (C.c_longlong, [vp]),
    "lgs_bb_batch_path": (C.c_int, [vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
    "lgs_group_create": (C.c_int, [c_ip, C.c_int, C.POINTER(vp)]),
    "lgs_group_destroy": (C.c_int, [vp]),
    "lgs_group_size": (C.c_int, [vp]),
    "lgs_group_ctx": (vp, [vp, C.c_int]),
    "lgs_group_last_error": (C.c_char_p, [vp]),
    "lgs_group_bb_create": (C.c_int, [vp, C.POINTER(BbParams), C.POINTER(vp)]),
    "lgs_group_bb_destroy": (C.c_int, [vp]),
    "lgs_group_bb_detect": (C.c_int, [vp, C.POINTER(ScanBatch), C.c_int, c_ip, C.POINTER(vp), c_dp,
                                      C.POINTER(MatchResult)]),
    "lgs_group_bb_records": (C.c_int, [vp, C.POINTER(LoopRecord)]),
    "lgs_comm_unique_id": (C.c_int, [vp]),
    "lgs_comm_create": (C.c_int, [vp, C.c_int, C.c_int, vp, C.POINTER(vp)]),
    "lgs_comm_destroy": (C.c_int, [vp]),
    "lgs_comm_all_gather_records": (C.c_int, [vp, vp, vp, C.c_int]),
    "lgs_bb_match": (C.c_int, [vp, C.POINTER(BbParams), C.POINTER(ScanBatch), C.POINTER(vp), c_dp,
                               C.POINTER(MatchResult)]),
}

_lib = None


def lib():
    """Load liblgs_b200.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LgsError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; "
                           "g.build()'` (nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)
            f.restype, f.argtypes = res, args
        _lib = L
    return _lib


def _dptr(a):
    return a.ctypes.data_as(c_dp)


def device_count() -> int:
    return lib().lgs_device_count()


class Context:
    def __init__(self, device: int = 0):
        self.h = vp()
        self._children = weakref.WeakSet()   # device objects that must die before the context
        rc = lib().lgs_ctx_create(device, C.byref(self.h))
        if rc != 0:
            self.h = None
            raise LgsError(f"lgs_ctx_create(device={device}) failed with {ERRORS.get(rc, rc)}: "
                           "a B200-class GPU is required, there is no CPU fallback")

    def check(self, rc: int):
        if rc != 0:
            msg = lib().lgs_ctx_last_error(self.h)
            raise LgsError(f"{ERRORS.get(rc, rc)}: {msg.decode() if msg else ''}")

    def synchronize(self):
        self.check(lib().lgs_ctx_synchronize(self.h))

    def wait_for(self, other: "Context"):
        """Stream order: what this context enqueues from now on runs after what `other` has enqueued so far."""
        self.check(lib().lgs_ctx_wait_ctx(self.h, other.h))

    def stream(self) -> int:
        return lib().lgs_ctx_stream(self.h) or 0

    def timer_start(self):
        self.check(lib().lgs_ctx_timer_start(self.h))

    def timer_stop(self) -> float:
        ms = C.c_float()
        self.check(lib().lgs_ctx_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def launch_count(self) -> int:
        return lib().lgs_ctx_launch_count(self.h)

    def set_option(self, name: str, value: float):
        """Per-context tuning / test hook (lgs_ctx_set_option); never changes results."""
        self.check(lib().lgs_ctx_set_option(self.h, name.encode(), float(value)))

    def get_option(self, name: str) -> float:
        v = C.c_double()
        self.check(lib().lgs_ctx_get_option(self.h, name.encode(), C.byref(v)))
        return v.value

    def set_edge_eps(self, eps: float):
        self.set_option("edge_eps", eps)

    def adopt(self, child):
        self._children.add(child)

    def close(self):
        if self.h:
            for child in list(self._children):
                child.close()
            if not getattr(self, "_borrowed", False):      # a Group owns its members' contexts
                lib().lgs_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Grid:
    """Dense device grid (double[ny][nx], 0.0 = unknown, zero apron)."""

    def __init__(self, ctx: Context, nx, ny, min_x, min_y, res, apron=64):
        self.ctx = ctx
        self.nx, self.ny, self.min_x, self.min_y, self.res, self.apron = \
            int(nx), int(ny), float(min_x), float(min_y), float(res), int(apron)
        self.h = vp()
        ctx.check(lib().lgs_grid_create(ctx.h, self.nx, self.ny, self.min_x, self.min_y,
                                        self.res, self.apron, C.byref(self.h)))
        ctx.adopt(self)

    @classmethod
    def from_dense(cls, ctx, dense, min_x, min_y, res, apron=64):
        dense = np.ascontiguousarray(dense, dtype=np.float64)
        g = cls(ctx, dense.shape[1], dense.shape[0], min_x, min_y, res, apron)
        g.upload(dense)
        return g

    def like(self):
        g = Grid(self.ctx, self.nx, self.ny, self.min_x, self.min_y, self.res, self.apron)
        if getattr(self, "off", (0, 0)) != (0, 0):
            g.set_window(*self.off)
        return g

    def set_window(self, off_x: int, off_y: int):
        """This grid holds cells [off, off + n) of a larger map with corner (min_x, min_y)."""
        self.ctx.check(lib().lgs_grid_set_window(self.h, int(off_x), int(off_y)))
        self.off = (int(off_x), int(off_y))

    def upload(self, dense):
        dense = np.ascontiguousarray(dense, dtype=np.float64)
        assert dense.shape == (self.ny, self.nx), (dense.shape, (self.ny, self.nx))
        self.ctx.check(lib().lgs_grid_upload(self.h, _dptr(dense)))

    def download(self):
        out = np.empty((self.ny, self.nx), dtype=np.float64)
        self.ctx.check(lib().lgs_grid_download(self.h, _dptr(out)))
        return out

    def precompute(self, win: int) -> "Grid":
        out = self.like()
        self.ctx.check(lib().lgs_precompute(self.ctx.h, self.h, int(win), out.h))
        return out

    def close(self):
        if getattr(self, "h", None):
            lib().lgs_grid_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Pyramid:
    def __init__(self, ctx: Context, grid: Grid, height_max: int):
        self.ctx, self.grid, self.height_max = ctx, grid, int(height_max)
        self.h = vp()
        ctx.check(lib().lgs_pyramid_create(ctx.h, grid.h, self.height_max, C.byref(self.h)))
        ctx.adopt(self)

    @classmethod
    def create_many(cls, ctx: Context, grids, height_max: int) -> list:
        """The pyramids of all `grids` in one call (lgs_pyramid_create_many): one launch per pass."""
        n = len(grids)
        handles = (vp * max(n, 1))(*[g.h for g in grids])
        out = (vp * max(n, 1))()
        ctx.check(lib().lgs_pyramid_create_many(ctx.h, n, handles, int(height_max), out))
        pyrs = []
        for g, h in zip(grids, out):
            p = cls.__new__(cls)
            p.ctx, p.grid, p.height_max, p.h = ctx, g, int(height_max), vp(h)
            ctx.adopt(p)
            pyrs.append(p)
        return pyrs

    def download(self, level: int):
        out = np.empty((self.grid.ny, self.grid.nx), dtype=np.float64)
        self.ctx.check(lib().lgs_pyramid_download(self.h, int(level), _dptr(out)))
        return out

    def close(self):
        if getattr(self, "h", None):
            lib().lgs_pyramid_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Scans:
    """Host-side scan batch in the C-ABI layout (keeps the numpy arrays alive)."""

    def __init__(self, angles_list, ranges_list, sensor_poses, range_min=None, range_max=None):
        n = len(ranges_list)
        assert len(angles_list) == n and len(sensor_poses) == n
        counts = [len(r) for r in ranges_list]
        self.beam_begin = np.zeros(n + 1, dtype=np.int32)
        self.beam_begin[1:] = np.cumsum(counts)
        self.angles = np.ascontiguousarray(np.concatenate(angles_list) if n else np.zeros(0),
                                           dtype=np.float64)
        self.ranges = np.ascontiguousarray(np.concatenate(ranges_list) if n else np.zeros(0),
                                           dtype=np.float64)
        self.sensor_pose = np.ascontiguousarray(np.asarray(sensor_poses, dtype=np.float64)
                                                .reshape(n, 3))
        self.n = n
        self.range_min = None if range_min is None else np.ascontiguousarray(
            np.broadcast_to(np.asarray(range_min, dtype=np.float64), (n,)))
        self.range_max = None if range_max is None else np.ascontiguousarray(
            np.broadcast_to(np.asarray(range_max, dtype=np.float64), (n,)))
        self.c = ScanBatch(n, self.beam_begin.ctypes.data_as(c_ip), _dptr(self.angles),
                           _dptr(self.ranges), _dptr(self.sensor_pose),
                           None if self.range_min is None else _dptr(self.range_min),
                           None if self.range_max is None else _dptr(self.range_max))

    @property
    def nbytes(self) -> int:
        return (self.beam_begin.nbytes + self.angles.nbytes + self.ranges.nbytes +
                self.sensor_pose.nbytes)


class RtcsmBatch:
    """lgs_rtcsm_batch: upload (host prep + H2D) / run (kernels) / results (D2H)."""

    def __init__(self, ctx: Context, low_res=5, range_x=1.0, range_y=1.0,
                 range_theta=1.0471975512, scan_range_max=20.0):
        self.ctx = ctx
        self.params = RtcsmParams(int(low_res), float(range_x), float(range_y),
                                  float(range_theta), float(scan_range_max))
        self.h = vp()
        ctx.check(lib().lgs_rtcsm_batch_create(ctx.h, C.byref(self.params), C.byref(self.h)))
        ctx.adopt(self)
        self.n = 0

    def upload(self, grid: Grid, scans: Scans, norm_threshold=None):
        thr = None
        if norm_threshold is not None:
            self._thr = np.ascontiguousarray(np.broadcast_to(
                np.asarray(norm_threshold, dtype=np.float64), (scans.n,)))
            thr = _dptr(self._thr)
        self._scans = scans
        self.ctx.check(lib().lgs_rtcsm_batch_upload(self.h, grid.h, C.byref(scans.c), thr))
        self.n = scans.n

    def run(self, grid: Grid, coarse: Grid):
        self.ctx.check(lib().lgs_rtcsm_batch_run(self.h, grid.h, coarse.h))

    def run_timed(self, grid: Grid, coarse: Grid):
        """-> (ms_project, ms_sweep, ms_select), CUDA events around each kernel."""
        ms = (C.c_float * 3)()
        self.ctx.check(lib().lgs_rtcsm_batch_run_timed(self.h, grid.h, coarse.h, ms))
        return tuple(ms)

    def results(self, grid: Grid, coarse: Grid):
        out = (MatchResult * max(self.n, 1))()
        self.ctx.check(lib().lgs_rtcsm_batch_results(self.h, grid.h, coarse.h, out))
        return list(out)[:self.n]

    def work(self):
        h, g = C.c_longlong(), C.c_longlong()
        self.ctx.check(lib().lgs_rtcsm_batch_work(self.h, C.byref(h), C.byref(g)))
        return h.value, g.value

    def fine_tiles(self):
        """-> (fine tiles the last scoring pass summed, tiles of the exhaustive sweep)."""
        n, total = C.c_longlong(), C.c_longlong()
        self.ctx.check(lib().lgs_rtcsm_batch_fine_tiles(self.h, C.byref(n), C.byref(total)))
        return n.value, total.value

    def debug(self, m: int):
        dims = (C.c_int * 6)()
        self.ctx.check(lib().lgs_rtcsm_batch_debug(self.h, m, dims, None, None, None))
        nt, nxw, nyw, nbx, nby, nk = list(dims)
        fine = np.empty((nt, nyw, nxw), dtype=np.float64)
        coarse = np.empty((nt, nbx, nby), dtype=np.float64)
        cells = np.empty((nt, max(nk, 0), 2), dtype=np.int32)
        self.ctx.check(lib().lgs_rtcsm_batch_debug(self.h, m, dims, _dptr(fine), _dptr(coarse),
                                                   cells.ctypes.data_as(c_ip)))
        return fine, coarse, cells

    def close(self):
        if getattr(self, "h", None):
            lib().lgs_rtcsm_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BbBatch:
    """lgs_bb_batch: breadth-first branch-and-bound over a batch of (scan, pyramid) queries."""

    def __init__(self, ctx: Context, node_height_max=6, range_x=2.0, range_y=2.0, range_theta=1.0,
                 scan_range_max=20.0, score_range_min=0.01, score_range_max=20.0):
        self.ctx = ctx
        self.params = BbParams(int(node_height_max), float(range_x), float(range_y),
                               float(range_theta), float(scan_range_max),
                               float(score_range_min), float(score_range_max))
        self.h = vp()
        ctx.check(lib().lgs_bb_batch_create(ctx.h, C.byref(self.params), C.byref(self.h)))
        ctx.adopt(self)
        self.n = 0

    def upload(self, scans: Scans, pyramids, norm_threshold=0.6):
        assert len(pyramids) == scans.n
        self._pyr = (vp * max(scans.n, 1))(*[p.h for p in pyramids])
        self._keep = (scans, list(pyramids))
        thr = None
        if norm_threshold is not None:
            self._thr = np.ascontiguousarray(np.broadcast_to(
                np.asarray(norm_threshold, dtype=np.float64), (scans.n,)))
            thr = _dptr(self._thr)
        self.ctx.check(lib().lgs_bb_batch_upload(self.h, C.byref(scans.c), self._pyr, thr))
        self.n = scans.n

    def upload_pairs(self, scans: Scans, pair_scan, pyramids, norm_threshold=0.6):
        """Pair q = (scans[pair_scan[q]], pyramids[q]); shared scans are projected once."""
        n = len(pyramids)
        self._pairs = np.ascontiguousarray(pair_scan, dtype=np.int32)
        assert len(self._pairs) == n
        if getattr(self, "_pyr_src", None) is not pyramids:         # same list object: reuse the handle array
            self._pyr = (vp * max(n, 1))(*[p.h for p in pyramids])
            self._pyr_src = pyramids
        self._keep = (scans, pyramids)
        thr = None
        if norm_threshold is not None:
            self._thr = np.ascontiguousarray(np.broadcast_to(
                np.asarray(norm_threshold, dtype=np.float64), (n,)))
            thr = _dptr(self._thr)
        self.ctx.check(lib().lgs_bb_batch_upload_pairs(self.h, C.byref(scans.c), n,
                                                       self._pairs.ctypes.data_as(c_ip), self._pyr, thr))
        self.n = n

    def run(self):
        self.ctx.check(lib().lgs_bb_batch_run(self.h))

    def results(self):
        out = (MatchResult * max(self.n, 1))()
        self.ctx.check(lib().lgs_bb_batch_results(self.h, out))
        return list(out)[:self.n]

    def results_array(self) -> np.ndarray:
        """Results as a numpy structured array with MatchResult's fields (no per-record objects)."""
        out = np.zeros(max(self.n, 1), dtype=MATCH_DTYPE)
        self.ctx.check(lib().lgs_bb_batch_results(self.h, out.ctypes.data_as(C.POINTER(MatchResult))))
        return out[:self.n]

    def work(self):
        lv = (C.c_longlong * 21)()
        g = C.c_longlong()
        self.ctx.check(lib().lgs_bb_batch_work(self.h, lv, 21, C.byref(g)))
        return list(lv)[:self.params.node_height_max + 1], g.value

    def force_replay(self, on: bool):
        self.ctx.check(lib().lgs_bb_batch_force_replay(self.h, int(on)))

    def set_record_ids(self, ids):
        """ids[q] goes into record q (from the next upload on); None restores the batch index."""
        if ids is None:
            self.ctx.check(lib().lgs_bb_batch_set_record_ids(self.h, None, 0))
            return
        self._ids = np.ascontiguousarray(ids, dtype=np.int64)
        self.ctx.check(lib().lgs_bb_batch_set_record_ids(
            self.h, self._ids.ctypes.data_as(C.POINTER(C.c_longlong)), len(self._ids)))

    def set_record_sink(self, device_ptr: int, first_slot: int = 0):
        """The finalize phase stores record q at device_ptr[first_slot + q] (may be peer memory)."""
        self.ctx.check(lib().lgs_bb_batch_set_record_sink(self.h, vp(device_ptr) if device_ptr else None,
                                                          int(first_slot)))

    def records(self) -> np.ndarray:
        out = np.zeros(max(self.n, 1), dtype=RECORD_DTYPE)
        self.ctx.check(lib().lgs_bb_batch_records(self.h, out.ctypes.data_as(C.POINTER(LoopRecord))))
        return out[:self.n]

    def settle(self):
        self.ctx.check(lib().lgs_bb_batch_settle(self.h))

    def device_records(self) -> int:
        return lib().lgs_bb_batch_device_records(self.h) or 0

    def phase_times(self):
        """(us per phase, lanes-per-node per phase) of the last device-only run ("bb_host_timing" on)."""
        n = self.params.node_height_max + 4
        us = np.zeros(n, dtype=np.float64)
        g = np.zeros(n, dtype=np.int32)
        self.ctx.check(lib().lgs_bb_batch_phase_times(self.h, _dptr(us), g.ctypes.data_as(c_ip), n))
        return us, g

    def skipped_gathers(self) -> int:
        """Beams the last device-only run left out through early rejection."""
        return int(lib().lgs_bb_batch_skipped_gathers(self.h))

    def query_nodes(self, n: int) -> np.ndarray:
        """Nodes below the root level scored per query by the last device-only run ("bb_host_timing" on)."""
        out = np.zeros(n, dtype=np.int64)
        self.ctx.check(lib().lgs_bb_batch_query_nodes(self.h, out.ctypes.data_as(C.POINTER(C.c_longlong)), n))
        return out

    def path(self):
        """(device-only runs, exact-path runs) of this batch object so far."""
        d, e = C.c_longlong(), C.c_longlong()
        self.ctx.check(lib().lgs_bb_batch_path(self.h, C.byref(d), C.byref(e)))
        return d.value, e.value

    def close(self):
        if getattr(self, "h", None):
            lib().lgs_bb_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Group:
    """lgs_group: all devices of one box driven from this process (one context + host thread per device)."""

    def __init__(self, devices):
        self.devices = [int(d) for d in devices]
        arr = (C.c_int * len(self.devices))(*self.devices)
        self.h = vp()
        rc = lib().lgs_group_create(arr, len(self.devices), C.byref(self.h))
        if rc != 0:
            self.h = None
            raise LgsError(f"lgs_group_create({self.devices}) failed with {ERRORS.get(rc, rc)}: peer-capable "
                           "B200-class GPUs are required, there is no fallback")
        self.ctxs = []
        for m in range(len(self.devices)):
            c = Context.__new__(Context)
            c.h = vp(lib().lgs_group_ctx(self.h, m))
            c._children = weakref.WeakSet()
            c._borrowed = True
            self.ctxs.append(c)

    def check(self, rc: int):
        if rc != 0:
            msg = lib().lgs_group_last_error(self.h)
            raise LgsError(f"{ERRORS.get(rc, rc)}: {msg.decode() if msg else ''}")

    def close(self):
        if getattr(self, "h", None):
            for c in self.ctxs:
                for child in list(c._children):
                    child.close()
                c.h = None
            lib().lgs_group_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GroupBb:
    """lgs_group_bb: branch-and-bound loop detection sharded over a Group by the device of each pyramid."""

    def __init__(self, group: Group, node_height_max=6, range_x=2.0, range_y=2.0, range_theta=1.0,
                 scan_range_max=20.0, score_range_min=0.01, score_range_max=20.0):
        self.group = group
        self.params = BbParams(int(node_height_max), float(range_x), float(range_y), float(range_theta),
                               float(scan_range_max), float(score_range_min), float(score_range_max))
        self.h = vp()
        group.check(lib().lgs_group_bb_create(group.h, C.byref(self.params), C.byref(self.h)))
        self.n = 0

    def detect(self, scans: "Scans", pair_scan, pyramids, norm_threshold=0.6) -> np.ndarray:
        n = len(pyramids)
        pairs = np.ascontiguousarray(pair_scan, dtype=np.int32)
        assert len(pairs) == n
        if getattr(self, "_pyr_src", None) is not pyramids:
            self._pyr = (vp * max(n, 1))(*[p.h for p in pyramids])
            self._pyr_src = pyramids
        thr = None
        if norm_threshold is not None:
            self._thr = np.ascontiguousarray(np.broadcast_to(np.asarray(norm_threshold, dtype=np.float64), (n,)))
            thr = _dptr(self._thr)
        out = np.zeros(max(n, 1), dtype=MATCH_DTYPE)
        self.group.check(lib().lgs_group_bb_detect(self.h, C.byref(scans.c), n, pairs.ctypes.data_as(c_ip), self._pyr,
                                                   thr, out.ctypes.data_as(C.POINTER(MatchResult))))
        self.n = n
        return out[:n]

    def records(self) -> np.ndarray:
        out = np.zeros(max(self.n, 1), dtype=RECORD_DTYPE)
        self.group.check(lib().lgs_group_bb_records(self.h, out.ctypes.data_as(C.POINTER(LoopRecord))))
        return out[:self.n]

    def close(self):
        if getattr(self, "h", None) and getattr(self.group, "h", None):
            lib().lgs_group_bb_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Comm:
    """lgs_comm: NCCL all-gather of loop records between one-process-per-GPU ranks."""

    @staticmethod
    def unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        if lib().lgs_comm_unique_id(buf) != 0:
            raise LgsError("lgs_comm_unique_id failed: libnccl.so.2 not loadable")
        return buf.raw

    def __init__(self, ctx: Context, world: int, rank: int, uid: bytes):
        self.ctx, self.world, self.rank = ctx, int(world), int(rank)
        self.h = vp()
        buf = C.create_string_buffer(uid, 128)
        ctx.check(lib().lgs_comm_create(ctx.h, self.world, self.rank, buf, C.byref(self.h)))

    def all_gather_records(self, recv_device: int, count: int, send_device: int = 0):
        self.ctx.check(lib().lgs_comm_all_gather_records(self.h, vp(send_device) if send_device else None,
                                                         vp(recv_device), int(count)))

    def close(self):
        if getattr(self, "h", None):
            lib().lgs_comm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def device_alloc(ctx: Context, nbytes: int) -> int:
    p = vp()
    ctx.check(lib().lgs_device_alloc(ctx.h, int(nbytes), C.byref(p)))
    return p.value


def device_free(ctx: Context, ptr: int):
    ctx.check(lib().lgs_device_free(ctx.h, vp(ptr)))


def download_records(ctx: Context, device_ptr: int, n: int) -> np.ndarray:
    """n 32-byte loop records from a device buffer (lgs_device_download)."""
    out = np.zeros(max(n, 1), dtype=RECORD_DTYPE)
    ctx.check(lib().lgs_device_download(ctx.h, vp(device_ptr), out.ctypes.data_as(vp), n * RECORD_DTYPE.itemsize))
    return out[:n]


def download_into(ctx: Context, device_ptr: int, out: np.ndarray):
    """Device -> an existing (ideally page-locked) host array."""
    ctx.check(lib().lgs_device_download(ctx.h, vp(device_ptr), out.ctypes.data_as(vp), out.nbytes))


# ---- occupancy-grid integration + host geometry helpers ------------------------------------------
class HitBatch(C.Structure):
    _fields_ = [("n_scans", C.c_int), ("sensor_xy", c_dp), ("hit_begin", c_ip), ("hit_xy", c_dp)]


class Geometry(C.Structure):
    _fields_ = [("nx", C.c_int), ("ny", C.c_int), ("min_x", C.c_double), ("min_y", C.c_double),
                ("res", C.c_double), ("patch", C.c_int)]

    def as_tuple(self):
        return (self.nx, self.ny, self.min_x, self.min_y, self.res)


SIGNATURES.update({
    "lgs_grid_resize": (C.c_int, [vp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int]),
    "lgs_grid_clear": (C.c_int, [vp]),
    "lgs_grid_copy": (C.c_int, [vp, vp]),
    "lgs_grid_download_region": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, c_dp, C.c_longlong]),
    "lgs_grid_integrate_scans": (C.c_int, [vp, vp, C.POINTER(HitBatch), C.c_double, C.c_double,
                                           C.POINTER(C.c_longlong)]),
    "lgs_grid_integrate_submit": (C.c_int, [vp, vp, C.POINTER(HitBatch), C.c_double, C.c_double]),
    "lgs_grid_integrate_wait": (C.c_int, [vp, C.POINTER(C.c_longlong)]),
    "lgs_grid_integrate_many": (C.c_int, [vp, C.c_int, C.POINTER(vp), C.POINTER(HitBatch), C.c_double, C.c_double,
                                          C.POINTER(C.c_longlong)]),
    "lgs_pyramid_create_many": (C.c_int, [vp, C.c_int, C.POINTER(vp), C.c_int, C.POINTER(vp)]),
    "lgs_ctx_integrate_fallback_cells": (C.c_longlong, [vp]),
    "lgs_scan_hit_points": (C.c_int, [c_dp, C.c_int, c_dp, c_dp, C.c_double, C.c_double, c_dp,
                                      c_ip, c_dp]),
    "lgs_geometry_resize": (C.c_int, [C.POINTER(Geometry)] + [C.c_double] * 4 +
                            [C.POINTER(Geometry), c_ip, c_ip]),
    "lgs_geometry_expand": (C.c_int, [C.POINTER(Geometry)] + [C.c_double] * 5 +
                            [C.POINTER(Geometry), c_ip, c_ip, c_ip]),
    "lgs_grid_construct_many": (C.c_int, [vp, C.c_int, C.POINTER(vp), C.POINTER(ScanBatch), C.POINTER(Geometry),
                                          C.c_double, C.c_double, C.POINTER(Geometry), c_dp,
                                          C.POINTER(C.c_longlong)]),
    "lgs_ctx_construct_host_points": (C.c_int, [vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
})


def scan_hit_points(sensor_pose, angles, ranges, range_min, range_max):
    """Range filter + HitPoint + bbox with the host's glibc arithmetic -> (hit_xy, bbox)."""
    a = np.ascontiguousarray(angles, dtype=np.float64)
    r = np.ascontiguousarray(ranges, dtype=np.float64)
    sp = np.ascontiguousarray(sensor_pose, dtype=np.float64)
    out = np.empty((len(a), 2), dtype=np.float64)
    n = C.c_int()
    bbox = np.empty(4, dtype=np.float64)
    rc = lib().lgs_scan_hit_points(_dptr(sp), len(a), _dptr(a), _dptr(r), range_min, range_max,
                                   _dptr(out), C.byref(n), _dptr(bbox))
    if rc != 0:
        raise LgsError(ERRORS.get(rc, rc))
    return out[:n.value].copy(), bbox


def geometry_expand(geo: Geometry, bbox, enlarge_step=5.0):
    out = Geometry()
    sx, sy, ch = C.c_int(), C.c_int(), C.c_int()
    rc = lib().lgs_geometry_expand(C.byref(geo), bbox[0], bbox[1], bbox[2], bbox[3], enlarge_step,
                                   C.byref(out), C.byref(sx), C.byref(sy), C.byref(ch))
    if rc != 0:
        raise LgsError(ERRORS.get(rc, rc))
    return out, sx.value, sy.value, bool(ch.value)


def geometry_resize(geo: Geometry, bbox):
    out = Geometry()
    sx, sy = C.c_int(), C.c_int()
    rc = lib().lgs_geometry_resize(C.byref(geo), bbox[0], bbox[1], bbox[2], bbox[3], C.byref(out),
                                   C.byref(sx), C.byref(sy))
    if rc != 0:
        raise LgsError(ERRORS.get(rc, rc))
    return out, sx.value, sy.value


def grid_resize(grid: Grid, geo: Geometry, shift_x: int, shift_y: int):
    grid.ctx.check(lib().lgs_grid_resize(grid.h, geo.nx, geo.ny, geo.min_x, geo.min_y, shift_x, shift_y))
    grid.nx, grid.ny, grid.min_x, grid.min_y = geo.nx, geo.ny, geo.min_x, geo.min_y


def grid_copy(src: Grid, dst: Grid):
    """Device -> device: dst takes src's geometry and cells (lgs_grid_copy)."""
    dst.ctx.check(lib().lgs_grid_copy(src.h, dst.h))
    dst.nx, dst.ny, dst.min_x, dst.min_y = src.nx, src.ny, src.min_x, src.min_y


def grid_download_region(grid: Grid, x0: int, y0: int, w: int, h: int) -> np.ndarray:
    """Cells [x0, x0 + w) x [y0, y0 + h) of the grid as an (h, w) array (lgs_grid_download_region)."""
    out = np.empty((h, w), dtype=np.float64)
    grid.ctx.check(lib().lgs_grid_download_region(grid.h, x0, y0, w, h, _dptr(out), max(w, 1)))
    return out


def grid_clear(grid: Grid):
    grid.ctx.check(lib().lgs_grid_clear(grid.h))


class PackedHits:
    """Host-side lgs_hit_batch (contiguous arrays kept alive), built once and integrated many times."""

    def __init__(self, sensor_xy, hits_list):
        n = len(hits_list)
        self.n = n
        self.begin = np.zeros(n + 1, dtype=np.int32)
        self.begin[1:] = np.cumsum([len(h) for h in hits_list])
        self.hit = np.ascontiguousarray(np.concatenate(hits_list) if n and self.begin[-1] else np.zeros((0, 2)),
                                        dtype=np.float64)
        sxy = np.asarray(sensor_xy, dtype=np.float64)
        self.sxy = np.ascontiguousarray(sxy.reshape(n, -1)[:, :2]) if n else np.zeros((0, 2))
        self.c = HitBatch(n, _dptr(self.sxy), self.begin.ctypes.data_as(c_ip), _dptr(self.hit))

    @property
    def nbytes(self):
        return self.hit.nbytes + self.sxy.nbytes + self.begin.nbytes


def integrate_packed(ctx: Context, grid: Grid, packed: PackedHits, p_hit=0.6, p_miss=0.45) -> int:
    cnt = C.c_longlong()
    ctx.check(lib().lgs_grid_integrate_scans(ctx.h, grid.h, C.byref(packed.c), p_hit, p_miss, C.byref(cnt)))
    return cnt.value


def integrate_submit(ctx: Context, grid: Grid, packed: PackedHits, p_hit=0.6, p_miss=0.45):
    """First half of integrate_packed: returns once the call is queued (up to two calls in flight)."""
    ctx.check(lib().lgs_grid_integrate_submit(ctx.h, grid.h, C.byref(packed.c), p_hit, p_miss))


def integrate_wait(ctx: Context) -> int:
    """Second half: cell updates of the oldest submitted call, once it is complete."""
    cnt = C.c_longlong()
    ctx.check(lib().lgs_grid_integrate_wait(ctx.h, C.byref(cnt)))
    return cnt.value


def integrate_scans(ctx: Context, grid: Grid, sensor_xy, hits_list, p_hit=0.6, p_miss=0.45) -> int:
    """lgs_grid_integrate_scans for scans given as (sensor_xy[k][2], [hit_xy arrays]) -> updates."""
    return integrate_packed(ctx, grid, PackedHits(sensor_xy, hits_list), p_hit, p_miss)


def integrate_many(ctx: Context, grids, sensor_xy_list, hits_lists, p_hit=0.6, p_miss=0.45) -> np.ndarray:
    """lgs_grid_integrate_many: the scans of map i (sensor_xy_list[i], hits_lists[i]) into grids[i], all
    maps in one call -> updates per map (int64 array)."""
    n = len(grids)
    assert len(sensor_xy_list) == n and len(hits_lists) == n
    packs = [PackedHits(s, h) for s, h in zip(sensor_xy_list, hits_lists)]
    batches = (HitBatch * max(n, 1))(*[p.c for p in packs])
    handles = (vp * max(n, 1))(*[g.h for g in grids])
    out = np.zeros(max(n, 1), dtype=np.int64)
    ctx.check(lib().lgs_grid_integrate_many(ctx.h, n, handles, batches, p_hit, p_miss,
                                            out.ctypes.data_as(C.POINTER(C.c_longlong))))
    return out[:n]


def construct_many(ctx: Context, grids, scans_list, cur_geometries, p_hit=0.6, p_miss=0.45):
    """lgs_grid_construct_many: ConstructMapFromScans of every map from raw scans (scans_list[i], a Scans with
    range_min / range_max) in one call; grids[i] is resized from cur_geometries[i] and rebuilt.
    -> (geometries [Geometry], bboxes [n][4] float64, updates [n] int64).  Each Grid's nx / ny / min_x / min_y
    follow its new geometry."""
    n = len(grids)
    assert len(scans_list) == n and len(cur_geometries) == n
    batches = (ScanBatch * max(n, 1))(*[s.c for s in scans_list])
    handles = (vp * max(n, 1))(*[g.h for g in grids])
    cur = (Geometry * max(n, 1))(*cur_geometries)
    geo = (Geometry * max(n, 1))()
    bbox = np.zeros((max(n, 1), 4), dtype=np.float64)
    out = np.zeros(max(n, 1), dtype=np.int64)
    ctx.check(lib().lgs_grid_construct_many(ctx.h, n, handles, batches, cur, p_hit, p_miss, geo, _dptr(bbox),
                                            out.ctypes.data_as(C.POINTER(C.c_longlong))))
    geos = [geo[i] for i in range(n)]
    for g, r in zip(grids, geos):
        g.nx, g.ny, g.min_x, g.min_y, g.res = r.nx, r.ny, r.min_x, r.min_y, r.res
    return geos, bbox[:n], out[:n]


def construct_host_points(ctx: Context):
    """(bbox candidates, near-edge hits) lgs_grid_construct_many re-derived on the host so far."""
    b, e = C.c_longlong(), C.c_longlong()
    ctx.check(lib().lgs_ctx_construct_host_points(ctx.h, C.byref(b), C.byref(e)))
    return b.value, e.value


def measure_gather_peak(ctx: Context, nx=960, ny=640, row_lanes=25, aligned=False, local=True) -> float:
    """Measured GB/s of warp-wide 8-byte row gathers from an nx x ny array (lgs_measure_gather_peak)."""
    g = C.c_double()
    ctx.check(lib().lgs_measure_gather_peak(ctx.h, nx, ny, row_lanes, int(aligned), int(local), C.byref(g)))
    return g.value


def pin(ctx: Context, *arrays):
    """Page-lock numpy arrays in place (lgs_host_pin) so uploads from them run at full speed."""
    for a in arrays:
        if a is not None and a.nbytes:
            ctx.check(lib().lgs_host_pin(ctx.h, a.ctypes.data_as(vp), a.nbytes))


def unpin(ctx: Context, *arrays):
    for a in arrays:
        if a is not None and a.nbytes:
            lib().lgs_host_unpin(ctx.h, a.ctypes.data_as(vp))


# ---- CostGreedyEndpoint: the matchers' tail ----------------------------------------------------
class CostParams(C.Structure):
    """lgs_cost_params: the CostGreedyEndpoint constructor's arguments, in its order."""
    _fields_ = [("usable_range_min", C.c_double), ("usable_range_max", C.c_double),
                ("hit_and_missed_dist", C.c_double), ("occupancy_threshold", C.c_double),
                ("kernel_size", C.c_int), ("scaling_factor", C.c_double),
                ("standard_deviation", C.c_double)]

    @classmethod
    def from_ctor_args(cls, args):
        a = list(args)
        return cls(a[0], a[1], a[2], a[3], int(a[4]), a[5], a[6])


# slam_launcher.cpp:60-72 with launcher_settings_default.json:2-10 (passes StandardDeviation in the
# scaling-factor slot and vice versa)
DEFAULT_COST_ARGS = (0.01, 20.0, 0.075, 0.1, 1, 0.05, 1.0)

SIGNATURES.update({
    "lgs_cost_greedy_endpoint": (C.c_int, [vp, vp, C.POINTER(CostParams), C.POINTER(ScanBatch), C.c_int,
                                           c_ip, c_dp, c_dp, c_ip]),
    "lgs_cost_tail": (C.c_int, [vp, vp, C.POINTER(CostParams), C.POINTER(ScanBatch), c_dp, c_dp, c_dp, c_ip]),
})


def cost_greedy_endpoint(ctx: Context, grid: Grid, scans: Scans, poses, pose_scan=None,
                         cost=DEFAULT_COST_ARGS):
    """CostGreedyEndpoint::Cost at each of `poses` ([n][3]) -> (costs, n_fixups)."""
    poses = np.ascontiguousarray(np.asarray(poses, dtype=np.float64).reshape(-1, 3))
    n = len(poses)
    ps = None if pose_scan is None else np.ascontiguousarray(pose_scan, dtype=np.int32)
    out = np.zeros(n, dtype=np.float64)
    fix = C.c_int()
    params = cost if isinstance(cost, CostParams) else CostParams.from_ctor_args(cost)
    ctx.check(lib().lgs_cost_greedy_endpoint(ctx.h, grid.h, C.byref(params), C.byref(scans.c), n,
                                             None if ps is None else ps.ctypes.data_as(c_ip),
                                             _dptr(poses), _dptr(out), C.byref(fix)))
    return out, fix.value


def cost_tail(ctx: Context, grid: Grid, scans: Scans, best_sensor_poses, cost=DEFAULT_COST_ARGS):
    """The matchers' tail per scan -> (normalised costs [n], covariances [n][3][3], n_fixups)."""
    best = np.ascontiguousarray(np.asarray(best_sensor_poses, dtype=np.float64).reshape(scans.n, 3))
    nc = np.zeros(scans.n, dtype=np.float64)
    cov = np.zeros((scans.n, 3, 3), dtype=np.float64)
    fix = C.c_int()
    params = cost if isinstance(cost, CostParams) else CostParams.from_ctor_args(cost)
    ctx.check(lib().lgs_cost_tail(ctx.h, grid.h, C.byref(params), C.byref(scans.c), _dptr(best), _dptr(nc),
                                  _dptr(cov), C.byref(fix)))
    return nc, cov, fix.value


# ---- exhaustive grid-search matcher ------------------------------------------------------------
class GsParams(C.Structure):
    _fields_ = [("range_x", C.c_double), ("range_y", C.c_double), ("range_theta", C.c_double),
                ("step_x", C.c_double), ("step_y", C.c_double), ("step_theta", C.c_double),
                ("score_range_min", C.c_double), ("score_range_max", C.c_double)]


SIGNATURES.update({
    "lgs_gs_match": (C.c_int, [vp, C.POINTER(GsParams), C.POINTER(ScanBatch), C.POINTER(vp), c_dp,
                               C.POINTER(MatchResult), c_dp]),
    "lgs_gs_offsets": (C.c_int, [C.c_double, C.c_double, c_dp, C.c_int, c_ip]),
})


def gs_offsets(rng: float, step: float) -> np.ndarray:
    """Offsets of the reference's accumulating loop for (range, step)."""
    n = C.c_int()
    rc = lib().lgs_gs_offsets(rng, step, None, 0, C.byref(n))
    if rc != 0:
        raise LgsError(f"lgs_gs_offsets({rng}, {step}) -> {rc}")
    out = np.zeros(n.value, dtype=np.float64)
    lib().lgs_gs_offsets(rng, step, _dptr(out), n.value, C.byref(n))
    return out


def gs_match(ctx: Context, scans: Scans, grids, *, range_x=2.0, range_y=2.0, range_theta=0.5, step_x=0.05,
             step_y=0.05, step_theta=0.005, score_range_min=0.01, score_range_max=20.0, norm_threshold=0.5,
             want_table=False):
    """ScanMatcherGridSearch for every scan of the batch against grids[q] -> list of MatchResult
    (+ the [nT][nY][nX] score table of a single query when want_table)."""
    assert len(grids) == scans.n
    params = GsParams(range_x, range_y, range_theta, step_x, step_y, step_theta, score_range_min,
                      score_range_max)
    handles = (vp * max(scans.n, 1))(*[g.h for g in grids])
    thr = None if norm_threshold is None else np.ascontiguousarray(
        np.broadcast_to(np.asarray(norm_threshold, dtype=np.float64), (scans.n,)))
    out = (MatchResult * max(scans.n, 1))()
    table = None
    if want_table:
        dims = [len(gs_offsets(range_theta, step_theta)), len(gs_offsets(range_y, step_y)),
                len(gs_offsets(range_x, step_x))]
        table = np.zeros(dims, dtype=np.float64)
    ctx.check(lib().lgs_gs_match(ctx.h, C.byref(params), C.byref(scans.c), handles,
                                 None if thr is None else _dptr(thr), out,
                                 None if table is None else _dptr(table)))
    res = [out[i] for i in range(scans.n)]
    return (res, table) if want_table else res
