"""Loop-closure rebuild probe: M local maps integrated again from their scans and their pyramids rebuilt, the
way GridMapBuilder::AfterLoopClosure and the loop detector's pyramid cache do after every loop closure.

Two versions, alternated within every repetition on the same grids:
  per_map  one lgs_grid_integrate_scans + one lgs_pyramid_create per map (what a caller of the one-map ABI pays);
  batched  one lgs_grid_integrate_many + one lgs_pyramid_create_many for all maps.
With --construct, ConstructMapFromScans from raw scans instead (no pyramids), the projection inside the window:
  host     lgs_scan_hit_points per scan, the bbox, lgs_geometry_resize, the grid resized and cleared per map,
           then one lgs_grid_integrate_many (the per-scan projection is a ctypes call from Python);
  raw      one lgs_grid_construct_many.
Both are driven through the C ABI directly (ctypes, pre-built handles and scan batches), so the host cost is
the library's.  Wall clock ends with a device synchronise; the CUDA-event time spans the same window on the
context stream.  Both versions must leave bit-identical cells, update counts and pyramid levels.

Local maps: windows of 10-40 consecutive scans (1081 beams, 270 degrees) of one trajectory through a
synth.World; map m starts at a random scan, so maps overlap like the local maps of a revisited area.

    python tools/rebuild_probe.py --maps 60 500 [--reps 5] [--height 6] [--construct]

Prints one JSON line.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from my_lidar_graph_slam_b200 import capi, synth  # noqa: E402

P_HIT, P_MISS = 0.6, 0.45


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout
        name, power = [s.strip() for s in out.splitlines()[0].split(",")]
        return name, power
    except Exception:
        return None, None


def make_maps(n_maps, seed):
    world = synth.World(60.0, 60.0, 20, seed=seed)
    angles = synth.beam_angles(1081, 270.0)
    n_scans = 1500
    traj = synth.trajectory(world, n_scans, step=0.25, seed=seed)
    noise = np.random.default_rng(seed + 1)
    hp = [capi.scan_hit_points(p, angles, synth.make_scan(world, p, angles, noise), 0.02, 20.0) for p in traj]
    rng = np.random.default_rng(seed + 2)
    maps = []
    for _ in range(n_maps):
        k = int(rng.integers(10, 41))
        lo = int(rng.integers(0, n_scans - k))
        sel = hp[lo:lo + k]
        bl = np.min([[b[0], b[1]] for _, b in sel], axis=0)
        tr = np.maximum(np.max([[b[2], b[3]] for _, b in sel], axis=0), np.finfo(np.float64).tiny)
        geo, _, _ = capi.geometry_resize(capi.Geometry(0, 0, 0.0, 0.0, 0.05, 64), (bl[0], bl[1], tr[0], tr[1]))
        maps.append((geo, capi.PackedHits(traj[lo:lo + k, :2], [h for h, _ in sel])))
    return maps


def make_raw_maps(n_maps, seed):
    """make_maps' local maps as raw scans (sensor pose = node pose, range window [0.02, 20])."""
    world = synth.World(60.0, 60.0, 20, seed=seed)
    angles = synth.beam_angles(1081, 270.0)
    n_scans = 1500
    traj = synth.trajectory(world, n_scans, step=0.25, seed=seed)
    noise = np.random.default_rng(seed + 1)
    ranges = [synth.make_scan(world, p, angles, noise) for p in traj]
    rng = np.random.default_rng(seed + 2)
    maps = []
    for _ in range(n_maps):
        k = int(rng.integers(10, 41))
        lo = int(rng.integers(0, n_scans - k))
        maps.append(capi.Scans([angles] * k, ranges[lo:lo + k], traj[lo:lo + k], range_min=0.02, range_max=20.0))
    return maps


class Construct:
    """ConstructMapFromScans of every map: `raw` in one lgs_grid_construct_many, `host` the way a caller without it
    does it."""

    def __init__(self, ctx, maps):
        self.ctx, self.L, self.n, self.maps = ctx, capi.lib(), len(maps), maps
        self.cur = (capi.Geometry * self.n)(*[capi.Geometry(0, 0, 0.0, 0.0, 0.05, 64)] * self.n)
        self.grids = [capi.Grid(ctx, 0, 0, 0.0, 0.0, 0.05, apron=2) for _ in maps]
        self.handles = (C.c_void_p * self.n)(*[g.h for g in self.grids])
        self.batches = (capi.ScanBatch * self.n)(*[s.c for s in maps])
        self.geo = (capi.Geometry * self.n)()
        self.bbox = np.zeros((self.n, 4))
        self.counts = np.zeros(self.n, dtype=np.int64)
        self.hit = [np.empty((int(s.beam_begin[-1]), 2)) for s in maps]
        self.hit_begin = [np.zeros(s.n + 1, dtype=np.int32) for s in maps]
        self.sensor = [np.ascontiguousarray(s.sensor_pose[:, :2]) for s in maps]
        self.hb = (capi.HitBatch * self.n)(*[capi.HitBatch(s.n, capi._dptr(self.sensor[i]),
                                                           self.hit_begin[i].ctypes.data_as(capi.c_ip),
                                                           capi._dptr(self.hit[i])) for i, s in enumerate(maps)])
        self.scratch = np.empty(4)

    def raw(self):
        self.ctx.check(self.L.lgs_grid_construct_many(self.ctx.h, self.n, self.handles, self.batches, self.cur, P_HIT,
                                                      P_MISS, self.geo, capi._dptr(self.bbox),
                                                      self.counts.ctypes.data_as(C.POINTER(C.c_longlong))))
        for g, geo in zip(self.grids, self.geo):
            g.nx, g.ny, g.min_x, g.min_y = geo.nx, geo.ny, geo.min_x, geo.min_y

    def host(self):
        L, nh = self.L, C.c_int()
        tiny, big = float(np.finfo(np.float64).tiny), float(np.finfo(np.float64).max)
        for i, s in enumerate(self.maps):
            bl, tr = [big, big], [tiny, tiny]
            hb, hit, bb = self.hit_begin[i], self.hit[i], self.scratch
            for k in range(s.n):
                b0 = int(s.beam_begin[k])
                L.lgs_scan_hit_points(capi._dptr(s.sensor_pose[k]), int(s.beam_begin[k + 1]) - b0,
                                      capi._dptr(s.angles[b0:]), capi._dptr(s.ranges[b0:]), float(s.range_min[k]),
                                      float(s.range_max[k]), capi._dptr(hit[hb[k]:]), C.byref(nh), capi._dptr(bb))
                hb[k + 1] = hb[k] + nh.value
                bl[0], bl[1] = min(bl[0], bb[0]), min(bl[1], bb[1])
                tr[0], tr[1] = max(tr[0], bb[2]), max(tr[1], bb[3])
            self.bbox[i] = (bl[0], bl[1], tr[0], tr[1])
            L.lgs_geometry_resize(C.byref(self.cur[i]), bl[0], bl[1], tr[0], tr[1], C.byref(self.geo[i]), None, None)
            g, geo = self.grids[i], self.geo[i]
            if (g.nx, g.ny, g.min_x, g.min_y) == (geo.nx, geo.ny, geo.min_x, geo.min_y):
                capi.grid_clear(g)                                         # Reset
            else:                                                          # Resize with nothing kept
                self.ctx.check(L.lgs_grid_resize(g.h, geo.nx, geo.ny, geo.min_x, geo.min_y, 1 << 30, 1 << 30))
            g.nx, g.ny, g.min_x, g.min_y = geo.nx, geo.ny, geo.min_x, geo.min_y
        self.ctx.check(L.lgs_grid_integrate_many(self.ctx.h, self.n, self.handles, self.hb, P_HIT, P_MISS,
                                                 self.counts.ctypes.data_as(C.POINTER(C.c_longlong))))

    def timed(self, fn):
        launches = self.ctx.launch_count()
        t0 = time.perf_counter()
        self.ctx.timer_start()
        fn()
        ms = self.ctx.timer_stop()
        self.ctx.synchronize()
        return (time.perf_counter() - t0) * 1e3, ms, self.ctx.launch_count() - launches

    def state(self):
        return ([tuple(self.geo[i].as_tuple()) for i in range(self.n)], self.bbox.copy(), self.counts.copy(),
                [g.download().view(np.int64) for g in self.grids])

    def close(self):
        for g in self.grids:
            g.close()


def run_construct(ctx, args, out):
    for m in args.maps:
        maps = make_raw_maps(m, args.seed)
        a, b = Construct(ctx, maps), Construct(ctx, maps)
        a.timed(a.host)                                        # warm-up: workspaces, pools, modules
        b.timed(b.raw)
        runs = {"host": [], "raw": []}
        for _ in range(args.reps):                             # alternated: both see the same box state
            runs["host"].append(a.timed(a.host))
            runs["raw"].append(b.timed(b.raw))
        sa, sb = a.state(), b.state()
        same = (sa[0] == sb[0] and np.array_equal(sa[1].view(np.int64), sb[1].view(np.int64)) and
                np.array_equal(sa[2], sb[2]) and all(np.array_equal(x, y) for x, y in zip(sa[3], sb[3])))
        assert same, f"{m} maps: raw and host differ"
        bbox_pts, edge_pts = capi.construct_host_points(ctx)
        res = {"maps": m, "scans": int(sum(s.n for s in maps)), "beams": int(sum(s.beam_begin[-1] for s in maps)),
               "hits": int(sum(int(h[-1]) for h in a.hit_begin)), "identical": same, "updates": int(b.counts.sum()),
               "host_points_so_far": {"bbox": bbox_pts, "edge": edge_pts}}
        for k, r in runs.items():
            wall = [x[0] for x in r]
            ev = [x[1] for x in r]
            res[k] = {"wall_ms": float(np.median(wall)), "wall_ms_min": float(np.min(wall)),
                      "wall_ms_max": float(np.max(wall)), "event_ms": float(np.median(ev)),
                      "event_ms_min": float(np.min(ev)), "event_ms_max": float(np.max(ev)), "launches": int(r[-1][2])}
        res["speedup_wall"] = res["host"]["wall_ms"] / res["raw"]["wall_ms"]
        out["results"].append(res)
        a.close()
        b.close()


class Version:
    def __init__(self, ctx, maps, height):
        L = capi.lib()
        self.ctx, self.L, self.height, self.n = ctx, L, height, len(maps)
        self.grids = [capi.Grid(ctx, g.nx, g.ny, g.min_x, g.min_y, g.res, apron=2) for g, _ in maps]
        self.handles = (C.c_void_p * self.n)(*[g.h for g in self.grids])
        self.batches = (capi.HitBatch * self.n)(*[p.c for _, p in maps])
        self.packs = [p for _, p in maps]
        self.counts = np.zeros(self.n, dtype=np.int64)
        self.pyrs = (C.c_void_p * self.n)()

    def reset(self):
        for p in range(self.n):
            if self.pyrs[p]:
                self.L.lgs_pyramid_destroy(self.pyrs[p])
                self.pyrs[p] = None
        for g in self.grids:
            capi.grid_clear(g)
        self.ctx.synchronize()

    def per_map(self):
        cnt = C.c_longlong()
        for i in range(self.n):
            self.ctx.check(self.L.lgs_grid_integrate_scans(self.ctx.h, self.handles[i], C.byref(self.batches[i]),
                                                           P_HIT, P_MISS, C.byref(cnt)))
            self.counts[i] = cnt.value
            h = C.c_void_p()
            self.ctx.check(self.L.lgs_pyramid_create(self.ctx.h, self.handles[i], self.height, C.byref(h)))
            self.pyrs[i] = h.value

    def batched(self):
        self.ctx.check(self.L.lgs_grid_integrate_many(self.ctx.h, self.n, self.handles, self.batches, P_HIT, P_MISS,
                                                      self.counts.ctypes.data_as(C.POINTER(C.c_longlong))))
        self.ctx.check(self.L.lgs_pyramid_create_many(self.ctx.h, self.n, self.handles, self.height, self.pyrs))

    def timed(self, fn):
        self.reset()
        launches = self.ctx.launch_count()
        t0 = time.perf_counter()
        self.ctx.timer_start()
        fn()
        ms = self.ctx.timer_stop()
        self.ctx.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        return wall, ms, self.ctx.launch_count() - launches

    def close(self):
        self.reset()
        for g in self.grids:
            g.close()


def identical(a: Version, b: Version) -> bool:
    if not np.array_equal(a.counts, b.counts):
        return False
    for i, (ga, gb) in enumerate(zip(a.grids, b.grids)):
        if not np.array_equal(ga.download().view(np.int64), gb.download().view(np.int64)):
            return False
        buf_a, buf_b = np.empty((ga.ny, ga.nx)), np.empty((gb.ny, gb.nx))
        for lvl in range(a.height + 1):
            a.ctx.check(a.L.lgs_pyramid_download(a.pyrs[i], lvl, capi._dptr(buf_a)))
            b.ctx.check(b.L.lgs_pyramid_download(b.pyrs[i], lvl, capi._dptr(buf_b)))
            if not np.array_equal(buf_a.view(np.int64), buf_b.view(np.int64)):
                return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--maps", type=int, nargs="+", default=[60, 500])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--height", type=int, default=6)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--construct", action="store_true", help="raw vs host ConstructMapFromScans instead")
    args = ap.parse_args()
    ctx = capi.Context(0)
    name, power = gpu_info()
    out = {"probe": "construct" if args.construct else "rebuild", "gpu": name, "power_limit": power,
           "height_max": args.height, "reps": args.reps, "results": []}
    if args.construct:
        run_construct(ctx, args, out)
    for m in ([] if args.construct else args.maps):
        maps = make_maps(m, args.seed)
        a, b = Version(ctx, maps, args.height), Version(ctx, maps, args.height)
        a.timed(a.per_map)                                     # warm-up: workspaces, pools, modules
        b.timed(b.batched)
        runs = {"per_map": [], "batched": []}
        for _ in range(args.reps):                             # alternated: both see the same box state
            runs["per_map"].append(a.timed(a.per_map))
            runs["batched"].append(b.timed(b.batched))
        res = {"maps": m, "scans": int(sum(p.n for _, p in maps)), "hits": int(sum(p.begin[-1] for _, p in maps)),
               "cells": int(sum(g.nx * g.ny for g, _ in maps)), "identical": identical(a, b),
               "updates": int(b.counts.sum())}
        for k, r in runs.items():
            wall = [x[0] for x in r]
            ev = [x[1] for x in r]
            res[k] = {"wall_ms": float(np.median(wall)), "wall_ms_min": float(np.min(wall)),
                      "wall_ms_max": float(np.max(wall)), "event_ms": float(np.median(ev)),
                      "launches": int(r[-1][2]), "maps_per_s": m / (float(np.median(wall)) / 1e3)}
        res["speedup_wall"] = res["per_map"]["wall_ms"] / res["batched"]["wall_ms"]
        out["results"].append(res)
        a.close()
        b.close()
    ctx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
