#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native scan-matching backend.

BASELINE.json metric: "pose hypotheses scored/sec; loop-closure queries/sec at 1/2/4/8 B200".

  --gpus 1   headline = C2 (BASELINE configs[1]): real-time correlative sweep, 1081-beam 270-degree scans,
             +-0.5 m / +-30 deg window at 0.05 m / 0.5 deg, lowRes 5, one ~800x800 map.  One STEP = the coarse
             win-max precompute of the map + one batch of `--matches` matches through the C ABI.
             metric = pose hypotheses scored per second.  The loop-closure half of the metric (C4) is
             measured in the same run and reported in the `loop_closure` block of the line.
  --gpus N   headline = C4 (BASELINE configs[3]): branch-and-bound loop detection against 500 submaps,
             7 precompute levels, STRONG scaling: submap i lives on rank i mod N, every rank searches its own
             pairs with ONE persistent kernel launch per device batch, the 32-byte result records are written
             by that kernel into the rank's slice of the exchange buffer and all-gathered in place on the
             device (lgs_comm: NCCL on the context stream).  value = loop queries/s for a step of 64 query
             scans x 500 submaps (the throughput form); `single_scan` = one scan x 500 submaps (the
             latency form).  Rank 0 also measures the same steps with all 500 submaps on its own GPU
             (`n1_same_run`), so the line carries its own strong-scaling reference.  The C2 replicas
             (weak scaling; the front-end match does not shard, SURVEY.md 8(e)) move to `extra`.

  value      kernels only, inputs resident in HBM, CUDA events on the context stream, max over ranks.
  e2e        the same step through the public API with HOST buffers (H2D of the inputs, kernels, record
             exchange, D2H of the records), wall clock with a device sync on both sides, max over ranks.
  roofline   bound "l1_gather": the scoring kernels read maps that are L1/L2 resident by design; achieved =
             algorithmic gathered bytes / kernel time, peak = the gather bandwidth measured in this run
             (lgs_measure_gather_peak), `peak_theoretical` = 148 SMs x 128 B/clk x f_sm; the HBM view is in
             `hbm` (traffic needs ncu: profiles/).
  cpu_baseline / --impl reference
             the UNMODIFIED reference classes (oracle/_ref/liblgs_ref.so) on the host cores: the correlative
             matcher at N = 1, the branch-and-bound matcher at N > 1 (rank 0 only).
  --dump-outputs DIR
             after the timed steps, what the last one computed as DIR/<name>.npy (float64): the C2 match
             records (c2_found, c2_ix, c2_iy, c2_it, c2_score, c2_window, c2_step) and coarse map
             (c2_coarse_map) of the kernels-only C2 loop, and the C4 records of the 64-scan step in pair order
             (c4_*), as gathered by the last step of its timed end-to-end loop (the kernels-only C4 loop gathers
             no records; it runs on the same inputs).  The inputs are seeded, so two builds run with the same
             arguments can be compared array for array.
Details that do not fit the one-line contract go to DIR/bench_details_n<N>.json with --details DIR.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from my_lidar_graph_slam_b200 import synth  # noqa: E402

C2 = dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=1.0471975512, scan_range_max=5.7296)
METRIC = "pose hypotheses scored/sec (C2 correlative sweep)"
UNIT = "hypotheses/s"


def build_map_on_gpu(ctx, poses, angles, ranges_list, apron, usable=(0.02, 20.0)):
    """Product path: range filter + hit points on the host (lgs_scan_hit_points), map geometry
    grown like GridMap::Expand (lgs_geometry_expand), then ONE lgs_grid_integrate_scans batch."""
    from my_lidar_graph_slam_b200 import capi
    geo = capi.Geometry(0, 0, float(poses[0][0]), float(poses[0][1]), 0.05, 64)
    hits = []
    for p, r in zip(poses, ranges_list):
        h, bbox = capi.scan_hit_points(p, angles, r, usable[0], usable[1])
        geo, _, _, _ = capi.geometry_expand(geo, bbox)
        hits.append(h)
    grid = capi.Grid(ctx, geo.nx, geo.ny, geo.min_x, geo.min_y, 0.05, apron=apron)
    updates = capi.integrate_scans(ctx, grid, np.asarray(poses)[:, :2], hits)
    return grid, updates


def c2_workload(n_matches: int, seed: int = 1):
    """Map scans + n_matches (scan, perturbed initial pose) pairs, all seeded."""
    world = synth.RoomsWorld(40.0, 5.0, seed=seed + 1)   # office-like: most ranges < 5.7 m
    angles = synth.beam_angles(1081, 270.0)
    traj = synth.trajectory(world, 10, step=0.4, seed=seed + 1)
    noise = np.random.default_rng(seed + 1)           # range noise
    map_scans = [synth.make_scan(world, p, angles, noise) for p in traj]
    pert = np.random.default_rng(seed + 2)            # pose perturbations
    ranges, inits = [], []
    while len(ranges) < n_matches:
        base = traj[pert.integers(0, len(traj))]
        true = base + np.array([pert.uniform(-0.6, 0.6), pert.uniform(-0.6, 0.6),
                                pert.uniform(-0.5, 0.5)])
        if not world.is_free(true[0], true[1], 0.3):
            continue
        ranges.append(synth.make_scan(world, true, angles, noise))
        inits.append(true + np.array([pert.uniform(-0.3, 0.3), pert.uniform(-0.3, 0.3),
                                      pert.uniform(-0.2, 0.2)]))
    return traj, map_scans, angles, ranges, np.asarray(inits)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100", "-i", str(self.device)], stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(smax) if smax else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ref_time_matches(dense, min_x, min_y, angles, ranges, inits, n_threads):
    """Time the reference matcher (incl. its own coarse-map precompute, as OptimizePose(query)
    does once per call) over the given matches on n_threads host threads."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import refapi as R
    refmap = R.RefMap.from_dense(dense, min_x, min_y)

    def one(k):
        return R.rtcsm_match(refmap, angles, ranges[k], inits[k], **C2)   # pre=None: precompute inside

    one(0)   # warm-up (page in, allocate)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=n_threads) as ex:   # ctypes releases the GIL
        res = list(ex.map(one, range(len(ranges))))
    return time.perf_counter() - t0, res


def hyps_per_match(res):
    nbx = (2 * res.winX) // 5 + 1
    nby = (2 * res.winY) // 5 + 1
    return (2 * res.winT + 1) * (nbx * 5 * nby * 5 + nbx * nby)



def c2_config(M):
    """The `config` object of the C2 line -- shared by both arms so that they describe the same workload."""
    return {"workload": "C2 rtcsm 1081 beams +-0.5m/+-30deg", "matches_per_step": int(M), **C2}


# ---- C4: branch-and-bound loop detection -------------------------------------------------------------
BB = dict(node_height_max=6, range_x=2.0, range_y=2.0, range_theta=1.0, scan_range_max=20.0,
          score_range_min=0.01, score_range_max=20.0)
C4_METRIC = "loop-closure queries/sec (C4 branch-and-bound)"
C4_UNIT = "loop queries/s"
C4_SCANS = 64


def c4_config(n_submaps, world):
    return {"workload": f"C4 B&B {C4_SCANS} scans x {n_submaps} submaps, 7 levels",
            "submaps": int(n_submaps), "scans_per_step": C4_SCANS, **BB}


def c4_submap_scans(world, angles, submap_id, n_scans, anchor):
    """Deterministic scans of one submap: the first ten submaps start near `anchor` (they contain
    the query location), the others anywhere in the world."""
    rng = np.random.default_rng(10_000 + submap_id)
    if submap_id < 10:
        start = (anchor[0] + rng.uniform(-0.5, 0.5), anchor[1] + rng.uniform(-0.5, 0.5),
                 anchor[2] + rng.uniform(-0.3, 0.3))
        if not world.is_free(start[0], start[1], 0.6):
            start = tuple(anchor)
        traj = synth.trajectory(world, n_scans, step=0.3, seed=submap_id, start=start)
    else:
        traj = synth.trajectory(world, n_scans, step=0.3, seed=submap_id)
    return traj, [synth.make_scan(world, p, angles, rng) for p in traj]


def c4_scene():
    world = synth.RoomsWorld(60.0, 5.0, seed=4)
    angles = synth.beam_angles(1081, 270.0)
    anchor = synth.trajectory(world, 1, seed=77)[0]
    qrng = np.random.default_rng(5)
    truth = anchor + np.array([0.2, -0.1, 0.05])
    scans, inits = [synth.make_scan(world, truth, angles, qrng)], [truth + np.array([0.4, -0.3, 0.1])]
    for k in range(1, C4_SCANS):
        t = anchor + np.array([0.3 * np.cos(k), 0.3 * np.sin(k), 0.04 * k])
        scans.append(synth.make_scan(world, t, angles, qrng))
        inits.append(t + np.array([0.3, -0.2, 0.08]))
    return world, angles, anchor, scans, inits


class C4Shard:
    """The submaps `ids` of the C4 scene on one context (grids + pyramids), and the loop-detection steps
    of one rank against them."""

    def __init__(self, ctx, scene, ids, reuse=None):
        from my_lidar_graph_slam_b200 import capi
        world, angles, anchor, self.qscans, self.qinits = scene
        self.ctx, self.angles, self.ids = ctx, angles, np.asarray(ids, dtype=np.int64)
        self.grids, self.pyramids, self.cells = [], [], 0
        reuse = reuse or {}                                   # submap id -> grid already on this device (re-placement)
        for g in self.ids:
            grid = reuse.pop(int(g), None)
            if grid is None:
                traj, scans = c4_submap_scans(world, angles, int(g), 8, anchor)
                grid, _ = build_map_on_gpu(ctx, traj, angles, scans, apron=1)
            self.grids.append(grid)
            self.cells += grid.nx * grid.ny
        for grid in reuse.values():
            grid.close()
        # the first build of the pyramids grows the stream-ordered memory pool (one-time cost); the timed
        # build is a REbuild of every pyramid, which is what the loop detector does whenever a submap
        # has changed (loop_detector_branch_bound.cpp:44-53)
        warm = [capi.Pyramid(ctx, g, 6) for g in self.grids]
        for p in warm:
            p.close()
        ctx.synchronize()
        ctx.timer_start()
        self.pyramids = [capi.Pyramid(ctx, g, 6) for g in self.grids]
        self.pyramid_ms = ctx.timer_stop()

    def groups(self, n_scans, n_submaps_total, sub_scans):
        """Device sub-batches of `sub_scans` query scans x this shard's submaps: (Scans, pair_scan, pyramids,
        global pair ids) per sub-batch.  Pair id = scan * n_submaps_total + submap."""
        from my_lidar_graph_slam_b200 import capi
        out = []
        nq = len(self.ids)
        for k0 in range(0, n_scans, sub_scans):
            ks = list(range(k0, min(k0 + sub_scans, n_scans)))
            out.append(dict(
                scans=capi.Scans([self.angles] * len(ks), [self.qscans[k] for k in ks], [self.qinits[k] for k in ks],
                                 range_min=0.02, range_max=30.0),
                pair_scan=np.repeat(np.arange(len(ks), dtype=np.int32), nq),
                pyr=self.pyramids * len(ks),
                ids=np.concatenate([k * n_submaps_total + self.ids for k in ks]) if nq else np.zeros(0, dtype=np.int64)))
        return out

    def submap_cost_terms(self, n_submaps_total, thr=0.6):
        """One plain step of all query scans against this shard's submaps with the kernel's phase clock on:
        (deep nodes scored per submap, [root us, root nodes, deeper-level us, deeper-level nodes]).  Root
        nodes are the same for every pair; what differs between submaps is how deep the search goes, and a
        node of a deeper level costs more than a root node (scattered parents), so the placement weighs
        the two with their measured times."""
        from my_lidar_graph_slam_b200 import capi
        deep = np.zeros(n_submaps_total, dtype=np.float64)
        terms = np.zeros(4, dtype=np.float64)
        nq = len(self.ids)
        if nq == 0:
            return deep, terms
        sub = c4_sub_scans(len(self.qscans), nq)
        self.ctx.set_option("bb_host_timing", 1)
        try:
            for g in self.groups(len(self.qscans), n_submaps_total, sub):
                b = capi.BbBatch(self.ctx, **BB)
                b.upload_pairs(g["scans"], g["pair_scan"], g["pyr"], thr)
                b.run()
                res = b.results_array()
                b.run()                                           # pools sized: a clean device-only run to time
                res = b.results_array()
                us, _ = b.phase_times()
                levels, _ = b.work()
                np.add.at(deep, g["ids"] % n_submaps_total, b.query_nodes(len(g["ids"])).astype(np.float64))
                H = len(levels) - 1
                terms += [us[1], levels[-1], float(sum(us[2:2 + H])), float(sum(levels[:-1]))]
                b.close()
        finally:
            self.ctx.set_option("bb_host_timing", 0)
        return deep, terms

    def release_grids(self):
        """Close the pyramids and hand the grids over (submap id -> grid) to the shard that replaces this one."""
        for p in self.pyramids:
            p.close()
        self.pyramids = []
        out = {int(g): grid for g, grid in zip(self.ids, self.grids)}
        self.grids = []
        return out

    def close(self):
        for p in self.pyramids:
            p.close()
        for g in self.grids:
            g.close()


def c4_sub_scans(n_scans, nq):
    """Query scans per device sub-batch: ~8000 pairs (the hit points of a sub-batch, 2.7 MB per scan and
    layout, stay L2 resident while its levels are large enough to fill the persistent grid).  Measured at
    8 GPUs: one sub-batch of 64 x 63 pairs per rank 4.18 ms, two of 32 x 63 4.56 ms."""
    if "LGS_C4_SUB" in os.environ:
        return max(1, int(os.environ["LGS_C4_SUB"]))
    return max(1, min(n_scans, -(-8000 // max(nq, 1))))


def c4_steps(lanes, shard, rank, world, n_submaps, n_scans, steps, barrier, max_over_ranks, thr=0.6, placement=None,
             details=None):
    """Time the loop-detection step `n_scans` query scans x `n_submaps` submaps with this rank's shard:
    kernels only (inputs resident) and end to end (host scans in, gathered records out).
    lanes = [(ctx, comm), (ctx2, comm2)]: the end-to-end value pipelines consecutive steps over the two
    contexts (= two CUDA streams, each with its own batch objects, exchange buffer and communicator): the host
    preparation and upload of step k + 1 run under the kernel of step k, and every step still moves its own
    inputs to the device and its own gathered records back; `qps_e2e_sequential` is the strictly sequential
    figure (upload -> kernel -> exchange -> download, one step after the other)."""
    from my_lidar_graph_slam_b200 import capi, sharding
    nq = len(shard.ids)
    sub = c4_sub_scans(n_scans, nq)
    groups = shard.groups(n_scans, n_submaps, sub)
    seg = []
    if placement is None:
        placement = sharding.round_robin_placement(n_submaps, world)
    for r in range(world):
        cnt = len(placement[r])
        seg.append([cnt * len(range(k0, min(k0 + sub, n_scans))) for k0 in range(0, n_scans, sub)])
    L = []
    for ctx_l, comm_l in lanes:
        ex = sharding.RecordExchange(ctx_l, comm_l, n_scans * n_submaps, rank, world, seg)
        batches = [capi.BbBatch(ctx_l, **BB) for _ in groups]
        for k, (b, g) in enumerate(zip(batches, groups)):
            ex.attach(b, g["ids"], k)
        L.append(dict(ctx=ctx_l, ex=ex, batches=batches))
    ctx = L[0]["ctx"]

    lane_order = world > 1 and os.environ.get("LGS_C4_LANE_ORDER", "1") != "0"   # 8 GPUs: 6.9 -> 7.5 M queries/s end to end

    def submit(lane):
        for b, g in zip(lane["batches"], groups):
            b.upload_pairs(g["scans"], g["pair_scan"], g["pyr"], thr)
        if lane_order:
            # the uploads above may run under the other lane's kernels; this lane's persistent kernels (which
            # take every SM) start only behind the other lane's record exchange, whose NCCL kernel would
            # otherwise wait a whole step for an SM
            for other in L:
                if other is not lane:
                    lane["ctx"].wait_for(other["ctx"])
        for b in lane["batches"]:
            b.run()
        lane["ex"].launch_gather()

    def collect(lane):
        return lane["ex"].finish_launched(lane["batches"])

    def sync_all():
        for lane in L:
            lane["ctx"].synchronize()

    for lane in L:
        for _ in range(2):
            submit(lane)
            rec = collect(lane)
    sync_all()
    barrier()
    t0 = time.perf_counter()                                  # (a) strictly sequential
    for _ in range(steps):
        submit(L[0])
        rec = collect(L[0])
    sync_all()
    e2e_seq_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    t0 = time.perf_counter()                                  # (b) pipelined over the lanes
    submit(L[0])
    for k in range(1, steps):
        submit(L[k % len(L)])
        rec = collect(L[(k - 1) % len(L)])
    rec = collect(L[(steps - 1) % len(L)])
    sync_all()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    # kernels only: scans + pyramids resident, one persistent kernel launch per sub-batch and step
    batches = L[0]["batches"]
    for b, g in zip(batches, groups):
        b.upload_pairs(g["scans"], g["pair_scan"], g["pyr"], thr)
    sync_all()
    barrier()
    launches0 = ctx.launch_count()
    ctx.timer_start()
    for _ in range(steps):
        for b in batches:
            b.run()
    dev_ms_local = ctx.timer_stop()
    dev_ms = max_over_ranks(dev_ms_local)
    launches = ctx.launch_count() - launches0
    if os.environ.get("LGS_C4_RANK_DIAG"):                      # per-rank kernel time / work of this step shape (scratch)
        ctx.set_option("bb_host_timing", 1)
        ph = []
        for b in batches:
            b.run()
            b.results_array()
            ph.append([round(float(x), 1) for x in b.phase_times()[0]])
        ctx.set_option("bb_host_timing", 0)
        d = details or tempfile.gettempdir()
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, f"c4_rank{rank}_of{world}_q{n_scans}.json"), "w") as f:
            json.dump({"rank": rank, "submaps": int(nq), "ms_per_step": dev_ms_local / steps, "phases_us": ph,
                       "levels": [b.work()[0] for b in batches]}, f)
    nodes, gathers, skipped, dev_runs, exact_runs = 0, 0, 0, 0, 0
    for b in batches:
        lv, ga = b.work()
        nodes += int(sum(lv))
        gathers += int(ga)
        skipped += b.skipped_gathers()
    for lane in L:
        for b in lane["batches"]:
            d_, e_ = b.path()
            dev_runs += d_
            exact_runs += e_
    h2d = 0
    for g in groups:
        h2d += g["scans"].nbytes + len(g["ids"]) * 312          # scans + per-pair query descriptors
    pairs = n_scans * n_submaps
    out = {"qps": pairs * steps / (dev_ms * 1e-3), "qps_e2e": pairs * steps / e2e_s,
           "qps_e2e_sequential": pairs * steps / e2e_seq_s,
           "ms": dev_ms / steps, "ms_e2e": 1e3 * e2e_s / steps, "launches_per_step": launches / steps,
           "sub_batches": len(groups), "scans_per_sub_batch": sub, "nodes_rank0": nodes, "gathers_rank0": gathers,
           "gathers_issued_frac_rank0": (1.0 - skipped / gathers) if gathers else None,
           "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(L[0]["ex"].d2h_bytes),
           "device_runs": dev_runs, "exact_runs": exact_runs,
           "found": int((rec["found"] != 0).sum()), "best": sharding.best_candidate(rec),
           "sha": hashlib.sha256(rec.tobytes()).hexdigest()[:16]}
    for lane in L:
        for b in lane["batches"]:
            b.close()
        lane["ex"].close()
    return out, rec


# ---- C5: large map ---------------------------------------------------------------------------------------
def run_c5(ctx, comm, rank, world_size, barrier, max_over_ranks, sum_over_ranks, side, n_queries, steps, lane_b=None):
    """C5: one side x side map (8 x 8 stitched copies of a GPU-integrated 1000 x 1000 tile), 7 pyramid levels.
    Precompute: split into world_size row bands (band + margin per GPU, largemap.py; banded == whole map
    bit for bit, tests/test_gpu_largemap.py).  Batch loop closure: SURVEY 8(e) offers "each holding the
    full pyramid" -- the whole 7-level pyramid is 3.6 GB, so every GPU builds its own copy (cheaper than
    any exchange) and the queries are split round-robin; records are exchanged like C4's."""
    from my_lidar_graph_slam_b200 import capi, largemap, sharding
    T = 1000                                            # tile side (cells) = 50 m
    world = synth.RoomsWorld(40.0, 5.0, seed=12)
    angles = synth.beam_angles(1081, 270.0)
    traj = np.concatenate([synth.trajectory(world, 10, step=0.5, seed=40 + k, start=(x, y, 0.4 * k))
                           for k, (x, y) in enumerate(((-12.5, -12.5), (2.5, -7.5), (-7.5, 7.5), (12.5, 12.5)))])
    rng = np.random.default_rng(13)
    scans = [synth.make_scan(world, p, angles, rng) for p in traj]
    hits = [capi.scan_hit_points(p, angles, r, 0.02, 20.0)[0] for p, r in zip(traj, scans)]
    tile_grid = capi.Grid(ctx, T, T, -25.0, -25.0, 0.05, apron=1)
    capi.integrate_scans(ctx, tile_grid, traj[:, :2], hits)
    tile = tile_grid.download()
    tile_grid.close()
    n_t = side // T
    ny = nx = n_t * T

    def rows_provider(a, b):                            # rows [a, b) of the stitched map
        return np.tile(tile[np.arange(a, b) % T], (1, n_t))

    # (1) precompute sharded in row bands
    band = largemap.BandedMap(ctx, rows_provider, nx, ny, -25.0, -25.0, 0.05, rank, world_size, BB["node_height_max"],
                              reach_m=BB["score_range_max"], range_y_m=BB["range_y"])
    band.build_pyramid()                                # warm-up: grows the memory pool
    band.pyramid.close()
    ctx.synchronize()
    barrier()
    ctx.timer_start()
    band.build_pyramid()
    pyr_ms = max_over_ranks(ctx.timer_stop())
    owned_cells = (band.r1 - band.r0) * nx
    band_cells = band.cells
    band.close()
    # (2) batch loop closure: full pyramid on every GPU, queries round-robin
    whole = capi.Grid(ctx, nx, ny, -25.0, -25.0, 0.05, apron=1)
    whole.upload(rows_provider(0, ny))
    ctx.synchronize()
    ctx.timer_start()
    pyr = capi.Pyramid(ctx, whole, BB["node_height_max"])
    full_ms = ctx.timer_stop()
    qr = np.random.default_rng(14)
    n_distinct = min(n_queries, 256)                    # distinct query scans; query k re-uses scan k % n_distinct
    q_scans, q_base, q_init = [], [], []                # at another place of the stitched map / another first guess
    for k in range(n_distinct):
        q_base.append(traj[int(qr.integers(0, len(traj)))])
        q_scans.append(synth.make_scan(world, q_base[-1], angles, qr))
    for k in range(n_queries):
        off = np.array([qr.integers(0, n_t) * T * 0.05, qr.integers(0, n_t) * T * 0.05, 0.0])
        q_init.append(q_base[k % n_distinct] + off + np.array([qr.uniform(-0.4, 0.4), qr.uniform(-0.4, 0.4), qr.uniform(-0.1, 0.1)]))
    mine = sharding.owned(n_queries, rank, world_size)
    # a query = (scan, first guess): the sensor pose belongs to the pair, so every query is its own scan entry
    sc = capi.Scans([angles] * len(mine), [q_scans[k % n_distinct] for k in mine], [q_init[k] for k in mine],
                    range_min=0.02, range_max=30.0)
    plist = [pyr] * len(mine)
    pair = np.arange(len(mine), dtype=np.int32)
    # end to end like C4: consecutive steps alternate between two contexts (the second one reads the same
    # pyramid), so the upload and host work of step k + 1 run under the kernel of step k
    L = []
    for ctx_l, comm_l in ([(ctx, comm)] + ([lane_b] if lane_b else [])):
        ex_l = sharding.RecordExchange(ctx_l, comm_l, n_queries, rank, world_size)
        b_l = capi.BbBatch(ctx_l, **BB)
        ex_l.attach(b_l, mine)
        L.append(dict(ctx=ctx_l, ex=ex_l, batch=b_l))
    ex, batch = L[0]["ex"], L[0]["batch"]

    def submit(lane):
        lane["batch"].upload_pairs(sc, pair, plist, 0.6)
        if world_size > 1:
            for other in L:
                if other is not lane:
                    lane["ctx"].wait_for(other["ctx"])
        lane["batch"].run()
        lane["ex"].launch_gather()

    def collect(lane):
        return lane["ex"].finish_launched([lane["batch"]])

    for lane in L:
        for _ in range(2):
            submit(lane)
            rec = collect(lane)
    for lane in L:
        lane["ctx"].synchronize()
    barrier()
    t0 = time.perf_counter()
    submit(L[0])
    for k in range(1, steps):
        submit(L[k % len(L)])
        rec = collect(L[(k - 1) % len(L)])
    rec = collect(L[(steps - 1) % len(L)])
    for lane in L:
        lane["ctx"].synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    batch.upload_pairs(sc, pair, plist, 0.6)
    ctx.synchronize()
    barrier()
    ctx.timer_start()
    for _ in range(steps):
        batch.run()
    dev_ms = max_over_ranks(ctx.timer_stop())
    peak = measured_peaks()[0] * world_size
    algo = sum_over_ranks(float(band_cells)) * 6 * 16 / (pyr_ms * 1e-3) / 1e9
    out = {"map_cells": [int(nx), int(ny)], "bands": world_size,
           "precompute_ms": pyr_ms, "precompute_cells_levels_per_s": sum_over_ranks(float(owned_cells)) * 7 / (pyr_ms * 1e-3),
           "precompute_hbm_frac": algo / peak, "full_pyramid_ms_per_gpu": full_ms,
           "queries": n_queries, "qps": n_queries * steps / (dev_ms * 1e-3), "qps_e2e": n_queries * steps / e2e_s,
           "found": int((rec["found"] != 0).sum()), "sha": hashlib.sha256(rec.tobytes()).hexdigest()[:16]}
    for lane in L:
        lane["batch"].close()
        lane["ex"].close()
    pyr.close()
    whole.close()
    return out


def run_c3(ctx, n_distinct, n_total, with_cpu):
    """C3 (bounded sample): 1081-beam scans along a trajectory integrated into one pre-sized map
    in calls of up to 1024 scans, page-locked host hit points in, cell updates applied in (scan, beam) order."""
    from my_lidar_graph_slam_b200 import capi
    world = synth.RoomsWorld(40.0, 5.0, seed=6)
    angles = synth.beam_angles(1081, 270.0)
    traj = synth.trajectory(world, n_distinct, step=0.1, seed=6)
    rng = np.random.default_rng(7)
    ranges = [synth.make_scan(world, p, angles, rng) for p in traj]
    hits = [capi.scan_hit_points(p, angles, r, 0.02, 20.0)[0] for p, r in zip(traj, ranges)]
    geo = capi.Geometry(0, 0, -20.0, -20.0, 0.05, 64)
    geo, _, _, _ = capi.geometry_expand(geo, (-20.5, -20.5, 20.5, 20.5), 0.0)
    grid = capi.Grid(ctx, geo.nx, geo.ny, geo.min_x, geo.min_y, 0.05, apron=1)
    B = int(os.environ.get("C3_BATCH", "1024"))
    batches = [capi.PackedHits(traj[k:k + B, :2], hits[k:k + B]) for k in range(0, n_distinct, B)]
    for b in batches:                                                 # page-locked host inputs
        capi.pin(ctx, b.hit, b.sxy, b.begin)
    capi.integrate_packed(ctx, grid, batches[0])                      # warm-up
    capi.grid_clear(grid)
    ctx.synchronize()
    updates, done, h2d = 0, 0, 0
    t0 = time.perf_counter()
    # streamed: call k + 1 is submitted (host-to-device copy + pre-pass on the copy stream) while the passes of
    # call k run; every call still moves its own scans to the device and its update count back
    in_flight = 0
    while done < n_total:
        for b in batches:
            capi.integrate_submit(ctx, grid, b)
            in_flight += 1
            if in_flight == 2:
                updates += capi.integrate_wait(ctx)
                in_flight -= 1
            done += b.n
            h2d += b.nbytes
    while in_flight:
        updates += capi.integrate_wait(ctx)
        in_flight -= 1
    ctx.synchronize()
    dt = time.perf_counter() - t0
    # the same stream through the synchronous call (one call after the other)
    capi.grid_clear(grid)
    ctx.synchronize()
    t0 = time.perf_counter()
    done_seq = 0
    while done_seq < min(n_total, 16 * B):
        for b in batches:
            capi.integrate_packed(ctx, grid, b)
            done_seq += b.n
    ctx.synchronize()
    dt_seq = time.perf_counter() - t0
    out = {"workload": f"C3 occupancy-grid integration: {done} scans streamed ({n_distinct} distinct 1081-beam "
                       f"scans along a trajectory, repeated; calls of {B} scans) into one {geo.nx}x{geo.ny} map",
           "scans_per_s": done / dt, "scans_per_s_sequential_calls": done_seq / dt_seq, "cell_updates_per_s": updates / dt,
           "cell_updates_per_scan": updates / done, "e2e": True,
           "h2d_bytes_per_scan": h2d / done,
           "algorithmic_GBps": updates * 16 / dt / 1e9}
    peak, peak_src = measured_peaks()
    out["roofline"] = {"bound": "hbm", "achieved": out["algorithmic_GBps"], "peak": peak, "unit": "GB/s",
                       "frac": out["algorithmic_GBps"] / peak, "peak_source": peak_src,
                       "algorithmic_bytes": "16 B per cell update (read-modify-write of one double)",
                       "note": "end to end incl. H2D; the binding limits are the order-dependent per-cell update "
                               "chain (two IEEE double divisions, 283 cycles) and instruction issue of the touch "
                               "pass, not HBM: DESIGN.md 3.4, profiles/r1_kernels_v3.md"}
    if with_cpu:
        try:
            from oracle import refapi as R
            if R.available():
                m = R.RefMap.from_dense(np.zeros((geo.ny, geo.nx)), geo.min_x, geo.min_y)
                ns = min(n_distinct, 256)
                t0 = time.perf_counter()
                for k in range(ns):
                    R.map_integrate_hits(m, traj[k, :2], hits[k])
                dtc = time.perf_counter() - t0
                capi.grid_clear(grid)
                capi.integrate_scans(ctx, grid, traj[:ns, :2], hits[:ns])
                same = bool(np.array_equal(grid.download().view(np.int64), m.dense().view(np.int64)))
                out["cpu_baseline"] = {"value": ns / dtc, "unit": "scans/s", "cores": 1, "kind": "reference",
                                       "sample": f"{ns} scans through the reference integration loop on 1 thread "
                                                 f"({dtc:.1f} s; order-dependent, single map); GPU map bit-identical: {same}"}
        except Exception as e:
            out["cpu_baseline"] = {"value": None, "sample": f"failed: {e}"}
    for b in batches:
        capi.unpin(ctx, b.hit, b.sxy, b.begin)
    grid.close()
    return out


def run_tail(ctx, grid, dense, min_x, min_y, angles, ranges, inits, results, with_cpu):
    """SURVEY 8(f) rank 2: the tail both matchers run on the winning pose (CostGreedyEndpoint cost +
    finite-difference covariance = 7 cost evaluations per match), through the C ABI with host buffers."""
    from my_lidar_graph_slam_b200 import capi
    M = len(results)
    best = np.array([[inits[k][0] + r.ix * r.step_x, inits[k][1] + r.iy * r.step_y, inits[k][2] + r.it * r.step_t]
                     for k, r in enumerate(results)])
    scans = capi.Scans([angles] * M, ranges, inits, range_min=0.02, range_max=30.0)
    capi.pin(ctx, scans.angles, scans.ranges)
    capi.cost_tail(ctx, grid, scans, best)
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        nc, cov, fix = capi.cost_tail(ctx, grid, scans, best)
    dt = (time.perf_counter() - t0) / reps
    capi.unpin(ctx, scans.angles, scans.ranges)
    out = {"tails_per_s": M / dt, "ms_per_call": 1e3 * dt, "matches_per_call": M,
           "cost_evaluations_per_s": 7 * M / dt, "host_fixups": int(fix),
           "note": "lgs_cost_tail end to end (host scans in, normalised cost + 3x3 covariance out), "
                   "one launch of cost_kernel per call; bit-identical to CostGreedyEndpoint"}
    if with_cpu:
        try:
            from oracle import refapi as R
            if R.available():
                rm = R.RefMap.from_dense(dense, min_x, min_y)
                ns = min(M, 32)
                t0 = time.perf_counter()
                ref = [R.host_tail(rm, best[k], angles, ranges[k]) for k in range(ns)]
                cdt = (time.perf_counter() - t0) / ns
                same = sum(ref[k][0] == nc[k] and np.array_equal(ref[k][2], cov[k]) for k in range(ns))
                out["cpu_reference"] = {"tails_per_s": 1.0 / cdt, "cores": 1, "kind": "reference",
                                        "sample": f"{ns} tails; identical to the device on {same}/{ns}"}
        except Exception as e:                                   # noqa: BLE001
            out["cpu_reference"] = {"error": str(e)}
    return out


def run_gs(ctx, grid, dense, min_x, min_y, angles, ranges, inits, with_cpu, n_queries=64):
    """SURVEY 8(f) rank 3: the exhaustive grid-search matcher behind LoopDetectorGridSearch at the
    launcher's defaults (2 m x 2 m at 0.05 m, 0.5 rad at 0.005 rad: ~1.7e5 hypotheses per query)."""
    from my_lidar_graph_slam_b200 import capi
    Q = min(n_queries, len(ranges))
    scans = capi.Scans([angles] * Q, ranges[:Q], inits[:Q], range_min=0.02, range_max=30.0)
    capi.pin(ctx, scans.angles, scans.ranges)
    out = capi.gs_match(ctx, scans, [grid] * Q)
    reps = 3
    t0 = time.perf_counter()
    for _ in range(reps):
        out = capi.gs_match(ctx, scans, [grid] * Q)
    dt = (time.perf_counter() - t0) / reps
    capi.unpin(ctx, scans.angles, scans.ranges)
    hyp = sum(r.n_scored for r in out)
    res = {"queries_per_s": Q / dt, "hypotheses_per_s": hyp / dt, "ms_per_call": 1e3 * dt, "queries_per_call": Q,
           "hypotheses_per_query": hyp // Q, "found": int(sum(r.found for r in out)),
           "host_fixups": int(sum(r.n_fixups for r in out)),
           "note": "lgs_gs_match end to end (host scans in, result records out); kernels: gs_project, gs_score, "
                   "gs_select"}
    if with_cpu:
        try:
            from oracle import refapi as R
            if R.available():
                rm = R.RefMap.from_dense(dense, min_x, min_y)
                small = dict(range_x=0.5, range_y=0.5, range_theta=0.05, step_x=0.05, step_y=0.05, step_theta=0.005)
                t0 = time.perf_counter()
                ref = R.gs_match(rm, angles, ranges[0], inits[0], **small)
                cdt = time.perf_counter() - t0
                one = capi.Scans([angles], [ranges[0]], [inits[0]], range_min=0.02, range_max=30.0)
                (g,) = capi.gs_match(ctx, one, [grid], **small)
                same = (g.found, g.ix, g.iy, g.it, g.win_x, g.win_y, g.win_t) == \
                    (ref.found, ref.ix, ref.iy, ref.it, ref.winX, ref.winY, ref.winT) and \
                    (not g.found or g.score == ref.score)
                n = ref.winX * ref.winY * ref.winT
                res["cpu_reference"] = {"hypotheses_per_s": n / cdt, "cores": 1, "kind": "reference",
                                        "sample": f"one query on a reduced window ({n} hypotheses, {cdt:.1f} s); "
                                                  f"device winner and score identical: {bool(same)}"}
        except Exception as e:                                   # noqa: BLE001
            res["cpu_reference"] = {"error": str(e)}
    return res

# ---- C2: the real-time correlative sweep -----------------------------------------------------------------
def measure_c2(ctx, ctx_index, args, barrier, max_over_ranks, sum_over_ranks, with_clock_sampler):
    """One rank's C2 measurement (every rank the same batch against its own copy of the map)."""
    from my_lidar_graph_slam_b200 import capi
    M = args.matches
    traj, map_scans, angles, ranges, inits = c2_workload(M, seed=1)
    grid, _ = build_map_on_gpu(ctx, traj, angles, map_scans, apron=32)
    dense, min_x, min_y = grid.download(), grid.min_x, grid.min_y
    coarse = grid.like()
    scans = capi.Scans([angles] * M, ranges, inits)
    batch = capi.RtcsmBatch(ctx, **C2)
    lib = capi.lib()

    def step_device():
        ctx.check(lib.lgs_precompute(ctx.h, grid.h, 5, coarse.h))
        batch.run(grid, coarse)

    # host inputs of the end-to-end path are page-locked (lgs_host_pin), as the bench contract asks
    capi.pin(ctx, dense, scans.angles, scans.ranges, scans.sensor_pose)

    def step_e2e():
        grid.upload(dense)
        ctx.check(lib.lgs_precompute(ctx.h, grid.h, 5, coarse.h))
        batch.upload(grid, scans)
        batch.run(grid, coarse)
        return batch.results(grid, coarse)

    batch.upload(grid, scans)
    hyp, gathers = batch.work()
    for _ in range(max(args.warmup, 3)):
        step_device()
    ctx.synchronize()
    sampler = ClockSampler(ctx_index) if with_clock_sampler else None
    if sampler:
        sampler.start()
    barrier()
    launches0 = ctx.launch_count()
    ctx.timer_start()
    for _ in range(args.steps):
        step_device()
    ms = ctx.timer_stop()
    launches = ctx.launch_count() - launches0
    barrier()
    clocks = sampler.stop() if sampler else None
    ms = max_over_ranks(ms)
    # what the last timed step computed (--dump-outputs): the match records and the coarse map
    last = (batch.results(grid, coarse), coarse.download()) if args.dump_outputs else None
    total_hyp = sum_over_ranks(float(hyp)) * args.steps
    # per-kernel timing for the roofline (sweep kernel), CUDA events on the context stream
    sweep_ms = []
    for _ in range(max(3, min(args.steps, 10))):
        ctx.check(lib.lgs_precompute(ctx.h, grid.h, 5, coarse.h))
        sweep_ms.append(batch.run_timed(grid, coarse))
    k_proj, k_sweep, k_sel = (statistics.mean(x[i] for x in sweep_ms) for i in range(3))
    gnx, gny = int(dense.shape[1]), int(dense.shape[0])
    gather_peak = {"rows32_aligned_l1": capi.measure_gather_peak(ctx, gnx, gny, 32, True, True),
                   "rows25_unaligned_l1": capi.measure_gather_peak(ctx, gnx, gny, 25, False, True),
                   "rows25_unaligned_l2": capi.measure_gather_peak(ctx, gnx, gny, 25, False, False)}
    results_dev = batch.results(grid, coarse)
    # end to end, (a) strictly sequential: upload -> kernels -> results, one step after the other
    for _ in range(2):
        step_e2e()
    ctx.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res_e2e = step_e2e()
    ctx.synchronize()
    e2e_seq_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    # (b) the way a caller with a stream of match batches uses the API: two contexts (= two CUDA streams),
    # each with its own grid / batch object; step k + 1 is uploaded while step k's kernels run, and every
    # step still moves its own inputs to the device and its own result records back.
    ctx2 = capi.Context(ctx_index)
    grid2 = capi.Grid(ctx2, grid.nx, grid.ny, grid.min_x, grid.min_y, grid.res, apron=32)
    coarse2 = grid2.like()
    batch2 = capi.RtcsmBatch(ctx2, **C2)
    lanes = [(ctx, grid, coarse, batch), (ctx2, grid2, coarse2, batch2)]

    def submit(lane):
        c, g, cg, b = lane
        g.upload(dense)
        c.check(lib.lgs_precompute(c.h, g.h, 5, cg.h))
        b.upload(g, scans)
        b.run(g, cg)

    def collect(lane):
        return lane[3].results(lane[1], lane[2])

    for k in range(2):
        submit(lanes[k]); collect(lanes[k])
    ctx.synchronize(); ctx2.synchronize()
    barrier()
    t0 = time.perf_counter()
    submit(lanes[0])
    for k in range(1, args.steps):
        submit(lanes[k % 2])
        res_e2e = collect(lanes[(k - 1) % 2])
    res_e2e = collect(lanes[(args.steps - 1) % 2])
    ctx.synchronize(); ctx2.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    assert all((a.found, a.ix, a.iy, a.it, a.score) == (b.found, b.ix, b.iy, b.it, b.score)
               for a, b in zip(results_dev, res_e2e))
    batch2.close(); coarse2.close(); grid2.close(); ctx2.close()
    capi.unpin(ctx, dense, scans.angles, scans.ranges, scans.sensor_pose)
    return dict(value=total_hyp / (ms * 1e-3), ms_per_step=ms / args.steps, launches=int(launches), clocks=clocks,
                hyp=int(hyp), gathers=int(gathers), k_proj=k_proj, k_sweep=k_sweep, k_sel=k_sel,
                gather_peak=gather_peak, e2e=total_hyp / e2e_s, e2e_seq=total_hyp / e2e_seq_s,
                e2e_ms=1e3 * e2e_s / args.steps, h2d=int(dense.nbytes + scans.nbytes + M * 96), d2h=int(M * 32 + 4),
                grid=grid, coarse=coarse, batch=batch, dense=dense, min_x=min_x, min_y=min_y, angles=angles,
                ranges=ranges, inits=inits, results=results_dev, last=last)


def gather_roofline(achieved_gbps, gather_peak_gbps, sm_mhz, n_gpus, kernel, hbm_peak):
    """The `roofline` object of a scoring kernel: bound = the L1 gather path (maps are cache resident)."""
    theo = 148 * 128 * (sm_mhz or 1965.0) * 1e6 / 1e9 * n_gpus       # 148 SMs x 128 B/clk x f_sm
    peak = gather_peak_gbps * n_gpus
    return {"bound": "l1_gather", "achieved": r3(achieved_gbps), "peak": r3(peak), "unit": "GB/s",
            "frac": r3(achieved_gbps / peak), "peak_kind": "measured in-run gather peak",
            "peak_theoretical": r3(theo), "frac_theoretical": r3(achieved_gbps / theo), "kernel": kernel,
            "hbm_peak": r3(hbm_peak * n_gpus), "hbm_frac": r3(achieved_gbps / (hbm_peak * n_gpus)), "traffic": None}


# ---- reference arm ------------------------------------------------------------------------------------------
def run_reference(args, rank, world_size):
    """The UNMODIFIED reference classes on the box's host cores, same metric / unit / config as the GPU arm
    of the same N: the correlative matcher (C2) at N = 1, the branch-and-bound matcher (C4) at N > 1."""
    if rank != 0:
        return
    from concurrent.futures import ThreadPoolExecutor

    from oracle import refapi as R
    cores = os.cpu_count() or 1
    if not R.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/liblgs_ref.so not built"}))
        return
    if world_size == 1 and args.gpus <= 1:
        M = args.matches
        per_step = min(M, max(16 * cores, 64))      # bounded sample of every step: enough to keep every thread busy
        total = per_step * (args.steps + args.warmup)
        traj, map_scans, angles, ranges, inits = c2_workload(max(total, M), seed=1)
        builder = R.RefBuilder(n_latest=len(traj))
        for p, r in zip(traj, map_scans):
            builder.append_scan(p, angles, r)
        refmap = builder.local_map(0)
        dense = refmap.dense()
        _, _, min_x, min_y, _ = refmap.geometry()
        times, hyps = [], 0
        for s in range(args.steps + args.warmup):
            sl = slice(s * per_step, (s + 1) * per_step)
            dt, res = ref_time_matches(dense, min_x, min_y, angles, ranges[sl], inits[sl], cores)
            if s >= args.warmup:
                times.append(dt)
                hyps += sum(hyps_per_match(r) for r in res)
        total_t = sum(times)
        value = hyps / total_t
        sample = (f"{per_step} of the {M} C2 matches of a step, {args.steps} steps, {cores} threads; hypotheses = "
                  "full window per match (the CPU prunes inside it)")
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_t / args.steps * (M / per_step),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": c2_config(M),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    # N > 1: branch-and-bound loop detection (C4).  Sample: one query scan against the first submaps.
    scene = c4_scene()
    world, angles, anchor, qscans, qinits = scene
    n_maps = max(cores, 16)
    maps = []
    for g in range(n_maps):
        traj, scans = c4_submap_scans(world, angles, g, 8, anchor)
        b = R.RefBuilder(n_latest=len(traj))
        for p, r in zip(traj, scans):
            b.append_scan(p, angles, r)
        m = b.local_map(0)
        maps.append((m, m.pyramid(6)))

    def one(job):
        k, g = job
        return R.bb_match(maps[g][0], angles, qscans[k], qinits[k], pyramid=maps[g][1], thr=0.6)

    times, n_done = [], 0
    for s in range(args.steps + args.warmup):
        jobs = [((s + j // n_maps) % C4_SCANS, j % n_maps) for j in range(n_maps)]
        t0 = time.perf_counter()
        with ThreadPoolExecutor(max_workers=cores) as ex:
            list(ex.map(one, jobs))
        dt = time.perf_counter() - t0
        if s >= args.warmup:
            times.append(dt)
            n_done += len(jobs)
    total_t = sum(times)
    value = n_done / total_t
    pairs = C4_SCANS * args.submaps
    sample = (f"{n_maps} (scan, submap) pairs per step (first {n_maps} submaps, pyramids prebuilt) on {cores} threads, "
              f"{args.steps} steps; a full step is {pairs} pairs")
    print(json.dumps({
        "impl": "reference", "metric": C4_METRIC, "value": value, "unit": C4_UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * pairs / value,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": c4_config(args.submaps, args.gpus),
        "cpu_baseline": {"value": value, "unit": C4_UNIT, "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": C4_UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def write_details(d, n, details):
    if not d:
        return
    try:
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, f"bench_details_n{n}.json"), "w") as f:
            json.dump(details, f, indent=1, default=lambda o: float(o) if isinstance(o, np.floating) else str(o))
    except OSError:
        pass


DUMP_BUDGET = 60 * 10**6                             # bytes of array data: under 64 MB with the .npy headers


def dump_outputs(d, arrays):
    """Write each array as d/<name>.npy in float64.  When the set would exceed DUMP_BUDGET, an array larger than
    its share keeps a fixed, seeded sample of its rows (ascending; their indices go to <name>_rows.npy),
    so that two builds given the same arguments still compare value for value."""
    os.makedirs(d, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    over = sum(a.nbytes for a in arrays.values()) > DUMP_BUDGET
    share = DUMP_BUDGET // max(len(arrays), 1)
    for name, a in arrays.items():
        if over and a.nbytes > share:
            row_bytes = a.nbytes // len(a) + 8                   # + the float64 row index
            rows = np.sort(np.random.default_rng(0).choice(len(a), share // row_bytes, replace=False))
            a = a[rows]
            np.save(os.path.join(d, f"{name}_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(d, f"{name}.npy"), a)


def r3(x, digits=3):
    """3 significant digits (the one-line contract must stay short)."""
    return None if x is None else float(f"{float(x):.{digits}g}")


def run_b200(args, rank, world_size, local_rank):
    from my_lidar_graph_slam_b200 import capi, sharding
    dist = None
    if world_size > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()

    def reduce_(x, op):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=op)
        return float(t.item())

    def max_over_ranks(x):
        return reduce_(x, dist.ReduceOp.MAX) if dist is not None else x

    def sum_over_ranks(x):
        return reduce_(x, dist.ReduceOp.SUM) if dist is not None else x

    # C1 runs in child processes (the adapters' own executables): first, while this process holds no CUDA
    # context yet -- beside the bench's resident contexts the same loop measured 1.3 instead of 0.37 ms per frame
    c1_early = None
    if world_size == 1 and not args.no_extra:
        try:
            c1_early = run_c1()
        except Exception as e:                                   # noqa: BLE001
            c1_early = {"error": f"{type(e).__name__}: {e}"}

    ctx = capi.Context(local_rank)
    comm = sharding.make_comm(ctx, rank, world_size)
    ctx_b = capi.Context(local_rank)                    # second lane of the pipelined end-to-end steps
    comm_b = sharding.make_comm(ctx_b, rank, world_size)
    lanes = [(ctx, comm), (ctx_b, comm_b)]
    hbm_peak, hbm_src = measured_peaks()
    details = {"n_gpus": world_size}
    steps_side = max(3, min(args.steps, 10))
    # timed steps of the 64-scan loop-detection batch: the headline at N > 1 times exactly --steps of them
    c4_nsteps = args.steps if world_size > 1 else max(4, steps_side)

    # ---- C2 (headline at N = 1, `extra.c2_replicas` at N > 1) ------------------------------------------------
    c2 = measure_c2(ctx, local_rank, args, barrier, max_over_ranks, sum_over_ranks, rank == 0)
    sm_mhz = (c2["clocks"] or {}).get("sm_mhz") if rank == 0 else None
    gpeak = c2["gather_peak"]["rows32_aligned_l1"]
    c2_achieved = c2["gathers"] * 8 / (c2["k_sweep"] * 1e-3) / 1e9

    # ---- C4 loop closure: this rank's shard of the 500 submaps ---------------------------------------------------
    c4 = None
    if not args.no_c4:
        scene = c4_scene()
        mine = sharding.owned(args.submaps, rank, world_size)
        t0 = time.perf_counter()
        shard = C4Shard(ctx, scene, mine)
        build_s = time.perf_counter() - t0
        placement, balance = None, None
        if world_size > 1 and os.environ.get("LGS_C4_PLACEMENT", "lpt") != "rr":
            # cost-aware placement: the nodes scored against every submap in one plain step under round-robin
            # placement (all-reduced), spread over the ranks longest-first; the submaps that changed owner are
            # rebuilt there.  A few submaps (the true loop candidates) carry half of the work.
            import torch
            deep, terms = shard.submap_cost_terms(args.submaps)
            wt = torch.from_numpy(np.concatenate([deep, terms])).to(f"cuda:{local_rank}")
            dist.all_reduce(wt)
            wt = wt.cpu().numpy()
            deep, terms = wt[:args.submaps], wt[args.submaps:]
            us_root = terms[0] / max(terms[1], 1.0)               # us per root node, us per deeper node
            us_deep = terms[2] / max(terms[3], 1.0)
            weights = us_root * (terms[1] / args.submaps) + us_deep * np.maximum(deep, 0.0)
            placement = sharding.balanced_placement(weights, world_size)
            rr = [float(weights[sharding.owned(args.submaps, r, world_size)].sum()) for r in range(world_size)]
            lp = [float(weights[p].sum()) for p in placement]
            balance = {"round_robin_max_over_mean": max(rr) / (sum(rr) / world_size),
                       "lpt_max_over_mean": max(lp) / (sum(lp) / world_size),
                       "ns_per_root_node": 1e3 * us_root, "ns_per_deeper_node": 1e3 * us_deep}
            mine = placement[rank]
            shard = C4Shard(ctx, scene, mine, reuse=shard.release_grids())
        single, rec1 = c4_steps(lanes, shard, rank, world_size, args.submaps, 1, steps_side, barrier, max_over_ranks,
                                placement=placement, details=args.details)
        batched, recq = c4_steps(lanes, shard, rank, world_size, args.submaps, C4_SCANS, c4_nsteps,
                                 barrier, max_over_ranks, placement=placement, details=args.details)
        c4 = {"single": single, "batched": batched, "submaps_rank0": int(len(mine)), "placement": balance,
              "pyramid_rebuild_ms_rank0": shard.pyramid_ms, "submap_build_s_rank0": build_s,
              "pyramid_cells_levels_per_s_rank0": shard.cells * 7 / (shard.pyramid_ms * 1e-3) if shard.pyramid_ms > 0 else None}
        c4["gathers_all"] = sum_over_ranks(float(batched["gathers_rank0"]))
        shard.close()
        # the same steps with ALL submaps on rank 0's GPU alone: the strong-scaling reference of this very run
        if world_size > 1:
            n1 = None
            if rank == 0:
                full = C4Shard(ctx, scene, np.arange(args.submaps))
                nb = lambda: None
                solo = [(ctx, None), (ctx_b, None)]
                s1, r1 = c4_steps(solo, full, 0, 1, args.submaps, 1, steps_side, nb, lambda x: x, details=args.details)
                sq, rq = c4_steps(solo, full, 0, 1, args.submaps, C4_SCANS, c4_nsteps, nb, lambda x: x,
                                  details=args.details)
                full.close()
                n1 = {"single": s1, "batched": sq,
                      "records_identical": bool(r1.tobytes() == rec1.tobytes() and rq.tobytes() == recq.tobytes())}
            barrier()
            c4["n1_same_run"] = n1
        # CPU reference on a bounded sample, parity-checked (N = 1 only)
        if world_size == 1 and not args.no_cpu_baseline:
            try:
                from concurrent.futures import ThreadPoolExecutor

                from oracle import refapi as R
                if R.available():
                    cores = os.cpu_count() or 1
                    ns = max(cores, 16)
                    world, angles, anchor, qscans, qinits = scene
                    maps = []
                    for g in range(ns):
                        traj, scans = c4_submap_scans(world, angles, g, 8, anchor)
                        b = R.RefBuilder(n_latest=len(traj))
                        for p, r in zip(traj, scans):
                            b.append_scan(p, angles, r)
                        m = b.local_map(0)
                        maps.append((m, m.pyramid(6)))
                    t0 = time.perf_counter()
                    with ThreadPoolExecutor(max_workers=cores) as ex:
                        ref = list(ex.map(lambda g: R.bb_match(maps[g][0], angles, qscans[0], qinits[0],
                                                               pyramid=maps[g][1], thr=0.6), range(ns)))
                    dt = time.perf_counter() - t0
                    bad = sum((a.found, a.ix, a.iy, a.it) != (int(b["found"]), int(b["ix"]), int(b["iy"]), int(b["it"]))
                              or (a.found and a.score != float(b["score"])) for a, b in zip(ref, rec1[:ns]))
                    c4["cpu_baseline"] = {"value": ns / dt, "unit": C4_UNIT, "cores": cores, "kind": "reference",
                                          "sample": f"first {ns} submaps x 1 scan on {cores} threads ({dt:.1f} s), pyramids "
                                                    f"prebuilt; GPU records identical on {ns - bad}/{ns}"}
            except Exception as e:                                   # noqa: BLE001
                c4["cpu_baseline"] = {"value": None, "sample": f"failed: {e}"}
    details["c4"] = c4

    # ---- side measurements ---------------------------------------------------------------------------------------
    extra = {}

    def side(name, fn):
        """A side measurement must never take the headline line down with it (single process only: with
        several ranks a failure has to propagate, or the other ranks wait in a collective)."""
        if world_size > 1:
            details[name] = fn()
            return
        try:
            details[name] = fn()
        except Exception as e:                                   # noqa: BLE001
            details[name] = {"error": f"{type(e).__name__}: {e}"}

    if not args.no_extra:
        if args.c5_side > 0:
            side("c5", lambda: run_c5(ctx, comm, rank, world_size, barrier, max_over_ranks, sum_over_ranks,
                                      args.c5_side, args.c5_queries, max(4, min(args.steps, 10)), lane_b=(ctx_b, comm_b)))
        if rank == 0 and world_size == 1:
            cpu_side = not args.no_cpu_baseline
            side("matcher_tail", lambda: run_tail(ctx, c2["grid"], c2["dense"], c2["min_x"], c2["min_y"], c2["angles"],
                                                  c2["ranges"], c2["inits"], c2["results"], cpu_side))
            side("grid_search", lambda: run_gs(ctx, c2["grid"], c2["dense"], c2["min_x"], c2["min_y"], c2["angles"],
                                               c2["ranges"], c2["inits"], cpu_side))
            side("c3", lambda: run_c3(ctx, 1024, args.c3_scans, cpu_side))
            details["c1"] = c1_early
    if rank != 0:
        return

    # ---- CPU baseline of the headline: the unmodified reference on a bounded sample, parity-checked -----------------
    cpu = None
    if world_size == 1 and not args.no_cpu_baseline:
        try:
            from oracle import refapi as R
            if R.available():
                cores = os.cpu_count() or 1
                ns = min(args.matches, max(16 * cores, 64))
                dt, ref = ref_time_matches(c2["dense"], c2["min_x"], c2["min_y"], c2["angles"], c2["ranges"][:ns],
                                           c2["inits"][:ns], cores)
                bad = sum((a.found, a.ix, a.iy, a.it, a.score) != (b.found, b.ix, b.iy, b.it, b.score)
                          for a, b in zip(ref, c2["results"][:ns]))
                cpu = {"value": r3(sum(hyps_per_match(r) for r in ref) / dt), "unit": UNIT, "cores": cores,
                       "kind": "reference", "sample": f"first {ns} matches, {dt:.1f} s; GPU identical {ns - bad}/{ns}"}
        except Exception as e:   # the baseline is reported, never required
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {e}"}

    c2_block = {"value": r3(c2["value"]), "e2e": r3(c2["e2e"]), "e2e_sequential": r3(c2["e2e_seq"]),
                "ms_per_step": r3(c2["ms_per_step"]), "sweep_ms": r3(c2["k_sweep"])}
    details["c2"] = {k: v for k, v in c2.items() if k not in ("grid", "coarse", "batch", "dense", "angles", "ranges",
                                                              "inits", "results", "last")}
    short = {"precompute_ms": "pre_ms", "precompute_hbm_frac": "pre_hbm_frac", "qps": "qps", "qps_e2e": "qps_e2e",
             "found": "found", "scans_per_s": "scans_per_s", "cell_updates_per_s": "updates_per_s",
             "tails_per_s": "per_s", "hypotheses_per_s": "hyp_per_s", "frames_per_s": "fps", "ref_frames_per_s": "ref_fps",
             "identical": "same", "launcher_frames_per_s": "launch_fps", "launcher_ref_frames_per_s": "launch_ref_fps",
             "launcher_identical": "launch_same"}
    for name, out_name, keys in (("c5", "c5", ("precompute_ms", "precompute_hbm_frac", "qps", "qps_e2e", "found")),
                                 ("c3", "c3", ("scans_per_s", "cell_updates_per_s")), ("matcher_tail", "tail", ("tails_per_s",)),
                                 ("grid_search", "gs", ("hypotheses_per_s",)),
                                 ("c1", "c1", ("frames_per_s", "ref_frames_per_s", "identical", "launcher_frames_per_s",
                                               "launcher_ref_frames_per_s", "launcher_identical"))):
        d = details.get(name)
        if isinstance(d, dict):
            extra[out_name] = {short[k]: (r3(d[k]) if isinstance(d.get(k), float) else d.get(k)) for k in keys if k in d} \
                if "error" not in d else {"error": d["error"][:60]}

    def c4_compact(c):
        return {"q1": {"k": r3(c["single"]["qps"]), "e2e": r3(c["single"]["qps_e2e"]),
                       "e2e_seq": r3(c["single"]["qps_e2e_sequential"]), "ms": r3(c["single"]["ms"])},
                "q64": {"k": r3(c["batched"]["qps"]), "e2e": r3(c["batched"]["qps_e2e"]),
                        "e2e_seq": r3(c["batched"]["qps_e2e_sequential"]), "ms": r3(c["batched"]["ms"])}}

    if world_size == 1:
        line = {
            "metric": METRIC, "value": r3(c2["value"], 6), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": r3(c2["ms_per_step"], 6), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": c2_config(args.matches),
            "l2": "working set > L2",
            "e2e": {"value": r3(c2["e2e"], 6), "unit": UNIT, "h2d_bytes_per_step": c2["h2d"], "d2h_bytes_per_step": c2["d2h"],
                    "sequential_value": r3(c2["e2e_seq"])},
            "gpu_launches": c2["launches"], "clocks": c2["clocks"],
            "roofline": gather_roofline(c2_achieved, gpeak, sm_mhz, 1, "csm_sweep_rows_kernel<4,5>", hbm_peak),
            "cpu_baseline": cpu,
        }
        if c4:
            line["loop_closure"] = {"unit": C4_UNIT, **c4_compact(c4),
                                    "roof_frac": r3(c4["gathers_all"] * 8 / (c4["batched"]["ms"] * 1e-3) / 1e9 / gpeak),
                                    "sha": c4["batched"]["sha"], "found": c4["batched"]["found"],
                                    "cpu": r3((c4.get("cpu_baseline") or {}).get("value"))}
        line["extra"] = extra
    else:
        b = c4["batched"]
        line = {
            "metric": C4_METRIC, "value": r3(b["qps"], 6), "unit": C4_UNIT, "n_gpus": world_size, "steps": c4_nsteps,
            "warmup": 3, "ms_per_step": r3(b["ms"], 6), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": c4_config(args.submaps, world_size),
            "l2": "pyramids >> L2",
            "parallelism": ("submaps on ranks by measured cost (LPT), " if c4.get("placement") else f"submap i on rank i%{world_size}, ") +
                           "in-place NCCL all-gather",
            "placement": ({k: r3(v) for k, v in c4["placement"].items()} if c4.get("placement") else None),
            "e2e": {"value": r3(b["qps_e2e"], 6), "unit": C4_UNIT, "h2d_bytes_per_step": b["h2d_bytes_per_step"],
                    "d2h_bytes_per_step": b["d2h_bytes_per_step"], "sequential_value": r3(b["qps_e2e_sequential"])},
            "single_scan": {"value": r3(c4["single"]["qps"]), "e2e": r3(c4["single"]["qps_e2e"]),
                            "e2e_seq": r3(c4["single"]["qps_e2e_sequential"]), "ms": r3(c4["single"]["ms"])},
            "records_sha256": b["sha"], "loops_found": b["found"],
            "gpu_launches": int(round(b["launches_per_step"] * c4_nsteps)), "clocks": c2["clocks"],
            "roofline": gather_roofline(c4["gathers_all"] * 8 / (b["ms"] * 1e-3) / 1e9, gpeak, sm_mhz, world_size,
                                        "bb_run_kernel<16,2>", hbm_peak),
            "cpu_baseline": None,
        }
        if c4.get("n1_same_run"):
            n1 = c4["n1_same_run"]
            line["n1_same_run"] = {**c4_compact(n1), "records_identical": n1["records_identical"]}
        extra["c2_replicas"] = c2_block
        line["extra"] = extra
    write_details(args.details, world_size, details)
    if args.dump_outputs:
        res, coarse = c2["last"]
        out = {"c2_" + f: np.array([getattr(r, f) for r in res]) for f in ("found", "ix", "iy", "it", "score")}
        out["c2_window"] = np.array([(r.win_x, r.win_y, r.win_t) for r in res])
        out["c2_step"] = np.array([(r.step_x, r.step_y, r.step_t) for r in res])
        out["c2_coarse_map"] = coarse
        if c4:                              # records of the last end-to-end step, in pair order
            out.update({"c4_" + f: recq[f] for f in ("found", "ix", "iy", "it", "score")})
        dump_outputs(args.dump_outputs, out)
    print(json.dumps(line))


def run_c1():
    """C1 (BASELINE configs[0]): default launcher settings on a synthetic 180-beam log.
    (1) adapters/test_adapters --c1-json: the front end's frame loop (correlative match + map update per
        frame) through the C++ adapters beside the reference's own classes: frames/s of both, and whether
        every pose and every map came out identical although the poses feed back into the maps;
    (2) adapters/_build/lgs_slam_launch: the same configuration from a CARMEN log file and
        launcher_settings_default.json through the reference's own reader, LidarGraphSlam, front end and
        back end -- once with the unchanged settings (CPU matcher and loop detector), once with the B200
        type strings; the written pose graphs must be the same."""
    import tempfile
    out = {}
    exe = os.path.join(ROOT, "adapters", "_build", "test_adapters")
    if not os.path.exists(exe):
        return {"error": "adapters/_build/test_adapters not built (needs the reference tree at build time)"}
    # two to four runs, the fastest one counts (the first processes on a fresh box measured anything from 0.37 to
    # 13 ms per frame, all of it in the waits of the integration calls; alone on a settled box the loop takes
    # 0.37-0.39 ms per frame every time); every run has to be identical to the reference
    runs = []
    for _ in range(4):
        p = subprocess.run([exe, "--c1-json"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
        if p.returncode != 0:
            return {"error": f"test_adapters --c1-json exit {p.returncode}: {p.stdout[-200:]} {p.stderr[-200:]}"}
        runs.append(json.loads(p.stdout.strip().splitlines()[-1]))
        if len(runs) >= 2 and runs[-1]["frames_per_s"] >= 1500.0:
            break                                  # a settled box: ~0.4 ms per frame
    best = max(runs, key=lambda r: r["frames_per_s"])
    best["identical"] = all(r["identical"] for r in runs)
    best["frames_per_s_runs"] = [r["frames_per_s"] for r in runs]
    out.update(best)
    launch = os.path.join(ROOT, "adapters", "_build", "lgs_slam_launch")
    settings = os.path.join(ROOT, "tests", "golden", "launcher_settings_default.json")
    if os.path.exists(launch):
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import make_carmen_log
        with tempfile.TemporaryDirectory() as tmp:
            log = os.path.join(tmp, "c1.log")
            make_carmen_log.write_log(log, 600, 5)
            runs = {}
            for name, sets in (("cpu", []), ("b200", ["Frontend.LocalSlam.ScanMatcherType=RealTimeCorrelativeCuda",
                                                      "Backend.LoopDetectorType=BranchBoundCuda"])):
                cmd = [launch, log, settings, os.path.join(tmp, name), "--set", "Backend.PoseGraphOptimizerType=None"]
                for kv in sets:
                    cmd += ["--set", kv]
                q = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
                if q.returncode != 0:
                    out["launcher_error"] = f"{name}: exit {q.returncode}: {q.stderr[-200:]}"
                    return out
                runs[name] = json.loads(q.stdout.strip().splitlines()[-1])
            same = all(open(os.path.join(tmp, "cpu" + ext)).read() == open(os.path.join(tmp, "b200" + ext)).read()
                       for ext in (".poses.txt", ".edges.txt"))
            out["launcher"] = {"frames": runs["b200"]["frames"], "loop_edges": runs["b200"]["loop_edges"],
                               "frames_per_s": runs["b200"]["frames_per_s"], "ref_frames_per_s": runs["cpu"]["frames_per_s"],
                               "pose_graph_identical": bool(same)}
            out["launcher_frames_per_s"] = runs["b200"]["frames_per_s"]
            out["launcher_ref_frames_per_s"] = runs["cpu"]["frames_per_s"]
            out["launcher_identical"] = bool(same)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline (C2 at N = 1, C4 at N > 1); side measurements take 3-10")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--matches", type=int, default=1000, help="C2: matches per step (1000)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the C3 / C5 / C1 / tail / grid-search side measurements")
    ap.add_argument("--no-c4", action="store_true", help="skip the loop-closure measurement (N = 1 only)")
    ap.add_argument("--submaps", type=int, default=500, help="C4: submaps")
    ap.add_argument("--c5-side", type=int, default=8000, help="C5: map side in cells (multiple of 1000; 0 = skip)")
    ap.add_argument("--c5-queries", type=int, default=1024, help="C5: loop queries per batch")
    ap.add_argument("--c3-scans", type=int, default=102400, help="C3: scans streamed (BASELINE config: 100k)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float64, at most 64 MB)")
    ap.add_argument("--details", metavar="DIR", help="write the measurements behind the line to DIR/bench_details_n<N>.json")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 arm")
    rank = int(os.environ.get("RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world_size > 1:
        args.no_c4 = False
    if args.impl == "reference":
        run_reference(args, rank, world_size)
    else:
        try:
            run_b200(args, rank, world_size, local_rank)
        finally:
            if world_size > 1:
                import torch.distributed as dist
                if dist.is_initialized():
                    dist.destroy_process_group()


if __name__ == "__main__":
    main()
