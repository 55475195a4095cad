#!/usr/bin/env python
"""Generates tests/golden/*.npz from the UNMODIFIED reference objects (oracle/_ref/liblgs_ref.so).

Run where the reference sources are at hand (oracle/Makefile `make ref`):  python tests/golden/make_golden.py
The reference ships no golden vectors of its own (SURVEY.md section 4); these fixtures pin the
plain-C oracle port (and, through it, the CUDA path) wherever the reference objects are absent.

reference_randomised.npz holds the answers to the seeded randomised cases of tests/test_oracle_port.py
(the inputs are drawn there; the file records which backend wrote it under `source`).  The committed file
was written with `--randomised-from-port`, by the plain-C port: at commit f3c2a39 the tests these cases
were made from, drawing the same inputs in the same order, passed bit for bit against the reference
objects built from the unmodified sources, and the port (oracle/) and synth.py are unchanged since, so
the port's answers on these inputs are the reference's.  The port also reproduces every reference-written file above.  Where the reference
objects can be built, the plain run regenerates it from them with the other files.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from my_lidar_graph_slam_b200 import synth  # noqa: E402
from oracle import refapi as R  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.float64).tobytes()).hexdigest()


def res_tuple(r):
    return [r.found, r.ix, r.iy, r.it, r.winX, r.winY, r.winT], [r.score, r.stepT]


def primitives():
    rng = np.random.default_rng(42)
    ends = rng.integers(-40, 41, size=(200, 4)).astype(np.int32)
    ends[:8] = [[0, 0, 0, 0], [0, 0, 5, 5], [0, 0, -5, 5], [3, 3, 3, 9], [3, 3, 9, 3], [0, 0, 7, 3],
                [0, 0, -3, -7], [2, -1, -6, 3]]
    cells, offs = [], [0]
    for e in ends:
        c = R.bresenham(*[int(v) for v in e])
        cells.append(c)
        offs.append(offs[-1] + len(c))
    # Bayes update: random hit/miss sequences from unknown
    seqs = rng.random((64, 48)) < 0.4            # True = hit
    finals = []
    for s in seqs:
        v = 0.0
        trace = []
        for h in s:
            v = R.bayes_update(v, 0.6 if h else 0.45)
            trace.append(v)
        finals.append(trace)
    sw_in = np.where(rng.random((12, 97)) < 0.5, rng.random((12, 97)), 0.0)
    sw_w = np.array([1, 2, 3, 5, 8, 16, 33, 64, 96, 97, 98, 200], dtype=np.int32)
    sw_out = np.stack([R.sliding_window_max(sw_in[k], int(sw_w[k])) for k in range(12)])
    np.savez_compressed(os.path.join(OUT, "primitives.npz"), bres_ends=ends,
                        bres_cells=np.concatenate(cells), bres_offs=np.asarray(offs, dtype=np.int32),
                        bayes_hits=seqs, bayes_trace=np.asarray(finals), sw_in=sw_in, sw_w=sw_w,
                        sw_out=sw_out)


def scene():
    world = synth.RoomsWorld(24.0, 4.0, seed=7)
    angles = synth.beam_angles(181, 180.0)
    traj = synth.trajectory(world, 18, step=0.3, seed=7)
    noise = np.random.default_rng(8)
    scans = np.stack([synth.make_scan(world, p, angles, noise) for p in traj])
    b = R.RefBuilder()
    for p, s in zip(traj[:12], scans[:12]):
        b.append_scan(p, angles, s)
    local, latest = b.local_map(0), b.latest_map()
    pyr = local.pyramid(6)
    out = dict(angles=angles, traj=traj, scans=scans, local_dense=local.dense(),
               local_geom=np.array(local.geometry()), latest_dense=latest.dense(),
               latest_geom=np.array(latest.geometry()),
               pyr_sha=np.array([sha(p.dense()) for p in pyr]),
               pre5_sha=np.array(sha(latest.precompute(5).dense())),
               pyr3=pyr[3].dense())
    sp, hits, bbox = R.hit_points(traj[3], angles, scans[3])
    out.update(hit_sensor=sp, hit_xy=hits, hit_bbox=bbox)
    rt_params = [dict(low_res=5, range_x=0.2, range_y=0.2, range_theta=0.5, scan_range_max=20.0),
                 dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=1.0471975512, scan_range_max=5.7296),
                 dict(low_res=3, range_x=0.6, range_y=0.4, range_theta=0.3, scan_range_max=8.0)]
    rt_i, rt_f, bb_i, bb_f, inits = [], [], [], [], []
    prng = np.random.default_rng(9)
    for k in range(12, 18):
        init = traj[k] + np.array([prng.uniform(-0.25, 0.25), prng.uniform(-0.25, 0.25), prng.uniform(-0.15, 0.15)])
        inits.append(init)
        for p in rt_params:
            i, f = res_tuple(R.rtcsm_match(latest, angles, scans[k], init, **p))
            rt_i.append(i); rt_f.append(f)
        for thr in (0.6, 0.3):
            i, f = res_tuple(R.bb_match(local, angles, scans[k], init, pyramid=pyr, thr=thr))
            bb_i.append(i); bb_f.append(f)
    out.update(inits=np.asarray(inits), rt_int=np.asarray(rt_i, dtype=np.int64), rt_f=np.asarray(rt_f),
               bb_int=np.asarray(bb_i, dtype=np.int64), bb_f=np.asarray(bb_f))
    np.savez_compressed(os.path.join(OUT, "scene_rooms.npz"), **out)


def edge_scene():
    """Scans hanging over the lower-left edge of a tight map: the win-max values are not upper
    bounds there (SURVEY.md H12) and the reference's pruned searches become order dependent."""
    rng = np.random.default_rng(7)
    ny, nx = 128, 128
    dense = np.where(rng.random((ny, nx)) < 0.25, rng.uniform(0.05, 0.95, (ny, nx)), 0.0)
    dense[:12, :] = rng.uniform(0.5, 0.99, (12, nx))
    dense[:, :12] = rng.uniform(0.5, 0.99, (ny, 12))
    dense = np.round(dense, 3)                    # compresses well, still arbitrary doubles
    m = R.RefMap.from_dense(dense, -1.0, -2.0)
    pre = m.precompute(5)
    pyr = m.pyramid(4)
    angles = synth.beam_angles(181, 180.0)
    rt = dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=0.2, scan_range_max=20.0)
    bb = dict(height_max=4, range_x=1.0, range_y=1.0, range_theta=0.2)
    ranges, inits, thrs, rt_i, rt_f, bb_i, bb_f = [], [], [], [], [], [], []
    for k in range(10):
        r = rng.uniform(0.1, 0.5, angles.shape)
        init = np.array([-1.0 + rng.uniform(0.0, 0.3), -2.0 + rng.uniform(0.5, 3.0), np.pi + rng.uniform(-0.3, 0.3)])
        thr = float(rng.uniform(0.2, 0.5))
        ranges.append(r); inits.append(init); thrs.append(thr)
        i, f = res_tuple(R.rtcsm_match(m, angles, r, init, pre=pre, **rt))
        rt_i.append(i); rt_f.append(f)
        i, f = res_tuple(R.bb_match(m, angles, r, init, pyramid=pyr, thr=thr, **bb))
        bb_i.append(i); bb_f.append(f)
    np.savez_compressed(os.path.join(OUT, "scene_edge.npz"), dense=dense, angles=angles,
                        ranges=np.asarray(ranges), inits=np.asarray(inits), thrs=np.asarray(thrs),
                        rt_int=np.asarray(rt_i, dtype=np.int64), rt_f=np.asarray(rt_f),
                        bb_int=np.asarray(bb_i, dtype=np.int64), bb_f=np.asarray(bb_f))


COST_SETS = [(0.01, 20.0, 0.075, 0.1, 1.0, 0.05, 1.0),      # launcher defaults as the launcher passes them
             (0.01, 20.0, 0.075, 0.1, 1.0, 1.0, 0.05),      # the header's meaning of the last two
             (0.5, 6.0, 0.1, 0.3, 2.0, 2.5, 0.08),
             (0.01, 20.0, 0.05, 0.5, 0.0, 1.0, 0.05),       # kernel size 0
             (0.01, 20.0, 0.075, 0.05, 3.0, 1.0, 0.1)]


def cost_scene():
    """CostGreedyEndpoint::Cost and the matchers' host tail on the latest map of scene_rooms."""
    g = np.load(os.path.join(OUT, "scene_rooms.npz"))
    angles, traj, scans = g["angles"], g["traj"], g["scans"]
    b = R.RefBuilder()
    for p, s in zip(traj[:12], scans[:12]):
        b.append_scan(p, angles, s)
    latest = b.latest_map()
    rng = np.random.default_rng(21)
    poses, which, costs, ncost, cov = [], [], [], [], []
    for k in range(6, 18):
        for _ in range(3):
            pose = traj[k] + np.array([rng.uniform(-0.2, 0.2), rng.uniform(-0.2, 0.2), rng.uniform(-0.1, 0.1)])
            poses.append(pose); which.append(k)
            costs.append([R.cost_greedy_endpoint(latest, pose, angles, scans[k], cost=c) for c in COST_SETS])
            tails = [R.host_tail(latest, pose, angles, scans[k], cost=c) for c in COST_SETS]
            ncost.append([t[0] for t in tails]); cov.append([t[2] for t in tails])
    np.savez_compressed(os.path.join(OUT, "scene_cost.npz"), poses=np.asarray(poses),
                        scan=np.asarray(which, dtype=np.int32), cost_sets=np.asarray(COST_SETS),
                        cost=np.asarray(costs), normalized=np.asarray(ncost), cov=np.asarray(cov))


GS_PARAMS = [dict(range_x=0.6, range_y=0.5, range_theta=0.12, step_x=0.05, step_y=0.05, step_theta=0.01),
             dict(range_x=0.4, range_y=0.4, range_theta=0.1, step_x=0.03, step_y=0.07, step_theta=0.013),
             dict(range_x=0.3, range_y=0.3, range_theta=0.05, step_x=0.1, step_y=0.1, step_theta=0.005)]


def gs_scene():
    """ScanMatcherGridSearch on the first local map of scene_rooms (small windows: the CPU search costs
    a full projection of the scan per hypothesis)."""
    g = np.load(os.path.join(OUT, "scene_rooms.npz"))
    angles, traj, scans = g["angles"], g["traj"], g["scans"]
    b = R.RefBuilder()
    for p, s in zip(traj[:12], scans[:12]):
        b.append_scan(p, angles, s)
    local = b.local_map(0)
    rng = np.random.default_rng(23)
    inits, which, ints, flts, thrs = [], [], [], [], []
    for k in range(12, 18):
        init = traj[k] + np.array([rng.uniform(-0.15, 0.15), rng.uniform(-0.15, 0.15), rng.uniform(-0.03, 0.03)])
        for pi, p in enumerate(GS_PARAMS):
            thr = 0.3 if pi != 2 else 0.9            # the last one is not found
            r = R.gs_match(local, angles, scans[k], init, thr=thr, **p)
            inits.append(init); which.append(k); thrs.append(thr)
            ints.append([r.found, r.ix, r.iy, r.it, r.winX, r.winY, r.winT])
            flts.append([r.score, r.normalizedCost] + list(r.estPose) + list(r.cov))
    np.savez_compressed(os.path.join(OUT, "scene_gs.npz"), inits=np.asarray(inits),
                        scan=np.asarray(which, dtype=np.int32), thr=np.asarray(thrs),
                        ints=np.asarray(ints, dtype=np.int64), flts=np.asarray(flts))


def reference_randomised(M):
    """Answers of backend M to the randomised cases of tests/test_oracle_port.py (fixed seeds)."""
    sys.path.insert(0, os.path.dirname(OUT))
    import test_oracle_port as T
    out = {"source": np.array(M.__name__.rsplit(".", 1)[-1])}
    for name, case in T.RANDOMISED.items():
        out.update({f"{name}__{k}": np.asarray(v) for k, v in case(M).items()})
    np.savez_compressed(os.path.join(OUT, "reference_randomised.npz"), **out)


if __name__ == "__main__" and sys.argv[1:] == ["--randomised-from-port"]:
    from oracle import portapi
    reference_randomised(portapi)
elif __name__ == "__main__":
    reference_randomised(R)
    primitives()
    scene()
    edge_scene()
    cost_scene()
    gs_scene()
    for f in sorted(os.listdir(OUT)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(OUT, f)))
