"""CPU tests: the plain-C oracle port (oracle/lgs_oracle.c) against the golden vectors generated from
the unmodified reference objects, and against those objects directly where they exist."""
import hashlib
import os

import numpy as np

from my_lidar_graph_slam_b200 import synth
from oracle import portapi as P
from oracle import refapi as R

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

RT_PARAMS = [dict(low_res=5, range_x=0.2, range_y=0.2, range_theta=0.5, scan_range_max=20.0),
             dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=1.0471975512, scan_range_max=5.7296),
             dict(low_res=3, range_x=0.6, range_y=0.4, range_theta=0.3, scan_range_max=8.0)]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.float64).tobytes()).hexdigest()


def ints(r):
    return [r.found, r.ix, r.iy, r.it, r.winX, r.winY, r.winT]


def check_match(r, gi, gf):
    assert ints(r)[:1] == list(gi[:1]) and ints(r)[4:] == list(gi[4:])
    assert r.stepT == gf[1]
    if gi[0]:
        assert ints(r)[1:4] == list(gi[1:4]) and r.score == gf[0]


def test_primitives_golden():
    g = np.load(os.path.join(GOLD, "primitives.npz"))
    for k, e in enumerate(g["bres_ends"]):
        want = g["bres_cells"][g["bres_offs"][k]:g["bres_offs"][k + 1]]
        assert np.array_equal(P.bresenham(*[int(v) for v in e]), want)
    for hits, trace in zip(g["bayes_hits"], g["bayes_trace"]):
        v = 0.0
        for h, want in zip(hits, trace):
            v = P.bayes_update(v, 0.6 if h else 0.45)
            assert v == want
    for a, w, want in zip(g["sw_in"], g["sw_w"], g["sw_out"]):
        assert np.array_equal(P.sliding_window_max(a, int(w)), want)


def test_bresenham_closed_form_used_by_the_kernel():
    """The O(1) membership test of lgs_integrate.cu (rayTouch) against the oracle's Bresenham."""
    rng = np.random.default_rng(3)

    def touch(rx, ry, ex, ey):        # same division-free logic as rayTouch in lgs_integrate.cu
        ax, ay = abs(ex), abs(ey)
        if ax > ay:
            k, t, amaj, amin = (-rx if ex < 0 else rx), (-ry if ey < 0 else ry), ax, ay
        else:
            k, t, amaj, amin = (-ry if ey < 0 else ry), (-rx if ex < 0 else rx), ay, ax
        if k < 0 or k > amaj or t < 0:
            return 0
        if amaj == 0:
            return 2 if t == 0 else 0
        lhs, m2 = 2 * amin * k + amaj, 2 * amaj
        if m2 * t > lhs or lhs >= m2 * (t + 1):
            return 0
        return 2 if k == amaj else 1

    for _ in range(300):
        ex, ey = (int(v) for v in rng.integers(-25, 26, 2))
        cells = {tuple(c): (2 if i == len(cs) - 1 else 1)
                 for cs in [P.bresenham(0, 0, ex, ey)] for i, c in enumerate(cs)}
        for rx in range(-27, 28):
            for ry in range(-27, 28):
                assert touch(rx, ry, ex, ey) == cells.get((rx, ry), 0)


def test_scene_golden_maps_pyramids_matches():
    g = np.load(os.path.join(GOLD, "scene_rooms.npz"))
    angles, traj, scans = g["angles"], g["traj"], g["scans"]
    b = P.PortBuilder()
    for p, s in zip(traj[:12], scans[:12]):
        b.append_scan(p, angles, s)
    local, latest = b.local_map(0), b.latest_map()
    assert list(local.geometry()) == list(g["local_geom"])
    assert list(latest.geometry()) == list(g["latest_geom"])
    assert np.array_equal(local.dense().view(np.int64), g["local_dense"].view(np.int64))
    assert np.array_equal(latest.dense().view(np.int64), g["latest_dense"].view(np.int64))
    pyr = local.pyramid(6)
    assert [sha(p.dense()) for p in pyr] == list(g["pyr_sha"])
    assert np.array_equal(pyr[3].dense(), g["pyr3"])
    assert sha(latest.precompute(5).dense()) == str(g["pre5_sha"])
    sp, hits, bbox = P.hit_points(traj[3], angles, scans[3])
    assert np.array_equal(sp, g["hit_sensor"]) and np.array_equal(hits, g["hit_xy"])
    assert np.array_equal(bbox, g["hit_bbox"])
    rt, bb = iter(zip(g["rt_int"], g["rt_f"])), iter(zip(g["bb_int"], g["bb_f"]))
    for k, init in zip(range(12, 18), g["inits"]):
        for p in RT_PARAMS:
            check_match(P.rtcsm_match(latest, angles, scans[k], init, **p), *next(rt))
        for thr in (0.6, 0.3):
            check_match(P.bb_match(local, angles, scans[k], init, pyramid=pyr, thr=thr), *next(bb))


def test_edge_scene_golden_order_dependent_results():
    g = np.load(os.path.join(GOLD, "scene_edge.npz"))
    m = P.PortMap.from_dense(g["dense"], -1.0, -2.0)
    pre, pyr = m.precompute(5), m.pyramid(4)
    rt = dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=0.2, scan_range_max=20.0)
    bb = dict(height_max=4, range_x=1.0, range_y=1.0, range_theta=0.2)
    for k in range(len(g["ranges"])):
        check_match(P.rtcsm_match(m, g["angles"], g["ranges"][k], g["inits"][k], pre=pre, **rt),
                    g["rt_int"][k], g["rt_f"][k])
        check_match(P.bb_match(m, g["angles"], g["ranges"][k], g["inits"][k], pyramid=pyr,
                               thr=float(g["thrs"][k]), **bb), g["bb_int"][k], g["bb_f"][k])


def test_cost_function_golden():
    """CostGreedyEndpoint::Cost / ComputeCovariance (the matchers' host tail), bit for bit."""
    g, c = np.load(os.path.join(GOLD, "scene_rooms.npz")), np.load(os.path.join(GOLD, "scene_cost.npz"))
    angles, traj, scans = g["angles"], g["traj"], g["scans"]
    b = P.PortBuilder()
    for p, s in zip(traj[:12], scans[:12]):
        b.append_scan(p, angles, s)
    latest = b.latest_map()
    assert len(set(c["cost"][:, 0].tolist())) > 10 and np.all(c["cost"][:, 0] < 0.0)
    for pose, k, want, wn, wc in zip(c["poses"], c["scan"], c["cost"], c["normalized"], c["cov"]):
        for j, cs in enumerate(c["cost_sets"]):
            assert P.cost_greedy_endpoint(latest, pose, angles, scans[k], cost=tuple(cs)) == want[j]
            n, _, cov = P.host_tail(latest, pose, angles, scans[k], cost=tuple(cs))
            assert n == wn[j] and np.array_equal(cov, wc[j])


GS_PARAMS = [dict(range_x=0.6, range_y=0.5, range_theta=0.12, step_x=0.05, step_y=0.05, step_theta=0.01),
             dict(range_x=0.4, range_y=0.4, range_theta=0.1, step_x=0.03, step_y=0.07, step_theta=0.013),
             dict(range_x=0.3, range_y=0.3, range_theta=0.05, step_x=0.1, step_y=0.1, step_theta=0.005)]


def test_grid_search_golden():
    """ScanMatcherGridSearch: winner (as loop counters), loop lengths and score."""
    g, c = np.load(os.path.join(GOLD, "scene_rooms.npz")), np.load(os.path.join(GOLD, "scene_gs.npz"))
    angles, traj, scans = g["angles"], g["traj"], g["scans"]
    b = P.PortBuilder()
    for p, s in zip(traj[:12], scans[:12]):
        b.append_scan(p, angles, s)
    local = b.local_map(0)
    assert c["ints"][:, 0].sum() >= 10 and (c["ints"][:, 0] == 0).sum() >= 4
    for n, (init, k, thr, gi, gf) in enumerate(zip(c["inits"], c["scan"], c["thr"], c["ints"], c["flts"])):
        r = P.gs_match(local, angles, scans[k], init, thr=float(thr), **GS_PARAMS[n % 3])
        assert [r.found, r.ix, r.iy, r.it, r.winX, r.winY, r.winT] == list(gi)
        assert r.score == gf[0]


# ---- randomised cases: the port against the reference objects' answers on the same seeded inputs ----------------
# Each case draws its inputs from a fixed seed and runs them through backend M (the port P or the reference
# objects R).  tests/golden/reference_randomised.npz holds the reference's answers (make_golden.py); where
# oracle/_ref/liblgs_ref.so is built, the port is also compared with the live objects.
REF_GOLD = os.path.join(GOLD, "reference_randomised.npz")


def _map(M, dense, min_x, min_y):
    return (R.RefMap if M is R else P.PortMap).from_dense(dense, min_x, min_y)


def _drawn(*arrays):
    return sha(np.concatenate([np.ravel(np.asarray(a, dtype=np.float64)) for a in arrays]))


def cost_case(M):
    rng = np.random.default_rng(31)
    dense = np.where(rng.random((128, 192)) < 0.5, np.round(rng.uniform(1e-3, 0.999, (128, 192)), 2), 0.0)
    m = _map(M, dense, -3.0, -2.0)
    angles = synth.beam_angles(91, 360.0)
    drawn, cost, tail_n, tail_cov = [dense], [], [], []
    for _ in range(40):
        ranges = rng.uniform(0.0, 4.0, angles.shape)
        pose = np.array([rng.uniform(-3.5, 3.5), rng.uniform(-2.5, 3.0), rng.uniform(-4, 4)])   # partly off the map
        cs = (rng.uniform(0.0, 0.5), rng.uniform(2.0, 5.0), rng.uniform(0.02, 0.2), rng.uniform(0.05, 0.6),
              float(rng.integers(0, 4)), rng.uniform(0.1, 3.0), rng.uniform(0.02, 1.0))
        kw = dict(scan_min_range=float(rng.uniform(0, 0.3)), scan_max_range=float(rng.uniform(3, 6)), cost=cs)
        drawn += [ranges, pose, cs, [kw["scan_min_range"], kw["scan_max_range"]]]
        cost.append(M.cost_greedy_endpoint(m, pose, angles, ranges, **kw))
        n, _, cov = M.host_tail(m, pose, angles, ranges, **kw)
        tail_n.append(n)
        tail_cov.append(cov)
    return dict(inputs=_drawn(*drawn), cost=np.array(cost), tail_n=np.array(tail_n), tail_cov=np.array(tail_cov))


def primitives_case(M):
    rng = np.random.default_rng(11)
    ends, cells, offs = [], [], [0]
    for _ in range(300):
        e = [int(v) for v in rng.integers(-60, 61, 4)]
        c = np.asarray(M.bresenham(*e))
        ends.append(e)
        cells.append(c.reshape(-1, 2))
        offs.append(offs[-1] + len(cells[-1]))
    v, trace, hits = 0.0, [], rng.random(500) < 0.45
    for h in hits:
        v = M.bayes_update(v, 0.6 if h else 0.45)
        trace.append(v)
    sw_in, sw_out = [], []
    for n, win in [(50, 7), (50, 50), (50, 64), (7, 3), (1, 1), (130, 33)]:
        a = np.where(rng.random(n) < 0.6, rng.random(n), 0.0)
        sw_in.append(a)
        sw_out.append(np.asarray(M.sliding_window_max(a, win)))
    dense = np.where(rng.random((128, 192)) < 0.3, rng.uniform(1e-3, 0.999, (128, 192)), 0.0)
    m = _map(M, dense, -3.0, 2.0)
    return dict(inputs=_drawn(np.ravel(ends), hits, *sw_in, dense), bres_cells=np.concatenate(cells),
                bres_offs=np.array(offs), bayes_trace=np.array(trace), sw_out=np.concatenate(sw_out),
                pre_sha=np.array([sha(m.precompute(win).dense()) for win in (1, 2, 5, 9, 64, 150, 400)]),
                pyr_sha=np.array([sha(p.dense()) for p in m.pyramid(7)]))


def builder_case(M):
    world = synth.RoomsWorld(30.0, 5.0, seed=13)
    angles = synth.beam_angles(271, 270.0)
    traj = synth.trajectory(world, 30, step=0.3, seed=13)
    noise = np.random.default_rng(14)
    scans = [synth.make_scan(world, p, angles, noise) for p in traj]
    b = (R.RefBuilder if M is R else P.PortBuilder)(travel_thr=4.0)   # forces several local maps
    appended = [b.append_scan(p, angles, s) for p, s in zip(traj[:24], scans[:24])]
    n_local = b.num_local_maps()
    maps = [b.local_map(i) for i in range(n_local)]
    latest, lm = b.latest_map(), b.local_map(1)
    pyr = lm.pyramid(5)
    prng = np.random.default_rng(15)
    inits, rt_int, rt_f, bb_int, bb_score = [], [], [], [], []
    for k in range(24, 30):
        init = traj[k] + np.array([prng.uniform(-0.3, 0.3), prng.uniform(-0.3, 0.3), prng.uniform(-0.2, 0.2)])
        inits.append(init)
        for p in RT_PARAMS:
            r = M.rtcsm_match(latest, angles, scans[k], init, **p)
            rt_int.append(ints(r))
            rt_f.append([r.score, r.stepT])
        for thr in (0.55, 0.2):
            r = M.bb_match(lm, angles, scans[k], init, pyramid=pyr, thr=thr, height_max=5, range_x=1.5,
                           range_y=1.5, range_theta=0.6)
            bb_int.append(ints(r))
            bb_score.append(r.score if r.found else 0.0)           # a score is only defined when found
    return dict(inputs=_drawn(traj, *scans, *inits), appended=np.array(appended), n_local=np.array(n_local),
                local_geom=np.array([m.geometry() for m in maps], dtype=np.float64),
                local_sha=np.array([sha(m.dense()) for m in maps]),
                local_nodes=np.array([b.local_map_nodes(i) for i in range(n_local)]),
                latest_geom=np.array(latest.geometry(), dtype=np.float64), latest_sha=np.array(sha(latest.dense())),
                rt_int=np.array(rt_int), rt_f=np.array(rt_f), bb_int=np.array(bb_int), bb_score=np.array(bb_score))


RANDOMISED = {"cost": cost_case, "primitives": primitives_case, "builder": builder_case}


def check_randomised(name):
    got = RANDOMISED[name](P)
    gold = np.load(REF_GOLD)
    want = {k.split("__", 1)[1]: gold[k] for k in gold.files if k.startswith(name + "__")}
    assert sorted(got) == sorted(want)
    for k, v in got.items():
        assert np.array_equal(np.asarray(v), want[k]), (name, k)
    if R.available():
        live = RANDOMISED[name](R)
        for k, v in got.items():
            assert np.array_equal(np.asarray(v), np.asarray(live[k])), (name, k, "live reference objects")


def test_port_cost_matches_reference_objects_randomised():
    check_randomised("cost")


def test_port_matches_reference_objects_randomised():
    check_randomised("primitives")


def test_port_builder_and_matchers_match_reference_objects():
    check_randomised("builder")
    assert int(np.load(REF_GOLD)["builder__n_local"]) >= 2
