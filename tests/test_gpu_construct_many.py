"""GPU parity: lgs_grid_construct_many (ConstructMapFromScans of many maps from raw scans, one call) against the
oracle's PortBuilder.construct_into and against the host path -- lgs_scan_hit_points per scan, the bbox,
lgs_geometry_resize, lgs_grid_integrate_many.  Cells as int64, geometry fields, bbox doubles and update counts are
compared bit for bit."""
import math

import numpy as np
import pytest

from my_lidar_graph_slam_b200 import capi, synth
from oracle import portapi as P

pytestmark = pytest.mark.gpu

TINY = float(np.finfo(np.float64).tiny)
DBL_MAX = float(np.finfo(np.float64).max)
CON_LAUNCHES = 6          # count, offsets, project, candidates, near-edge, patch
INITIAL_CANDIDATES = 4096


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _geo(t, patch=64):
    nx, ny, mx, my, res = t
    return capi.Geometry(int(nx), int(ny), float(mx), float(my), float(res), patch)


def _host_path(ctx, scans_list, curs, apron=2):
    """lgs_scan_hit_points per scan, the bbox from DBL_MAX / DBL_MIN, lgs_geometry_resize, integrate_many."""
    geos, bboxes, grids, sensors, hits = [], [], [], [], []
    for sc, cur in zip(scans_list, curs):
        bl, tr, hs = [DBL_MAX, DBL_MAX], [TINY, TINY], []
        for k in range(sc.n):
            b0, b1 = sc.beam_begin[k], sc.beam_begin[k + 1]
            h, b = capi.scan_hit_points(sc.sensor_pose[k], sc.angles[b0:b1], sc.ranges[b0:b1],
                                        sc.range_min[k], sc.range_max[k])
            bl = [min(bl[0], b[0]), min(bl[1], b[1])]
            tr = [max(tr[0], b[2]), max(tr[1], b[3])]
            hs.append(h)
        geo, _, _ = capi.geometry_resize(cur, (bl[0], bl[1], tr[0], tr[1]))
        geos.append(geo)
        bboxes.append([bl[0], bl[1], tr[0], tr[1]])
        grids.append(capi.Grid(ctx, geo.nx, geo.ny, geo.min_x, geo.min_y, geo.res, apron=apron))
        sensors.append(sc.sensor_pose[:, :2])
        hits.append(hs)
    before = ctx.launch_count()
    counts = capi.integrate_many(ctx, grids, sensors, hits)
    return geos, np.asarray(bboxes), counts, grids, ctx.launch_count() - before


def _construct(ctx, scans_list, curs, apron=2):
    grids = [capi.Grid(ctx, c.nx, c.ny, c.min_x, c.min_y, c.res, apron=apron) for c in curs]
    before = ctx.launch_count()
    geos, bboxes, counts = capi.construct_many(ctx, grids, scans_list, curs)
    return geos, bboxes, counts, grids, ctx.launch_count() - before


def _assert_same(a, b, what=""):
    geos_a, bb_a, cnt_a, grids_a = a[:4]
    geos_b, bb_b, cnt_b, grids_b = b[:4]
    assert [g.as_tuple() for g in geos_a] == [g.as_tuple() for g in geos_b], what
    assert np.array_equal(_bits(bb_a), _bits(bb_b)), what
    assert list(cnt_a) == list(cnt_b), what
    for i, (ga, gb) in enumerate(zip(grids_a, grids_b)):
        assert (ga.nx, ga.ny, ga.min_x, ga.min_y) == (gb.nx, gb.ny, gb.min_x, gb.min_y), f"{what} map {i}"
        assert np.array_equal(_bits(ga.download()), _bits(gb.download())), f"{what} map {i}"


def _scans(poses, angles, ranges_list, rmin=0.02, rmax=20.0):
    return capi.Scans([angles] * len(poses), ranges_list, poses, range_min=rmin, range_max=rmax)


@pytest.fixture(scope="module")
def rebuild_scene():
    """The loop-closure rebuild of test_loop_closure_rebuild_matches_construct_map: RoomsWorld, 1081 beams,
    local maps built from the first trajectory, rebuilt from corrected poses."""
    world = synth.RoomsWorld(40.0, 5.0, seed=41)
    angles = synth.beam_angles(1081, 270.0)
    traj = synth.trajectory(world, 72, step=0.25, seed=41)
    noise = np.random.default_rng(42)
    scans = [synth.make_scan(world, p, angles, noise) for p in traj]
    builder = P.PortBuilder(travel_thr=2.0)
    for p, r in zip(traj, scans):
        builder.append_scan(p, angles, r)
    spans = [builder.local_map_nodes(i) for i in range(builder.num_local_maps())]
    curs = [_geo(builder.local_map(i).geometry()) for i in range(len(spans))]
    hi = len(traj) - 1
    spans.append((max(0, hi - builder.n_latest + 1), hi))               # the latest map's window
    curs.append(_geo(builder.latest_map().geometry()))
    corrected = traj + np.random.default_rng(43).normal(0.0, [0.04, 0.04, 0.01], traj.shape)
    rebuilt = P.PortBuilder(travel_thr=2.0)
    for p, r in zip(corrected, scans):
        rebuilt.append_node_only(p, angles, r)
    sensor = np.array([P.compound(p, rebuilt.rel) for p in corrected])
    lists = [_scans(sensor[lo:hi + 1], angles, scans[lo:hi + 1]) for lo, hi in spans]
    return dict(rebuilt=rebuilt, spans=spans, curs=curs, lists=lists, sensor=sensor, angles=angles, scans=scans)


def test_loop_closure_rebuild_matches_construct_map(ctx, rebuild_scene):
    """Every local map (cur = its previous geometry) plus the latest-map window in ONE call, against
    PortBuilder.construct_into and against the host path; launches = the host path's + a constant."""
    sc = rebuild_scene
    assert len(sc["spans"]) >= 9
    got = _construct(ctx, sc["lists"], sc["curs"])
    host = _host_path(ctx, sc["lists"], sc["curs"])
    _assert_same(got, host, "vs host path")
    assert got[4] == host[4] + CON_LAUNCHES
    for i, ((lo, hi), cur) in enumerate(zip(sc["spans"], sc["curs"])):
        m = P.PortMap(np.zeros((cur.ny, cur.nx)), cur.min_x, cur.min_y, cur.res, cur.patch)
        sc["rebuilt"].construct_into(m, lo, hi)
        assert got[0][i].as_tuple() == m.geometry(), f"map {i}"
        assert np.array_equal(_bits(got[3][i].download()), _bits(m.dense())), f"map {i}"


def test_everything_on_the_host_gives_the_same_maps(ctx, rebuild_scene):
    """With "integ_resolve_ulps" huge every hit is near-edge and every hit a bbox candidate."""
    sc = rebuild_scene
    want = _construct(ctx, sc["lists"], sc["curs"])
    b0, e0 = capi.construct_host_points(ctx)
    ctx.set_option("integ_resolve_ulps", 1e300)
    try:
        got = _construct(ctx, sc["lists"], sc["curs"])
    finally:
        ctx.set_option("integ_resolve_ulps", 8)
    hits = sum(int(np.count_nonzero(~((r >= s.range_max[k]) | (r <= s.range_min[k]))))
               for s in sc["lists"] for k in range(s.n) for r in [s.ranges[s.beam_begin[k]:s.beam_begin[k + 1]]])
    b1, e1 = capi.construct_host_points(ctx)
    assert e1 - e0 == hits and b1 - b0 == hits
    _assert_same(got, want, "all on the host")


def test_global_map_and_negative_coordinates(ctx, rebuild_scene):
    """ConstructGlobalMap: every node into one fresh map anchored at (0, 0); and a map whose every point lies at
    negative coordinates, where the DBL_MIN seed is the upper bound."""
    sc = rebuild_scene
    everything = _scans(sc["sensor"], sc["angles"], sc["scans"])
    shifted = _scans(sc["sensor"][:12] - np.array([80.0, 60.0, 0.0]), sc["angles"], sc["scans"][:12])
    curs = [capi.Geometry(0, 0, 0.0, 0.0, 0.05, 64)] * 2
    got = _construct(ctx, [everything, shifted], curs)
    _assert_same(got, _host_path(ctx, [everything, shifted], curs))
    assert got[1][1][2] == TINY and got[1][1][3] == TINY
    m = P.PortMap(np.zeros((0, 0)), 0.0, 0.0, 0.05, 64)
    sc["rebuilt"].construct_into(m, 0, len(sc["sensor"]) - 1)
    assert got[0][0].as_tuple() == m.geometry()
    assert np.array_equal(_bits(got[3][0].download()), _bits(m.dense()))


def test_range_filter(ctx):
    """Ranges exactly at range_min / range_max and beyond, a window per scan, NaN / inf beyond the filter, and
    scans without hits (the bbox is then the sensor positions)."""
    rng = np.random.default_rng(5)
    angles = np.linspace(-2.0, 2.0, 400)
    poses = rng.uniform([-3.0, -3.0, -math.pi], [3.0, 3.0, math.pi], (9, 3))
    rmin = np.array([0.02, 0.5, 1.0, -1.0, 0.02, 0.3, 2.0, 0.1, 0.2])
    rmax = np.array([20.0, 4.0, 6.0, 3.0, 8.0, 5.0, 2.5, 7.0, 9.0])
    ranges = []
    for k in range(9):
        r = rng.uniform(rmin[k] - 1.0, rmax[k] + 1.0, len(angles))
        r[::7] = rmin[k]
        r[3::7] = rmax[k]
        r[5::11] = np.inf
        ranges.append(r)
    ranges[2][:] = rmax[2]                                   # a scan without hits
    ranges[8][::13] = -np.inf
    maps = [_scans(poses[:5], angles, ranges[:5], rmin[:5], rmax[:5]),
            _scans(poses[5:], angles, ranges[5:], rmin[5:], rmax[5:]),
            _scans(poses[2:3], angles, [np.full(len(angles), 9.0)], 0.02, 8.0)]    # no hits at all
    curs = [capi.Geometry(0, 0, 0.0, 0.0, 0.05, 64), capi.Geometry(128, 64, -1.0, 2.0, 0.1, 32),
            capi.Geometry(0, 0, 0.3, 0.7, 0.05, 16)]
    got = _construct(ctx, maps, curs)
    _assert_same(got, _host_path(ctx, maps, curs))
    px, py = poses[2][0], poses[2][1]
    assert got[2][2] == 0 and np.array_equal(_bits(got[1][2]), _bits([px, py, max(px, TINY), max(py, TINY)]))


def test_near_edge_beams(ctx):
    """Beams at angle 0 and pi/2 whose hits land exactly on cell edges (r = whole cells from a sensor on a cell
    corner, all exact in binary): the device interval straddles the edge, so they are re-derived on the host."""
    res = 0.25
    sensor = np.array([[1.0, 1.0, 0.0], [2.0, 0.5, 0.0], [0.5, 2.0, math.pi / 2]])
    angles = np.array([0.0, math.pi / 2, math.pi, -math.pi / 2] * 40)
    ranges = [np.repeat(res * np.arange(1, 41), 4) for _ in range(3)]
    maps = [_scans(sensor, angles, ranges, 0.01, 20.0)]
    curs = [capi.Geometry(0, 0, 0.0, 0.0, res, 16)]
    _, e0 = capi.construct_host_points(ctx)
    got = _construct(ctx, maps, curs)
    _, e1 = capi.construct_host_points(ctx)
    _assert_same(got, _host_path(ctx, maps, curs))
    assert e1 > e0


def test_bbox_ties_on_a_flat_wall(ctx):
    """A noise-free wall perpendicular to x: every beam that hits it ends at x = W (r = W / cos a), so every one
    is a candidate for the max-x side, more than the initial candidate buffer holds."""
    W = 4.0
    angles = np.linspace(-1.2, 1.2, 1201)
    n = 6
    poses = np.zeros((n, 3))
    poses[:, 1] = np.linspace(-0.5, 0.5, n)
    ranges = [W / np.cos(angles)] * n
    maps = [_scans(poses, angles, ranges, 0.02, 30.0)]
    curs = [capi.Geometry(0, 0, 0.0, 0.0, 0.05, 64)]
    b0, _ = capi.construct_host_points(ctx)
    got = _construct(ctx, maps, curs)
    b1, _ = capi.construct_host_points(ctx)
    _assert_same(got, _host_path(ctx, maps, curs))
    assert b1 - b0 > INITIAL_CANDIDATES


def test_launch_count_does_not_depend_on_the_number_of_maps(ctx, rebuild_scene):
    sc = rebuild_scene
    extra = []
    for m in (2, 60):
        lists = [sc["lists"][k % len(sc["lists"])] for k in range(m)]
        curs = [sc["curs"][k % len(sc["curs"])] for k in range(m)]
        got, host = _construct(ctx, lists, curs), _host_path(ctx, lists, curs)
        _assert_same(got, host, f"{m} maps")
        extra.append(got[4] - host[4])
    assert extra == [CON_LAUNCHES, CON_LAUNCHES]


def test_grids_of_another_context(ctx, rebuild_scene):
    sc = rebuild_scene
    other = capi.Context(0)
    try:
        lists, curs = sc["lists"][:3], sc["curs"][:3]
        foreign = [capi.Grid(other, c.nx, c.ny, c.min_x, c.min_y, c.res, apron=2) for c in curs]
        geos, bboxes, counts = capi.construct_many(ctx, foreign, lists, curs)
        _assert_same((geos, bboxes, counts, foreign), _host_path(ctx, lists, curs))
    finally:
        other.close()


def test_refusals_leave_the_grids_unchanged(ctx, rebuild_scene):
    sc = rebuild_scene
    lists, curs = sc["lists"][:2], sc["curs"][:2]
    grids = _construct(ctx, lists, curs)[3]
    before = [(g.download(), (g.nx, g.ny, g.min_x, g.min_y)) for g in grids]
    a = sc["angles"]

    def bad(poses=None, ranges=None, angles=None, rmin=0.02, rmax=20.0):
        p = sc["sensor"][:3] if poses is None else poses
        r = sc["scans"][:3] if ranges is None else ranges
        return capi.Scans([a if angles is None else angles] * 3, r, p, range_min=rmin, range_max=rmax)

    nan_pose = sc["sensor"][:3].copy()
    nan_pose[1, 2] = np.nan
    nan_range = [r.copy() for r in sc["scans"][:3]]
    nan_range[2][100] = np.nan
    inf_angle = a.copy()
    inf_angle[10:600:7] = np.inf
    cases = [(bad(poses=nan_pose), "non-finite sensor pose"), (bad(rmax=np.inf), "non-finite sensor pose or range"),
             (bad(ranges=nan_range), "map 1, scan 2: a beam"), (bad(angles=inf_angle), "non-finite angle"),
             (capi.Scans([], [], np.zeros((0, 3)), range_min=0.02, range_max=20.0), "no scans"),
             (capi.Scans([a], [sc["scans"][0]], sc["sensor"][:1]), "range_max are required")]
    for scans, msg in cases:
        with pytest.raises(capi.LgsError, match=msg):
            capi.construct_many(ctx, grids, [lists[0], scans], curs)
    with pytest.raises(capi.LgsError, match="twice"):
        capi.construct_many(ctx, [grids[0], grids[0]], lists, curs)
    windowed = capi.Grid(ctx, 64, 64, 0.0, 0.0, 0.05, apron=1)
    windowed.set_window(16, 0)
    with pytest.raises(capi.LgsError, match="windowed"):
        capi.construct_many(ctx, [grids[0], windowed], lists, curs)
    pending = capi.Grid(ctx, 256, 256, -6.4, -6.4, 0.05, apron=1)
    capi.integrate_submit(ctx, pending, capi.PackedHits(np.zeros((1, 2)), [np.zeros((1, 2))]))
    with pytest.raises(capi.LgsError, match="in flight"):
        capi.construct_many(ctx, grids, lists, curs)
    capi.integrate_wait(ctx)
    for g, (d, geo) in zip(grids, before):
        assert (g.nx, g.ny, g.min_x, g.min_y) == geo
        assert np.array_equal(_bits(g.download()), _bits(d))
