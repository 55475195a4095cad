"""GPU parity: lgs_grid_integrate_many / lgs_pyramid_create_many (many maps in one call) against the oracle's
ConstructMapFromScans and against one lgs_grid_integrate_scans / lgs_pyramid_create call per map (every
cell bit-exact)."""
import numpy as np
import pytest

from my_lidar_graph_slam_b200 import capi, synth

pytestmark = pytest.mark.gpu

PRE_PASS_LAUNCHES = 2          # sensor cells + beam end cells
ROUND_LAUNCHES = 4             # mark, pairs, touch, fold


def _bits(a):
    return np.ascontiguousarray(a).view(np.int64)


def _random_maps(seed, scan_counts, beams=300):
    """Maps of different size, resolution and apron; scans of random rays that end inside the map, with
    some scans that have no hits."""
    rng = np.random.default_rng(seed)
    shapes = [(128, 96), (200, 160), (64, 64), (300, 120), (96, 256), (160, 160), (72, 200)]
    maps = []
    for k, n_scans in enumerate(scan_counts):
        nx, ny = shapes[k % len(shapes)]
        res = (0.05, 0.1, 0.025)[k % 3]
        apron = (1, 2, 4, 7)[k % 4]
        mx, my = rng.uniform(-20.0, 20.0, 2)
        sensors, hits = [], []
        for s in range(n_scans):
            sensor = np.array([mx + rng.uniform(0.2, 0.8) * nx * res, my + rng.uniform(0.2, 0.8) * ny * res])
            nb = 0 if s % 17 == 5 else beams
            ang = np.sort(rng.uniform(-np.pi, np.pi, nb))
            rad = rng.uniform(0.0, 0.7, nb) * max(nx, ny) * res
            h = sensor[None, :] + rad[:, None] * np.stack([np.cos(ang), np.sin(ang)], 1)
            h[:, 0] = np.clip(h[:, 0], mx + 1e-3, mx + nx * res - 1e-3)
            h[:, 1] = np.clip(h[:, 1], my + 1e-3, my + ny * res - 1e-3)
            sensors.append(sensor)
            hits.append(np.ascontiguousarray(h.reshape(nb, 2)))
        maps.append(dict(geo=(nx, ny, mx, my, res), apron=apron, sensors=np.asarray(sensors).reshape(-1, 2),
                         hits=hits))
    return maps


def _grids(ctx, maps):
    return [capi.Grid(ctx, *m["geo"], apron=m["apron"]) for m in maps]


def _per_map(ctx, maps, grids):
    return [capi.integrate_scans(ctx, g, m["sensors"], m["hits"]) for g, m in zip(grids, maps)]


def _many(ctx, maps, grids, order=None):
    order = list(range(len(maps))) if order is None else list(order)
    got = capi.integrate_many(ctx, [grids[i] for i in order], [maps[i]["sensors"] for i in order],
                              [maps[i]["hits"] for i in order])
    counts = np.zeros(len(maps), dtype=np.int64)
    counts[order] = got
    return counts


def test_loop_closure_rebuild_matches_construct_map(ctx):
    """GridMapBuilder::AfterLoopClosure: every local map rebuilt from corrected poses, all in one call, against
    ConstructMapFromScans per map (cells and Update counts), in ONE round of launches."""
    from oracle import backend
    R = backend()
    world = synth.RoomsWorld(40.0, 5.0, seed=41)
    angles = synth.beam_angles(1081, 270.0)
    traj = synth.trajectory(world, 72, step=0.25, seed=41)
    noise = np.random.default_rng(42)
    scans = [synth.make_scan(world, p, angles, noise) for p in traj]
    builder = R.RefBuilder(travel_thr=2.0)
    for p, r in zip(traj, scans):
        builder.append_scan(p, angles, r)
    spans = [builder.local_map_nodes(i) for i in range(builder.num_local_maps())]
    assert len(spans) >= 8
    # the optimiser's correction: every node moves a little
    corrected = traj + np.random.default_rng(43).normal(0.0, [0.04, 0.04, 0.01], traj.shape)
    rebuilt = R.RefBuilder(travel_thr=2.0)
    for p, r in zip(corrected, scans):
        rebuilt.append_node_only(p, angles, r)
    hits = [capi.scan_hit_points(p, angles, r, 0.02, 20.0)[0] for p, r in zip(corrected, scans)]
    refs, want, grids = [], [], []
    for lo, hi in spans:
        ref = rebuilt.construct_map(lo, hi)
        nx, ny, mx, my, res = ref.geometry()
        replay = R.RefMap.from_dense(np.zeros((ny, nx)), mx, my)
        want.append(sum(R.map_integrate_hits(replay, corrected[k][:2], hits[k]) for k in range(lo, hi + 1)))
        assert np.array_equal(_bits(replay.dense()), _bits(ref.dense()))
        refs.append(ref)
        grids.append(capi.Grid(ctx, nx, ny, mx, my, res, apron=2))
    assert max(hi - lo + 1 for lo, hi in spans) <= 64
    before = ctx.launch_count()
    got = capi.integrate_many(ctx, grids, [corrected[lo:hi + 1, :2] for lo, hi in spans],
                              [hits[lo:hi + 1] for lo, hi in spans])
    assert ctx.launch_count() - before == PRE_PASS_LAUNCHES + ROUND_LAUNCHES
    assert got.tolist() == want
    for i, (g, ref) in enumerate(zip(grids, refs)):
        assert np.array_equal(_bits(g.download()), _bits(ref.dense())), f"local map {i}"


def test_many_equals_per_map_calls_over_several_rounds(ctx):
    """Maps of 0, 1, 63, 64, 65 and 200 scans (several rounds, rounds that hold fewer maps than the first),
    of different size, resolution and apron, with hitless scans, passed in a shuffled order."""
    maps = _random_maps(7, [0, 1, 63, 64, 65, 200, 3])
    solo, many = _grids(ctx, maps), _grids(ctx, maps)
    want = _per_map(ctx, maps, solo)
    order = np.random.default_rng(8).permutation(len(maps))
    before = ctx.launch_count()
    got = _many(ctx, maps, many, order)
    assert ctx.launch_count() - before == PRE_PASS_LAUNCHES + 4 * ROUND_LAUNCHES   # the 200-scan map: 4 chunks
    assert got.tolist() == want and want[0] == 0 and min(want[1:]) > 0
    for i, (a, b) in enumerate(zip(solo, many)):
        assert np.array_equal(_bits(a.download()), _bits(b.download())), f"map {i}"
    # again on top of the maps (the fold reads what the first call left), and an empty call
    want = _per_map(ctx, maps, solo)
    assert _many(ctx, maps, many).tolist() == want
    for i, (a, b) in enumerate(zip(solo, many)):
        assert np.array_equal(_bits(a.download()), _bits(b.download())), f"map {i}, second pass"
    assert capi.integrate_many(ctx, [], [], []).tolist() == []
    assert capi.integrate_many(ctx, many[:2], [np.zeros((0, 2))] * 2, [[], []]).tolist() == [0, 0]


def test_very_long_rays_split_the_round(ctx):
    """Rays of 2000-4000 cells over 24 wide maps: their record bounds exceed one round's budget, so the chunks
    are spread over more than one round -- results as with one call per map."""
    rng = np.random.default_rng(31)
    nx, ny = 4480, 448
    maps = []
    for k in range(24):
        sensors, hits = [], []
        for s in range(8):
            sensor = np.array([rng.uniform(1.0, 12.0), rng.uniform(8.0, 14.0)])
            ang = np.sort(rng.uniform(-0.04, 0.04, 64))
            rad = np.where(rng.random(64) < 0.7, rng.uniform(110.0, 205.0, 64), rng.uniform(0.3, 40.0, 64))
            h = sensor[None, :] + rad[:, None] * np.stack([np.cos(ang), np.sin(ang)], 1)
            h[:, 0] = np.clip(h[:, 0], 0.01, nx * 0.05 - 0.01)
            h[:, 1] = np.clip(h[:, 1], 0.01, ny * 0.05 - 0.01)
            sensors.append(sensor)
            hits.append(np.ascontiguousarray(h))
        maps.append(dict(geo=(nx, ny, 0.0, 0.0, 0.05), apron=1, sensors=np.asarray(sensors), hits=hits))
    solo, many = _grids(ctx, maps), _grids(ctx, maps)
    want = _per_map(ctx, maps, solo)
    before = ctx.launch_count()
    assert _many(ctx, maps, many).tolist() == want
    rounds = (ctx.launch_count() - before - PRE_PASS_LAUNCHES) // ROUND_LAUNCHES
    assert 2 <= rounds < len(maps)
    for i, (a, b) in enumerate(zip(solo, many)):
        assert np.array_equal(_bits(a.download()), _bits(b.download())), f"map {i}"


def _scene_maps(seeds, n):
    maps = []
    for seed in seeds:
        world = synth.RoomsWorld(40.0, 5.0, seed=seed)
        angles = synth.beam_angles(1081, 270.0)
        traj = synth.trajectory(world, n, step=0.25, seed=seed)
        noise = np.random.default_rng(seed + 1)
        geo = capi.Geometry(0, 0, traj[0][0], traj[0][1], 0.05, 64)
        hits = []
        for p in traj:
            h, bbox = capi.scan_hit_points(p, angles, synth.make_scan(world, p, angles, noise), 0.02, 20.0)
            geo, _, _, _ = capi.geometry_expand(geo, bbox)
            hits.append(h)
        maps.append(dict(geo=geo.as_tuple(), apron=1, sensors=traj[:, :2], hits=hits))
    return maps


def test_exhausted_side_buffer_falls_back_across_maps(ctx):
    """With the side buffer shrunk to nothing, long mixed sequences of every map take the exhaustive path of the
    fold; the maps stay identical to per-map calls with the default buffer."""
    maps = _scene_maps([11, 12, 13], 12)
    solo, many = _grids(ctx, maps), _grids(ctx, maps)
    want = _per_map(ctx, maps, solo)
    ctx.set_option("integ_side_words", 8)
    try:
        before = capi.lib().lgs_ctx_integrate_fallback_cells(ctx.h)
        assert _many(ctx, maps, many).tolist() == want
        assert capi.lib().lgs_ctx_integrate_fallback_cells(ctx.h) > before
    finally:
        ctx.set_option("integ_side_words", 0)
    for i, (a, b) in enumerate(zip(solo, many)):
        assert np.array_equal(_bits(a.download()), _bits(b.download())), f"map {i}"


def test_a_scan_outside_its_grid_fails_the_whole_call(ctx):
    maps = _random_maps(21, [5, 9, 4, 6])
    grids = _grids(ctx, maps)
    _many(ctx, maps, grids)
    before = [g.download() for g in grids]
    bad = [list(m["hits"]) for m in maps]
    nx, ny, mx, my, res = maps[2]["geo"]
    bad[2][1] = np.vstack([bad[2][1], [[mx + nx * res + 1.0, my + 0.5]]])
    with pytest.raises(capi.LgsError, match=r"map 2, scan 1 touches cells outside"):
        capi.integrate_many(ctx, grids, [m["sensors"] for m in maps], bad)
    for i, (g, b) in enumerate(zip(grids, before)):
        assert np.array_equal(_bits(g.download()), _bits(b)), f"map {i} changed"


def test_rejections(ctx):
    maps = _random_maps(22, [3, 4])
    grids = _grids(ctx, maps)
    sensors, hits = [m["sensors"] for m in maps], [m["hits"] for m in maps]
    with pytest.raises(capi.LgsError, match="twice"):
        capi.integrate_many(ctx, [grids[0], grids[0]], [sensors[0]] * 2, [hits[0]] * 2)
    windowed = capi.Grid(ctx, *maps[1]["geo"], apron=1)
    windowed.set_window(16, 0)
    with pytest.raises(capi.LgsError, match="windowed"):
        capi.integrate_many(ctx, [grids[0], windowed], sensors, hits)
    # a submitted call not yet waited for
    pending = capi.Grid(ctx, *maps[0]["geo"], apron=1)
    capi.integrate_submit(ctx, pending, capi.PackedHits(sensors[0], hits[0]))
    with pytest.raises(capi.LgsError, match="in flight"):
        capi.integrate_many(ctx, grids, sensors, hits)
    assert capi.integrate_wait(ctx) > 0
    solo = _grids(ctx, maps)
    want = _per_map(ctx, maps, solo)
    assert capi.integrate_many(ctx, grids, sensors, hits).tolist() == want
    for a, b in zip(solo, grids):
        assert np.array_equal(_bits(a.download()), _bits(b.download()))


@pytest.mark.skipif(capi.device_count() < 2, reason="needs a second GPU")
def test_grids_on_another_device_are_refused(ctx):
    """The one-map and the batched calls, integration and pyramids alike, refuse a grid of another device."""
    maps = _random_maps(25, [3])
    sensors, hits = maps[0]["sensors"], maps[0]["hits"]
    other = capi.Context(1)
    try:
        g = capi.Grid(other, *maps[0]["geo"], apron=1)
        calls = [lambda: capi.integrate_scans(ctx, g, sensors, hits),
                 lambda: capi.integrate_submit(ctx, g, capi.PackedHits(sensors, hits)),
                 lambda: capi.integrate_many(ctx, [g], [sensors], [hits]),
                 lambda: capi.Pyramid(ctx, g, 3),
                 lambda: capi.Pyramid.create_many(ctx, [g], 3)]
        for call in calls:
            with pytest.raises(capi.LgsError, match="lives on device 1"):
                call()
        assert capi.integrate_wait(ctx) == 0
        assert not g.download().any()
    finally:
        other.close()


def test_grids_of_another_context(ctx):
    """Grids owned by a second context of the same device (e.g. the builder's), ordered like lgs_grid_copy:
    the owner's pending uploads come first."""
    maps = _random_maps(23, [10, 70, 1])
    other = capi.Context(0)
    try:
        rng = np.random.default_rng(24)
        seeds = [np.where(rng.random((m["geo"][1], m["geo"][0])) < 0.2, 0.7, 0.0) for m in maps]
        foreign = [capi.Grid.from_dense(other, d, *m["geo"][2:], apron=m["apron"]) for d, m in zip(seeds, maps)]
        solo = [capi.Grid.from_dense(ctx, d, *m["geo"][2:], apron=m["apron"]) for d, m in zip(seeds, maps)]
        want = _per_map(ctx, maps, solo)
        assert _many(ctx, maps, foreign).tolist() == want
        for a, b in zip(solo, foreign):
            assert np.array_equal(_bits(a.download()), _bits(b.download()))
    finally:
        other.close()


@pytest.mark.parametrize("height", [0, 3, 7])
def test_pyramid_create_many_matches_single_builds_and_the_oracle(ctx, height):
    """Grids of different size and apron, some smaller than the largest window 2^height, one empty."""
    from oracle import backend
    R = backend()
    rng = np.random.default_rng(50 + height)
    shapes = [(64, 64), (64, 192), (128, 64), (320, 256), (64, 128)]
    dense = [np.where(rng.random(s) < 0.3, rng.uniform(0.001, 0.999, s), 0.0) for s in shapes]
    grids = [capi.Grid.from_dense(ctx, d, -3.2 + k, 1.6 - k, 0.05, apron=(1, 2, 4, 9, 3)[k])
             for k, d in enumerate(dense)]
    grids.append(capi.Grid(ctx, 0, 0, 0.0, 0.0, 0.05, apron=3))
    before = ctx.launch_count()
    pyrs = capi.Pyramid.create_many(ctx, grids, height)
    assert ctx.launch_count() - before == height + 2          # apron clear, level 0, one launch per level
    for k, (g, d) in enumerate(zip(grids, dense)):
        single = capi.Pyramid(ctx, g, height)
        ref = R.RefMap.from_dense(d, -3.2 + k, 1.6 - k).pyramid(height)
        for h in range(height + 1):
            got = pyrs[k].download(h)
            assert np.array_equal(_bits(got), _bits(single.download(h))), f"grid {k} level {h}"
            assert np.array_equal(_bits(got), _bits(ref[h].dense())), f"grid {k} level {h} vs oracle"
    assert capi.lib().lgs_pyramid_levels(pyrs[-1].h) == height + 1
    for p in pyrs:
        p.close()
    assert capi.Pyramid.create_many(ctx, [], height) == []


def test_branch_and_bound_on_batched_pyramids(ctx):
    """A loop-detection batch over create_many pyramids returns the records of one over separately built ones
    (the aprons, which the search reads beyond the map edges, are zero too)."""
    from oracle import backend
    R = backend()
    world = synth.World(16.0, 16.0, 5, seed=4)
    angles = synth.beam_angles(361, 180.0)
    traj = synth.trajectory(world, 24, step=0.2, seed=4)
    noise = np.random.default_rng(5)
    builder = R.RefBuilder(travel_thr=1.0)
    for p in traj[:20]:
        builder.append_scan(p, angles, synth.make_scan(world, p, angles, noise))
    grids = []
    for i in range(builder.num_local_maps()):
        m = builder.local_map(i)
        nx, ny, mx, my, res = m.geometry()
        grids.append(capi.Grid.from_dense(ctx, m.dense(), mx, my, res, apron=2))
    assert len(grids) >= 3
    # dirty pool memory first: an all-ones pyramid of every size, freed
    for g in grids:
        ones = capi.Grid.from_dense(ctx, np.full((g.ny, g.nx), 0.999), g.min_x, g.min_y, g.res, apron=2)
        capi.Pyramid(ctx, ones, 6).close()
    many = capi.Pyramid.create_many(ctx, grids, 6)
    single = [capi.Pyramid(ctx, g, 6) for g in grids]
    queries = [synth.make_scan(world, traj[20 + k % 4], angles, np.random.default_rng(60 + k)) for k in range(len(grids))]
    inits = [traj[20 + k % 4] + np.array([0.3, -0.2, 0.05]) for k in range(len(grids))]
    scans = capi.Scans([angles] * len(grids), queries, inits, range_min=0.02, range_max=30.0)
    out = []
    for pyrs in (many, single):
        batch = capi.BbBatch(ctx, node_height_max=6, range_x=2.0, range_y=2.0, range_theta=0.4)
        batch.upload(scans, pyrs, 0.2)
        batch.run()
        out.append((batch.results_array(), batch.records()))
        batch.close()
    assert np.array_equal(out[0][0], out[1][0])
    assert np.array_equal(out[0][1], out[1][1])
