"""GPU: the theta-grouped row sweep (csm_sweep_rows_kernel) against the reference's exhaustive score tables.

A thread of the row sweep scores a group of consecutive theta slices and shares map loads between them.
Every fine and coarse score of every slice must still be the reference's, bit for bit, where groups are
cut short (nT is odd, so the last group of every match is partial), where the matches of one batch have
different nT, where the window has rows == 4 and a short last row group, and where scans hang off the
map (clamped offsets that read the zero apron)."""
import numpy as np
import pytest

from my_lidar_graph_slam_b200 import capi, synth

pytestmark = pytest.mark.gpu


def _tables_equal(R, refmap, pre, batch, outs, params, ins):
    L = params["low_res"]
    for m, (angles, scan, init) in enumerate(ins):
        ref = R.rtcsm_match(refmap, angles, scan, init, pre=pre, **params)
        out = outs[m]
        assert (out.win_x, out.win_y, out.win_t, out.step_t) == (ref.winX, ref.winY, ref.winT, ref.stepT)
        assert (out.found, out.ix, out.iy, out.it) == (ref.found, ref.ix, ref.iy, ref.it)
        assert out.score == ref.score
        fine, coarse, _ = batch.debug(m)
        nt, nyw, nxw = fine.shape
        assert nt == 2 * ref.winT + 1
        tab, _, _ = R.rtcsm_score_table(refmap, pre, False, L, params["scan_range_max"], init, angles, scan,
                                        ref.stepT, ref.winT, -ref.winX, nxw, -ref.winY, nyw)
        assert np.array_equal(tab.view(np.int64), fine.view(np.int64)), f"fine table of match {m}"
        ctab, _, _ = R.rtcsm_score_table(refmap, pre, True, L, params["scan_range_max"], init, angles, scan,
                                         ref.stepT, ref.winT, -ref.winX, nxw, -ref.winY, nyw)
        ref_coarse = ctab[:, ::L, ::L].transpose(0, 2, 1)        # [t][bx][by]
        assert np.array_equal(ref_coarse.view(np.int64), coarse.view(np.int64)), f"coarse table of match {m}"


def _run(ctx, grid, coarse, params, ins):
    batch = capi.RtcsmBatch(ctx, **params)
    batch.upload(grid, capi.Scans([a for a, _, _ in ins], [s for _, s, _ in ins], [p for _, _, p in ins]))
    batch.run(grid, coarse)
    return batch, batch.results(grid, coarse)


def _edge_scene(rng):
    """A 128 x 128 map with strong structure along all four edges, and scans of different maximum range
    (so different theta steps and nT) from poses near the edges, many beams leaving the map."""
    from oracle import backend
    R = backend()
    ny, nx = 128, 128
    dense = np.where(rng.random((ny, nx)) < 0.3, rng.uniform(0.05, 0.95, (ny, nx)), 0.0)
    for sl in (np.s_[:10, :], np.s_[-10:, :], np.s_[:, :10], np.s_[:, -10:]):
        dense[sl] = rng.uniform(0.5, 0.99, dense[sl].shape)
    refmap = R.RefMap.from_dense(dense, -1.0, -2.0)
    angles = synth.beam_angles(181, 180.0)
    ins = []
    for k, max_r in enumerate((0.6, 1.5, 2.5, 4.0, 0.9, 3.2)):
        ranges = rng.uniform(0.1, max_r, angles.shape)
        corner = k % 4
        x = -1.0 + (rng.uniform(0.0, 0.4) if corner in (0, 3) else 6.4 - rng.uniform(0.0, 0.4))
        y = -2.0 + (rng.uniform(0.0, 0.4) if corner in (0, 1) else 6.4 - rng.uniform(0.0, 0.4))
        heading = np.arctan2(-2.0 + 3.2 - y, -1.0 + 3.2 - x) + np.pi + rng.uniform(-0.4, 0.4)   # away from the centre
        ins.append((angles, ranges, np.array([x, y, heading])))
    return R, refmap, ins


@pytest.mark.parametrize("params", [
    dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=0.5, scan_range_max=20.0),    # rows 5
    dict(low_res=3, range_x=1.5, range_y=1.0, range_theta=0.4, scan_range_max=20.0),    # rows 4, 21 rows, 2 x chunks
    dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=0.02, scan_range_max=20.0),   # nT = 3: one partial group
])
def test_theta_groups_match_reference_tables_off_the_map(ctx, params):
    R, refmap, ins = _edge_scene(np.random.default_rng(21))
    pre = refmap.precompute(params["low_res"])
    nx, ny, mx, my, res = refmap.geometry()
    grid = capi.Grid.from_dense(ctx, refmap.dense(), mx, my, res, apron=48)
    coarse = grid.precompute(params["low_res"])
    batch, outs = _run(ctx, grid, coarse, params, ins)
    nts = {batch.debug(m)[0].shape[0] for m in range(len(ins))}
    assert len(nts) > 1 or params["range_theta"] < 0.05       # matches of different nT in one batch
    _tables_equal(R, refmap, pre, batch, outs, params, ins)


def test_theta_groups_room_scene_different_ranges(ctx):
    """C2 window on a room map; scans cut to different maximum ranges give different nT in one batch."""
    from oracle import backend
    from scenes import room_scene
    R = backend()
    world, angles, traj, builder = room_scene(seed=4)
    refmap = builder.latest_map()
    params = dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=1.0471975512, scan_range_max=5.7296)
    pre = refmap.precompute(5)
    nx, ny, mx, my, res = refmap.geometry()
    grid = capi.Grid.from_dense(ctx, refmap.dense(), mx, my, res, apron=32)
    coarse = grid.precompute(5)
    rng = np.random.default_rng(5)
    ins = []
    for k, cut in enumerate((None, 2.0, 3.5, None, 1.2)):
        true = traj[3 + k]
        scan = synth.make_scan(world, true, angles, np.random.default_rng(50 + k))
        if cut is not None:
            scan = np.minimum(scan, cut)
        init = true + np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3), rng.uniform(-0.2, 0.2)])
        ins.append((angles, scan, init))
    batch, outs = _run(ctx, grid, coarse, params, ins)
    assert len({batch.debug(m)[0].shape[0] for m in range(len(ins))}) >= 3
    _tables_equal(R, refmap, pre, batch, outs, params, ins)


def test_theta_groups_near_edge_fixups_reread_patched_offsets(ctx):
    """A widened edge band sends many points through the host re-derivation, which patches the offsets and
    runs the sweep again: the grouped sweep must read the patched values and give the un-widened answer."""
    params = dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=0.5, scan_range_max=20.0)
    R, refmap, ins = _edge_scene(np.random.default_rng(22))
    pre = refmap.precompute(5)
    nx, ny, mx, my, res = refmap.geometry()
    grid = capi.Grid.from_dense(ctx, refmap.dense(), mx, my, res, apron=48)
    coarse = grid.precompute(5)
    plain, plain_outs = _run(ctx, grid, coarse, params, ins)
    try:
        ctx.set_edge_eps(0.3)
        wide, wide_outs = _run(ctx, grid, coarse, params, ins)
    finally:
        ctx.set_edge_eps(0.0)            # restores the default band
    assert sum(o.n_fixups for o in wide_outs) > 100
    assert sum(o.n_fixups for o in plain_outs) < sum(o.n_fixups for o in wide_outs)
    for m in range(len(ins)):
        a, b = plain_outs[m], wide_outs[m]
        assert (a.found, a.ix, a.iy, a.it, a.score) == (b.found, b.ix, b.iy, b.it, b.score)
        fa, ca, cells_a = plain.debug(m)
        fb, cb, cells_b = wide.debug(m)
        assert np.array_equal(cells_a, cells_b)
        assert np.array_equal(fa.view(np.int64), fb.view(np.int64))
        assert np.array_equal(ca.view(np.int64), cb.view(np.int64))
    _tables_equal(R, refmap, pre, wide, wide_outs, params, ins)
