"""GPU: the pruned sweep of row-mapped windows (csm_coarse_kernel, csm_prune_kernel, csm_sweep_tiles_kernel).

The device scores every coarse hypothesis but only the fine tiles whose coarse scores can still reach the
match's best fine score.  Every record must still be the reference's: on the bench's C2 geometry (where the
scored tiles must be a small part of the exhaustive sweep, so a silent fall-back to exhaustive scoring
fails), with equal fine maxima in different blocks and slices, with a threshold nothing beats, with flagged
(lower map edge) and unflagged matches in one batch, with forced near-edge fix-ups, and for the tables that
debug() returns after a pruned run."""
import numpy as np
import pytest

from my_lidar_graph_slam_b200 import capi, synth

pytestmark = pytest.mark.gpu

C2 = dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=1.0471975512, scan_range_max=5.7296)


def _run(ctx, grid, coarse, params, ins, thr=None):
    batch = capi.RtcsmBatch(ctx, **params)
    batch.upload(grid, capi.Scans([a for a, _, _ in ins], [s for _, s, _ in ins], [p for _, _, p in ins]), thr)
    batch.run(grid, coarse)
    return batch, batch.results(grid, coarse)


def _records_equal(R, refmap, pre, params, ins, outs, thr=None):
    for m, ((angles, scan, init), out) in enumerate(zip(ins, outs)):
        ref = R.rtcsm_match(refmap, angles, scan, init, pre=pre, thr=thr, **params)
        assert (out.found, out.ix, out.iy, out.it) == (ref.found, ref.ix, ref.iy, ref.it), f"match {m}"
        assert out.score == ref.score, f"match {m}"
        assert (out.win_x, out.win_y, out.win_t) == (ref.winX, ref.winY, ref.winT)


def _device_maps(ctx, refmap, low_res, apron=32):
    nx, ny, mx, my, res = refmap.geometry()
    grid = capi.Grid.from_dense(ctx, refmap.dense(), mx, my, res, apron=apron)
    return grid, grid.precompute(low_res)


def _c2_scene(n):
    """The bench's C2 workload: its map scans built into a reference map, n seeded matches."""
    import bench
    from oracle import backend
    R = backend()
    traj, map_scans, angles, ranges, inits = bench.c2_workload(n, seed=1)
    builder = R.RefBuilder()
    for p, r in zip(traj, map_scans):
        builder.append_scan(p, angles, r)
    refmap = builder.latest_map()
    return R, refmap, [(angles, r, p) for r, p in zip(ranges, inits)]


def _edge_map(rng):
    """A 128 x 128 map with strong structure along the lower x and y edges (SURVEY.md H12)."""
    dense = np.where(rng.random((128, 128)) < 0.25, rng.uniform(0.05, 0.95, (128, 128)), 0.0)
    dense[:12, :] = rng.uniform(0.5, 0.99, (12, 128))
    dense[:, :12] = rng.uniform(0.5, 0.99, (128, 12))
    return dense


def test_pruned_c2_batch_scores_few_tiles(ctx):
    R, refmap, ins = _c2_scene(16)
    pre = refmap.precompute(5)
    grid, coarse = _device_maps(ctx, refmap, 5)
    batch, outs = _run(ctx, grid, coarse, C2, ins)
    _records_equal(R, refmap, pre, C2, ins, outs)
    scored, total = batch.fine_tiles()
    assert total == sum(((2 * o.win_t + 1 + 1) // 2) * 5 for o in outs)   # theta pairs x 5 row groups
    assert 0 < scored < 0.1 * total, (scored, total)
    assert not any(o.exact_replay for o in outs)
    # work and n_scored still count the whole window the result is exact over
    hyp, _ = batch.work()
    assert hyp == sum(o.n_scored for o in outs) == sum((2 * o.win_t + 1) * (625 + 25) for o in outs)


def test_pruned_equal_maxima_take_the_first_visit(ctx):
    """A constant plateau: many hypotheses of different blocks and theta slices have the same, maximal
    score (same values summed in the same order), and their coarse scores tie with it."""
    from oracle import backend
    R = backend()
    dense = np.zeros((192, 192))
    dense[60:140, 60:140] = 0.75
    dense[90:94, 80:120] = 0.9               # a ridge: equal maxima only along it, in several slices
    refmap = R.RefMap.from_dense(dense, -4.8, -4.8)
    pre = refmap.precompute(5)
    grid, coarse = _device_maps(ctx, refmap, 5)
    angles = synth.beam_angles(8, 20.0)
    rng = np.random.default_rng(3)
    ins = [(angles, np.full(angles.shape, 0.05), np.array([0.0, 0.0, 0.0])),       # every hypothesis on the plateau
           (angles, np.full(angles.shape, 0.05), np.array([0.1, -0.2, 0.3]))]      # on the ridge
    for _ in range(3):
        ins.append((angles, rng.uniform(0.02, 0.15, angles.shape),
                    np.array([rng.uniform(-0.5, 0.5), rng.uniform(-0.4, 0.0), rng.uniform(-1, 1)])))
    params = dict(C2, range_theta=0.5)
    batch, outs = _run(ctx, grid, coarse, params, ins)
    _records_equal(R, refmap, pre, params, ins, outs)
    for m in (0, 1):
        fine, _, _ = batch.debug(m)
        assert outs[m].found and (fine == fine.max()).sum() > 1     # the winner had equal rivals


def test_pruned_threshold_nothing_beats(ctx):
    R, refmap, ins = _c2_scene(4)
    pre = refmap.precompute(5)
    grid, coarse = _device_maps(ctx, refmap, 5)
    batch, outs = _run(ctx, grid, coarse, C2, ins, thr=0.99)
    _records_equal(R, refmap, pre, C2, ins, outs, thr=0.99)
    assert not any(o.found for o in outs)
    scored, total = batch.fine_tiles()
    assert scored < 0.1 * total


def test_pruned_batch_mixes_flagged_and_unflagged_matches(ctx):
    """C2 matches, and the same scans moved next to the map's lower-left corner, where beams read the band
    of coarse indices in (-lowRes, 0): those matches are flagged and score every tile."""
    R, refmap, ins = _c2_scene(8)
    pre = refmap.precompute(5)
    grid, coarse = _device_maps(ctx, refmap, 5)
    nx, ny, mx, my, res = refmap.geometry()
    corner = [(a, s, np.array([mx + 0.4, my + 0.4, p[2]])) for a, s, p in ins[:4]]
    mixed = [x for pair in zip(ins[:4], corner) for x in pair]
    batch, outs = _run(ctx, grid, coarse, C2, mixed)
    _records_equal(R, refmap, pre, C2, mixed, outs)
    half, half_outs = _run(ctx, grid, coarse, C2, mixed[0::2])
    assert [(o.found, o.ix, o.iy, o.it, o.score) for o in half_outs] == \
        [(o.found, o.ix, o.iy, o.it, o.score) for o in outs[0::2]]
    # the unflagged half scores the same tiles alone as in the mixed batch; the flagged half adds all of its own
    scored, total = batch.fine_tiles()
    half_scored, half_total = half.fine_tiles()
    assert 0 < half_scored < 0.1 * half_total
    assert scored == half_scored + (total - half_total)


def test_pruned_with_forced_near_edge_fixups(ctx):
    R, refmap, ins = _c2_scene(6)
    pre = refmap.precompute(5)
    grid, coarse = _device_maps(ctx, refmap, 5)
    try:
        ctx.set_edge_eps(0.3)
        batch, outs = _run(ctx, grid, coarse, C2, ins)
    finally:
        ctx.set_edge_eps(0.0)            # restores the default band
    assert sum(o.n_fixups for o in outs) > 100
    _records_equal(R, refmap, pre, C2, ins, outs)
    scored, total = batch.fine_tiles()
    assert scored < total


def test_debug_after_pruned_run_returns_the_reference_tables(ctx):
    R, refmap, ins = _c2_scene(3)
    pre = refmap.precompute(5)
    grid, coarse = _device_maps(ctx, refmap, 5)
    batch, outs = _run(ctx, grid, coarse, C2, ins)
    scored, total = batch.fine_tiles()
    assert scored < total
    for m, (angles, scan, init) in enumerate(ins):
        ref = R.rtcsm_match(refmap, angles, scan, init, pre=pre, **C2)
        fine, coarse_t, _ = batch.debug(m)
        nt, nyw, nxw = fine.shape
        tab, _, _ = R.rtcsm_score_table(refmap, pre, False, 5, C2["scan_range_max"], init, angles, scan,
                                        ref.stepT, ref.winT, -ref.winX, nxw, -ref.winY, nyw)
        assert np.array_equal(tab.view(np.int64), fine.view(np.int64)), f"fine table of match {m}"
        ctab, _, _ = R.rtcsm_score_table(refmap, pre, True, 5, C2["scan_range_max"], init, angles, scan,
                                         ref.stepT, ref.winT, -ref.winX, nxw, -ref.winY, nyw)
        ref_coarse = ctab[:, ::5, ::5].transpose(0, 2, 1)
        assert np.array_equal(ref_coarse.view(np.int64), coarse_t.view(np.int64)), f"coarse table of match {m}"
    # the records of results() after debug() are unchanged
    again = batch.results(grid, coarse)
    assert [(o.found, o.ix, o.iy, o.it, o.score) for o in again] == [(o.found, o.ix, o.iy, o.it, o.score) for o in outs]
