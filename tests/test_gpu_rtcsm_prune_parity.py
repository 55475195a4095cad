"""GPU: the pruned correlative sweep (csm_project_kernel's flag, csm_coarse_kernel, csm_prune_kernel,
csm_sweep_tiles_kernel, csm_select_kernel) against its CPU model (test_rtcsm_prune_model), tile for tile.

Correct records alone cannot tell a right pruned sweep from one that scores too much: a bound that is too
low, a flag that fires too often or a tile map that lists extra tiles all give the reference's answer, only
slower.  So every match here is checked twice: its record is bit-identical to the reference's, and the number
of warp tiles the device scored equals the model's count from the reference's own fine and coarse tables.
The windows cover the shapes where the index arithmetic differs (one-cell blocks, blocks across a 32-lane x
chunk or a row group, tall windows, fewer coarse blocks than seeds, 512 fine hypotheses per slice and just
under); batches mix ragged scans, flagged and unflagged matches and per-match thresholds, including one at a
match's best score; the flattened exhaustive kernel and the exhaustive row sweep give the same tables; and a
batch reused across grids, results() calls and uploads follows its new inputs."""
import functools

import numpy as np
import pytest

from my_lidar_graph_slam_b200 import capi, synth
from test_rtcsm_prune_model import _blocks, band_edge_scene, flagged, model_select, near_edge

pytestmark = pytest.mark.gpu

RES = 0.05
TINY = float(np.finfo(np.float64).tiny)     # the 1-argument overload's threshold (DBL_MIN)
APRON = 48                                  # >= every window side below (42 for the tall case)

# Window cases at res 0.05: parameters, and (nbx, nby, nxw, nyw, rows, x chunks) they must give; rows = 0 is
# the flattened kernel.  ceil(0.5 * range / res) decides the shapes, so they are asserted, not assumed.
CASES = {
    "low_res1": (dict(low_res=1, range_x=1.5, range_y=1.0), (31, 21, 31, 21, 4, 1)),      # nbx = nxw
    "low_res3_two_chunks": (dict(low_res=3, range_x=1.5, range_y=1.0), (11, 7, 33, 21, 4, 2)),
    "low_res7_block_across_x32": (dict(low_res=7, range_x=1.5, range_y=0.7), (5, 3, 35, 21, 4, 2)),
    "low_res2_tall": (dict(low_res=2, range_x=0.6, range_y=2.0), (7, 21, 14, 42, 4, 1)),
    "low_res32_fewer_blocks_than_seeds": (dict(low_res=32, range_x=1.0, range_y=1.0, range_theta=0.01),
                                          (1, 1, 32, 32, 4, 1)),
    "low_res32_map_thinner_than_a_block": (dict(low_res=32, range_x=1.0, range_y=1.0, range_theta=0.01,
                                                scan_range_max=1.5), (1, 1, 32, 32, 4, 1)),
    "exactly_512": (dict(low_res=2, range_x=0.7, range_y=1.5), (8, 16, 16, 32, 4, 1)),
    "just_under_512": (dict(low_res=2, range_x=0.6, range_y=1.7), (7, 18, 14, 36, 0, 1)),
    "c2": (dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=1.0471975512, scan_range_max=5.7296),
           (5, 5, 25, 25, 5, 1)),
}
DEFAULTS = dict(range_theta=0.1, scan_range_max=5.0)


# ---- scenes ----------------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=1)
def _rooms():
    """Two by two 5 m rooms (synth.RoomsWorld), rasterised and cropped to 208 x 208 cells so that the outer
    walls lie 2-5 cells inside the map on every side.  Scans near the upper-right corner then read past the
    upper and right map edges; scans near the lower-left corner put cells in the band (-lowRes, 0) of coarse
    indices.  -> (world, dense, min_x, min_y)."""
    world = synth.RoomsWorld(10.0, 5.0, seed=3)
    angles = synth.beam_angles(361, 270.0)
    poses = np.array([[x, y, th] for x in (-2.5, 2.5) for y in (-2.5, 2.5) for th in (0.3, 2.0)])
    noise = np.random.default_rng(5)
    dense, mx, my = synth.rasterize_map(poses, angles, [synth.make_scan(world, p, angles, noise) for p in poses])
    k = int(round((-5.15 - mx) / RES))
    return world, np.ascontiguousarray(dense[k:k + 208, k:k + 208]), mx + k * RES, my + k * RES


def _scene_map(R, thin):
    """-> (dense, min_x, min_y, RefMap): the rooms map, or 16 of its rows with the upper wall at row 15 (a map
    thinner than a 32-cell block)."""
    _, dense, mx, my = _rooms()
    if thin:
        dense, my = np.ascontiguousarray(dense[-20:-4]), my + (dense.shape[0] - 20) * RES
    return dense, mx, my, R.RefMap.from_dense(dense, mx, my, RES, 16)


def _scan(world, rng, lo, hi, n_beams=361, fov=270.0, heading=(-np.pi, np.pi)):
    """A scan taken at a random pose in [lo, hi]^2 and its perturbed initial pose -> (angles, ranges, init)."""
    angles = synth.beam_angles(n_beams, fov)
    true = np.array([rng.uniform(lo, hi), rng.uniform(lo, hi), rng.uniform(*heading)])
    ranges = synth.make_scan(world, true, angles, rng)
    return angles, ranges, true + np.array([rng.uniform(-0.2, 0.2), rng.uniform(-0.2, 0.2), rng.uniform(-0.05, 0.05)])


def _case_scans(thin, seed=11):
    """Three scans in the upper-right room (against the upper and right map edges, too far from the lower-left
    edges for any kept beam to reach them), two near the lower-left corner, and one in the upper-right room
    whose initial pose is 0.8 m left of where the scan fits best."""
    world = _rooms()[0]
    rng = np.random.default_rng(seed)
    if thin:        # below the upper wall, 50 degree scans facing it: every kept cell at rows >= 10
        return [_scan(world, rng, 4.2, 4.5, n, 50.0, (1.5, 1.65)) for n in (181, 241, 361)]
    ins = ([_scan(world, rng, 2.0, 4.5, n) for n in (181, 241, 361)] +
           [_scan(world, rng, -4.6, -3.6, n) for n in (181, 361)])
    angles = synth.beam_angles(241, 270.0)
    true = np.array([rng.uniform(2.5, 3.5), rng.uniform(2.5, 3.5), rng.uniform(-np.pi, np.pi)])
    return ins + [(angles, synth.make_scan(world, true, angles, rng), true - (0.8, 0.0, 0.0))]


# ---- the model of one match ------------------------------------------------------------------------------

class Model:
    """Reference record, tables and the model's flag and tile count of one match."""

    def __init__(self, R, refmap, pre, params, angles, ranges, init, thr, eps):
        self.ref = ref = R.rtcsm_match(refmap, angles, ranges, init, pre=pre, thr=thr, **params)
        L = self.L = params["low_res"]
        self.nxw, self.nyw = ((2 * ref.winX) // L + 1) * L, ((2 * ref.winY) // L + 1) * L
        args = (L, params["scan_range_max"], init, angles, ranges, ref.stepT, ref.winT, -ref.winX, self.nxw,
                -ref.winY, self.nyw)
        self.fine, idx, cnt = R.rtcsm_score_table(refmap, pre, False, *args)
        self.coarse, _, _ = R.rtcsm_score_table(refmap, pre, True, *args)
        nx, ny, mx, my, res = refmap.geometry()
        kept = ranges < params["scan_range_max"]
        self.cells = idx[:, :cnt[0]]
        edge = near_edge(init, angles[kept], ranges[kept], ref.stepT, ref.winT, mx, my, res, eps)
        geo = (ref.winX, ref.winY, self.nxw, self.nyw, L, nx, ny)
        self.basic_flag = flagged(self.cells, *geo)
        self.flag = flagged(self.cells, *geo, edge)
        self.thr_abs = (TINY if thr is None else thr) * len(ranges)
        found, ix, iy, it, score, self.n, self.total = model_select(self.fine, self.coarse, L, self.thr_abs, self.flag)
        assert found == ref.found
        if found:
            assert (ix - ref.winX, iy - ref.winY, it - ref.winT, score) == (ref.ix, ref.iy, ref.it, ref.score)
        F, C, _ = _blocks(self.fine, self.coarse, L)
        assert self.flag or (C >= F).all(), "a coarse score below its block in an unflagged match"
        self.nB = C.size
        # some kept point's window reads past the upper or right map edge
        self.overhang = cnt[0] > 0 and bool((self.cells[..., 0] + self.nxw - ref.winX > nx).any() or
                                            (self.cells[..., 1] + self.nyw - ref.winY > ny).any())


def _models(R, refmap, pre, params, ins, thrs, eps):
    return [Model(R, refmap, pre, params, a, r, p, t, eps) for (a, r, p), t in zip(ins, thrs)]


# ---- device runs -----------------------------------------------------------------------------------------

def _device_maps(ctx, dense, mx, my, low_res, pre):
    grid = capi.Grid.from_dense(ctx, dense, mx, my, RES, apron=APRON)
    coarse = grid.precompute(low_res)
    assert np.array_equal(coarse.download().view(np.int64), pre.dense().view(np.int64)), "coarse map"
    return grid, coarse


def _thr_arg(thrs):
    return None if all(t is None for t in thrs) else [TINY if t is None else t for t in thrs]


def _run(ctx, grid, coarse, params, ins, thrs, batch=None):
    """upload, run, results -> (batch, records, fine_tiles() read before any debug())."""
    batch = batch or capi.RtcsmBatch(ctx, **params)
    batch.upload(grid, capi.Scans([a for a, _, _ in ins], [r for _, r, _ in ins], [p for _, _, p in ins]),
                 _thr_arg(thrs))
    batch.run(grid, coarse)
    outs = batch.results(grid, coarse)
    return batch, outs, batch.fine_tiles()


def _record(o):
    return (o.found, o.ix, o.iy, o.it, o.score, o.win_x, o.win_y, o.win_t)


def _same_records(outs, models):
    for m, (o, md) in enumerate(zip(outs, models)):
        ref = md.ref
        assert _record(o) == (ref.found, ref.ix, ref.iy, ref.it, ref.score, ref.winX, ref.winY, ref.winT), f"match {m}"


def _bits(a):
    return np.ascontiguousarray(a).view(np.int64)


def _three_ways(ctx, batch, grid, coarse, params, ins, thrs, models, outs):
    """The pruned run's records, the flattened exhaustive kernel's records, and the tables of debug() after
    each (the exhaustive row sweep after the pruned run, the flat kernel's own) against rtcsm_score_table."""
    pruned_tabs = [batch.debug(m)[:2] for m in range(len(ins))]
    flat0 = ctx.get_option("csm_flat")
    try:
        ctx.set_option("csm_flat", 1)            # read by upload: set before it
        flat, flat_outs, (scored, total) = _run(ctx, grid, coarse, params, ins, thrs)
        flat_tabs = [flat.debug(m)[:2] for m in range(len(ins))]
    finally:
        ctx.set_option("csm_flat", flat0)
    assert scored == total                       # the flattened kernel scores everything
    assert [_record(o) for o in flat_outs] == [_record(o) for o in outs]
    L = params["low_res"]
    for m, ((pf, pc), (ff, fc), md) in enumerate(zip(pruned_tabs, flat_tabs, models)):
        ref_c = md.coarse[:, ::L, ::L].transpose(0, 2, 1)
        assert np.array_equal(_bits(pf), _bits(md.fine)) and np.array_equal(_bits(ff), _bits(md.fine)), f"fine {m}"
        assert np.array_equal(_bits(pc), _bits(ref_c)) and np.array_equal(_bits(fc), _bits(ref_c)), f"coarse {m}"


def _shape(o, L):
    nbx, nby = (2 * o.win_x) // L + 1, (2 * o.win_y) // L + 1
    nxw, nyw = nbx * L, nby * L
    rows = 0 if nxw * nyw < 512 else (5 if nyw % 5 == 0 else 4)
    return nbx, nby, nxw, nyw, rows, (nxw + 31) // 32


def _flat_tiles(o, L):
    """Warps of the flattened kernel per theta slice: one thread per 4 hypotheses from 512 on, else per one."""
    nxw, nyw = _shape(o, L)[2:4]
    hpt = 4 if nxw * nyw >= 512 else 1
    return (2 * o.win_t + 1) * (((nxw * nyw + hpt - 1) // hpt + 31) // 32)


# ---- 1 + 2: work per match, window shapes ----------------------------------------------------------------

@pytest.mark.parametrize("case", list(CASES))
def test_pruned_work_per_match_equals_the_model(ctx, case):
    from oracle import backend
    R = backend()
    shape_params, want = CASES[case]
    params = dict(DEFAULTS, **shape_params)
    L = params["low_res"]
    thin = case == "low_res32_map_thinner_than_a_block"
    dense, mx, my, refmap = _scene_map(R, thin)
    if thin:
        assert dense.shape[0] < L
    pre = refmap.precompute(L)
    grid, coarse = _device_maps(ctx, dense, mx, my, L, pre)
    ins = _case_scans(thin)
    thrs = [None] * len(ins)
    eps = ctx.get_option("edge_eps")
    models = _models(R, refmap, pre, params, ins, thrs, eps)

    # every match alone: its record and its tiles
    for m, (x, md) in enumerate(zip(ins, models)):
        _, (o,), (scored, total) = _run(ctx, grid, coarse, params, [x], [None])
        _same_records([o], [md])
        assert _shape(o, L) == want, (case, _shape(o, L))
        if want[4]:
            assert (scored, total) == (md.n, md.total), (case, m, md.flag, md.basic_flag)
        else:
            assert scored == total == _flat_tiles(o, L)
    # all of them in one batch: batching changes no match's work
    batch, outs, (scored, total) = _run(ctx, grid, coarse, params, ins, thrs)
    _same_records(outs, models)
    if want[4]:
        assert (scored, total) == (sum(md.n for md in models), sum(md.total for md in models))
        # the upper-right scans hang over the upper or right edge, unflagged, and ran pruned
        ran_pruned = [md for md in models if md.overhang and not md.flag]
        assert ran_pruned, case
        if want[0] * want[1] > 1:                       # one block per slice: a slice is all or nothing
            assert any(md.n < md.total for md in ran_pruned), case
    else:
        assert scored == total == sum(_flat_tiles(o, L) for o in outs)
    if case == "low_res1":                               # a best block in the window's last column, x = 30
        assert any(md.ref.found and md.ref.ix == md.ref.winX == 15 and not md.flag for md in models)
    if case == "low_res32_fewer_blocks_than_seeds":
        assert all(md.nB < 4 for md in models)          # the seed list has -1 entries
    nts = [2 * o.win_t + 1 for o in outs]
    print(f"\n{case}: nbx nby nxw nyw rows xchunks = {want}, nT {min(nts)}-{max(nts)}, "
          f"flagged {[int(md.flag) for md in models]}, tiles device {scored} / model "
          f"{[(md.n, md.total) for md in models] if want[4] else '-'} of {total}")
    _three_ways(ctx, batch, grid, coarse, params, ins, thrs, models, outs)


# ---- 1: the near-edge +-1 test decides the flag ----------------------------------------------------------

def test_near_edge_flag_follows_the_extended_model(ctx):
    """edge_eps = 0.3: most projected points are near an edge and go through the host fix-up.  The scans'
    lowest cells sit one cell above the band (-lowRes, 0), so only the +-1 test of near-edge points can flag
    a match; the extended model must predict each match's tiles exactly."""
    from oracle import backend
    R = backend()
    dense, mx, my, ins, params = band_edge_scene(np.random.default_rng(21))
    refmap = R.RefMap.from_dense(dense, mx, my)
    pre = refmap.precompute(params["low_res"])
    grid, coarse = _device_maps(ctx, dense, mx, my, params["low_res"], pre)
    eps0 = ctx.get_option("edge_eps")
    thrs = [None] * len(ins)
    models = _models(R, refmap, pre, params, ins, thrs, 0.3)
    assert not any(md.basic_flag for md in models)
    assert any(md.flag for md in models) and any(not md.flag and md.n < md.total for md in models)
    try:
        ctx.set_edge_eps(0.3)
        fixups = 0
        for m, (x, md) in enumerate(zip(ins, models)):
            _, (o,), (scored, total) = _run(ctx, grid, coarse, params, [x], [None])
            _same_records([o], [md])
            fixups += o.n_fixups
            assert (scored, total) == (md.n, md.total), (m, md.flag)
        batch, outs, (scored, total) = _run(ctx, grid, coarse, params, ins, thrs)
    finally:
        ctx.set_edge_eps(eps0)
    assert fixups > 100
    _same_records(outs, models)
    assert scored == sum(md.n for md in models)
    print(f"\nnear-edge: flagged {[int(md.flag) for md in models]}, fix-ups {fixups}, "
          f"tiles {[(md.n, md.total) for md in models]}")


# ---- 3: a mixed batch --------------------------------------------------------------------------------------

def _exact_threshold(score, nb):
    """The smallest normalised threshold thr with thr * nb == score, within 64 ulps of score / nb (None when
    no such thr exists: the product can step over score)."""
    hits = [t for t in _ulps(score / nb, 64) if t * float(nb) == score]
    if not hits:
        return None
    thr = min(hits)
    while np.nextafter(thr, -np.inf) * float(nb) == score:
        thr = np.nextafter(thr, -np.inf)
    return float(thr)


def _ulps(x, k):
    out, lo, hi = [x], x, x
    for _ in range(k):
        lo, hi = np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)
        out += [lo, hi]
    return out


def test_mixed_batch_thresholds_and_ragged_scans(ctx):
    from oracle import backend
    R = backend()
    params = dict(DEFAULTS, low_res=5, range_x=1.0, range_y=1.0)
    dense, mx, my, refmap = _scene_map(R, False)
    pre = refmap.precompute(5)
    grid, coarse = _device_maps(ctx, dense, mx, my, 5, pre)
    world = _rooms()[0]
    rng = np.random.default_rng(31)
    ur = [_scan(world, rng, 2.0, 4.5, n, fov) for n, fov in ((361, 270.0), (181, 180.0), (241, 240.0), (361, 270.0))]
    ll = [_scan(world, rng, -4.6, -3.6, n) for n in (241, 361)]
    a, r, p = ur[3]
    short = (a, np.minimum(r, 2.0), p)           # a smaller maximum range: a coarser theta step, fewer slices
    none_kept = (a, np.full(a.shape, params["scan_range_max"]), p)     # every beam dropped
    # the threshold at a match's best score, and one ulp below it
    for at in ur:
        best = R.rtcsm_match(refmap, *at, pre=pre, **params)
        thr_at = _exact_threshold(best.score, len(at[1])) if best.found else None
        if thr_at is not None:
            break
    assert thr_at is not None
    thr_below = float(np.nextafter(thr_at, -np.inf))
    ins = [at, at, ur[1], ll[0], short, none_kept, ur[2], ll[1], ur[3]]
    thrs = [thr_at, thr_below, None, 0.3, 0.3, None, 0.99, TINY, 0.3]
    eps = ctx.get_option("edge_eps")
    models = _models(R, refmap, pre, params, ins, thrs, eps)
    assert models[0].thr_abs == best.score and not models[0].ref.found
    assert models[1].ref.found and models[1].ref.score == best.score
    assert any(md.flag for md in models) and any(not md.flag and md.n < md.total for md in models)
    assert len({md.ref.winT for md in models}) > 1 and len({len(r) for _, r, _ in ins}) > 1

    batch, outs, (scored, total) = _run(ctx, grid, coarse, params, ins, thrs)
    _same_records(outs, models)
    assert (scored, total) == (sum(md.n for md in models), sum(md.total for md in models))
    o = outs[5]                                  # no kept beam: nothing scored, not found, initial indices
    assert models[5].n == 0 and not o.found and (o.ix, o.iy, o.it) == (-o.win_x, -o.win_y, -o.win_t)
    for m in (0, 1):                             # at and one ulp below the best score, alone
        _, (o,), (n, _) = _run(ctx, grid, coarse, params, [ins[m]], [thrs[m]])
        _same_records([o], [models[m]])
        assert n == models[m].n
    print(f"\nmixed: flagged {[int(md.flag) for md in models]}, nT {[2 * o.win_t + 1 for o in outs]}, "
          f"tiles {[(md.n, md.total) for md in models]}")
    _three_ways(ctx, batch, grid, coarse, params, ins, thrs, models, outs)


# ---- 5: one batch across grids, results() calls and uploads ------------------------------------------------

def test_batch_state_follows_new_inputs(ctx):
    from oracle import backend
    R = backend()
    params = dict(DEFAULTS, low_res=5, range_x=1.0, range_y=1.0)
    dense, mx, my, refmap = _scene_map(R, False)
    pre = refmap.precompute(5)
    grid, coarse = _device_maps(ctx, dense, mx, my, 5, pre)
    world = _rooms()[0]
    rng = np.random.default_rng(41)
    ins = [_scan(world, rng, 2.0, 4.5, n) for n in (181, 361, 241)] + [_scan(world, rng, -4.6, -3.6, 241)]
    thrs = [None, 0.3, None, None]
    eps = ctx.get_option("edge_eps")
    batch = capi.RtcsmBatch(ctx, **params)

    def check(outs, n, refmap_, pre_, ins_, thrs_):
        models = _models(R, refmap_, pre_, params, ins_, thrs_, eps)
        _same_records(outs, models)
        assert n == sum(md.n for md in models)
        return models

    # 1. upload, run, results
    _, outs, (n, _) = _run(ctx, grid, coarse, params, ins, thrs, batch)
    check(outs, n, refmap, pre, ins, thrs)
    # 2. the same upload run on another grid of the same geometry: more scans integrated, coarse map again
    grid2 = capi.Grid.from_dense(ctx, dense, mx, my, RES, apron=APRON)
    extra = [np.array([x, y, th]) for x, y, th in ((3.0, 3.5, 0.4), (-3.0, 3.0, 1.0), (3.5, -3.0, 2.0))]
    hits = [capi.scan_hit_points(p, ins[1][0], synth.make_scan(world, p, ins[1][0], rng), 0.02, 20.0)[0]
            for p in extra]
    capi.integrate_scans(ctx, grid2, [p[:2] for p in extra], hits)
    dense2 = grid2.download()
    assert not np.array_equal(dense2, dense)
    refmap2 = R.RefMap.from_dense(dense2, mx, my, RES, 16)
    pre2 = refmap2.precompute(5)
    coarse2 = grid2.precompute(5)
    assert np.array_equal(_bits(coarse2.download()), _bits(pre2.dense()))
    batch.run(grid2, coarse2)
    outs2 = batch.results(grid2, coarse2)
    n2 = batch.fine_tiles()[0]
    check(outs2, n2, refmap2, pre2, ins, thrs)
    # 3. results twice: nothing changes
    for _ in range(2):
        again = batch.results(grid2, coarse2)
        assert [_record(o) for o in again] == [_record(o) for o in outs2]
        assert batch.fine_tiles()[0] == n2
    # 4. a smaller batch and another window (res 0.04: 30 x 30 cells, five-row groups) on the same batch object
    refmap3 = R.RefMap.from_dense(dense2, mx, my, 0.04, 16)
    pre3 = refmap3.precompute(5)
    grid3 = capi.Grid.from_dense(ctx, dense2, mx, my, 0.04, apron=APRON)
    coarse3 = grid3.precompute(5)
    ins3, thrs3 = [ins[3], ins[0]], [None, 0.3]
    batch.upload(grid3, capi.Scans([a for a, _, _ in ins3], [r for _, r, _ in ins3], [p for _, _, p in ins3]),
                 _thr_arg(thrs3))
    batch.run(grid3, coarse3)
    outs3 = batch.results(grid3, coarse3)
    models3 = check(outs3, batch.fine_tiles()[0], refmap3, pre3, ins3, thrs3)
    assert _shape(outs3[0], 5) == (6, 6, 30, 30, 5, 1)
    assert batch.fine_tiles()[1] == sum(md.total for md in models3)
    # and back to the first inputs
    _, outs, (n, _) = _run(ctx, grid, coarse, params, ins, thrs, batch)
    check(outs, n, refmap, pre, ins, thrs)
