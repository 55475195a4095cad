"""CPU model of the pruned correlative sweep (csm_project_kernel's flag, csm_prune_kernel, csm_select_kernel,
csrc/lgs_csm.cu) on the reference's own score tables.

  * flag: a match whose clamped projected cell plus some block origin lies in (-lowRes, 0) on either axis
    (SURVEY.md H12) is scored exhaustively and selected as before (test_rtcsm_device_model._select);
  * seed: the fine maxima of the K best coarse blocks in (C desc, visit asc) order give L <= F*;
  * keep: C[b] >= L and C[b] > thrAbs; only kept blocks are candidates of the selection;
  * tiles: the (theta pair, warp of the row sweep) tiles holding a kept block of either slice are scored.

The model must return the reference's answer, every match where a coarse score fails to bound its block
must be flagged, and on the bench's C2 workload the scored tiles are a small part of the exhaustive sweep."""
import math

import numpy as np

from my_lidar_graph_slam_b200 import synth
from test_rtcsm_device_model import _select

K = 4       # csm_prune_kernel's kSeedBlocks
TG = 2      # theta slices per tile (kThetaGroup)


def _blocks(fine, coarse, L):
    """-> F, C [t][bx][by] in visit order, first-visit argmax A (window x, y)."""
    nt, nyw, nxw = fine.shape
    nbx, nby = nxw // L, nyw // L
    blk = fine.reshape(nt, nby, L, nbx, L).transpose(0, 3, 1, 4, 2).reshape(nt, nbx, nby, L * L)   # fx, fy
    k = blk.argmax(axis=3)
    F = np.take_along_axis(blk, k[..., None], 3)[..., 0]
    A = np.stack([np.arange(nbx)[None, :, None] * L + k // L, np.arange(nby)[None, None, :] * L + k % L], -1)
    C = coarse[:, ::L, ::L].transpose(0, 2, 1)
    return F, C, A


def near_edge(pose, angles, ranges, step_t, win_t, min_x, min_y, res, eps):
    """csm_project_kernel's near-edge test [t][beam] for kept beams: the projected point's fractional cell
    lies within eps of a cell edge on either axis.  The projection's operation order, with the host's libm
    (the device's sincos can differ by an ulp, which matters only within an ulp of the band's limits)."""
    out = np.zeros((2 * win_t + 1, len(ranges)), bool)
    for t in range(2 * win_t + 1):
        theta = pose[2] + step_t * (t - win_t)
        for i, (a, r) in enumerate(zip(angles, ranges)):
            qx = (pose[0] + r * math.cos(theta + a) - min_x) / res
            qy = (pose[1] + r * math.sin(theta + a) - min_y) / res
            fx, fy = qx - math.floor(qx), qy - math.floor(qy)
            out[t, i] = not (eps <= fx <= 1.0 - eps and eps <= fy <= 1.0 - eps)
    return out


def flagged(cells, win_x, win_y, nxw, nyw, L, nx, ny, edge=None):
    """csm_project_kernel's 'coarse may not bound' flag from projected cells [t][beam][2] (kept beams).
    Near-edge points (edge [t][beam], from near_edge) are tested at their clamped cell and one cell either
    side, since results() may re-derive them one cell away."""
    cx = np.clip(cells[..., 0].astype(np.int64), win_x - nxw, nx + win_x)
    cy = np.clip(cells[..., 1].astype(np.int64), win_y - nyw, ny + win_y)
    band = False
    for s in ((0,) if edge is None else (-1, 0, 1)):
        use = np.ones(cx.shape, bool) if s == 0 else edge
        rx = cx[..., None] + s - win_x + L * np.arange(nxw // L)
        ry = cy[..., None] + s - win_y + L * np.arange(nyw // L)
        band |= bool((((rx > -L) & (rx < 0)).any(-1) & use).any() or (((ry > -L) & (ry < 0)).any(-1) & use).any())
    return band


def prune(F, C, thr, k=K):
    """-> (L, keep mask) of csm_prune_kernel."""
    order = np.lexsort((np.arange(C.size), -C.ravel()))          # C desc, visit asc
    bound = F.ravel()[order[:k]].max()
    return bound, (C >= bound) & (C > thr)


def tiles(keep, nxw, nyw, L):
    """Warp tiles (theta pair, row group, x chunk) of the row sweep holding a kept block."""
    nt, nbx, nby = keep.shape
    rows = 5 if nyw % 5 == 0 else 4
    groups, rgs, xcs = (nt + TG - 1) // TG, (nyw + rows - 1) // rows, (nxw + 31) // 32
    need = np.zeros((groups, rgs, xcs), bool)
    for t, bx, by in zip(*np.nonzero(keep)):
        for rg in range(by * L // rows, (by * L + L - 1) // rows + 1):
            for xc in range(bx * L // 32, (bx * L + L - 1) // 32 + 1):
                need[t // TG, rg, xc] = True
    return int(need.sum()), need.size


def model_select(fine, coarse, L, thr, is_flagged):
    """-> (found, ix, iy, it, score, tiles scored, tiles in all) with window-relative indices."""
    nt, nyw, nxw = fine.shape
    if is_flagged:
        found, ix, iy, it, score, _, _ = _select(fine, coarse, L, thr)
        n = tiles(np.ones((nt, nxw // L, nyw // L), bool), nxw, nyw, L)
        return (found, ix, iy, it, score) + n
    F, C, A = _blocks(fine, coarse, L)
    _, keep = prune(F, C, thr)
    n = tiles(keep, nxw, nyw, L)
    cand = np.where(keep, F, -1.0)
    if not keep.any() or not cand.max() > thr:
        return (0, None, None, None, thr) + n
    t, bx, by = np.unravel_index(int(np.argmax(cand == cand.max())), cand.shape)   # first visit
    return (1, int(A[t, bx, by, 0]), int(A[t, bx, by, 1]), int(t), float(cand.max())) + n


def _check(R, refmap, pre, angles, ranges, init, params, thr=None):
    ref = R.rtcsm_match(refmap, angles, ranges, init, pre=pre, thr=thr, **params)
    L = params["low_res"]
    nxw, nyw = ((2 * ref.winX) // L + 1) * L, ((2 * ref.winY) // L + 1) * L
    args = (L, params["scan_range_max"], init, angles, ranges, ref.stepT, ref.winT, -ref.winX, nxw, -ref.winY, nyw)
    fine, idx, cnt = R.rtcsm_score_table(refmap, pre, False, *args)
    coarse, _, _ = R.rtcsm_score_table(refmap, pre, True, *args)
    nx, ny = refmap.geometry()[:2]
    flag = flagged(idx[:, :cnt[0]], ref.winX, ref.winY, nxw, nyw, L, nx, ny)
    thr_abs = (float(np.finfo(np.float64).tiny) if thr is None else thr) * len(ranges)
    found, ix, iy, it, score, n, total = model_select(fine, coarse, L, thr_abs, flag)
    assert found == ref.found
    if found:
        assert (ix - ref.winX, iy - ref.winY, it - ref.winT) == (ref.ix, ref.iy, ref.it)
        assert score == ref.score
    F, C, _ = _blocks(fine, coarse, L)
    bounded = bool((C >= F).all())
    assert flag or bounded, "a coarse score below its block in an unflagged match"
    return flag, bounded, n, total


def test_model_selects_the_reference_answer_on_the_room_scene():
    from oracle import backend
    from scenes import room_scene
    R = backend()
    world, angles, traj, builder = room_scene(seed=1, n_beams=361)
    refmap = builder.latest_map()
    pre = refmap.precompute(5)
    params = dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=0.6, scan_range_max=5.7296)
    rng = np.random.default_rng(3)
    scored = total = unflagged = 0   # the room's outer walls are the map's edges: most matches are flagged
    for k in range(6):
        true = traj[10 + k % 4]
        scan = synth.make_scan(world, true, angles, np.random.default_rng(100 + k))
        init = true + np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3), rng.uniform(-0.2, 0.2)])
        for thr in (None, 0.99):                            # 0.99: nothing beats it
            # beams that reach the outermost walls, the map's bounding box, flag their match
            flag, _, n, t = _check(R, refmap, pre, angles, scan, init, params, thr)
            if flag:
                continue
            if thr is None:
                scored, total, unflagged = scored + n, total + t, unflagged + 1
            else:
                assert n == 0
    if unflagged:
        assert scored < total


def test_model_flags_the_lower_edge_and_replays_it():
    """H12 scene (test_rtcsm_device_model): every match whose coarse scores fail to bound is flagged and
    replayed; the flagged ones give the reference's answer from full tables."""
    from oracle import backend
    R = backend()
    rng = np.random.default_rng(7)
    ny, nx = 128, 128
    dense = np.where(rng.random((ny, nx)) < 0.25, rng.uniform(0.05, 0.95, (ny, nx)), 0.0)
    dense[:12, :] = rng.uniform(0.5, 0.99, (12, nx))
    dense[:, :12] = rng.uniform(0.5, 0.99, (ny, 12))
    refmap = R.RefMap.from_dense(dense, -1.0, -2.0)
    pre = refmap.precompute(5)
    params = dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=0.2, scan_range_max=20.0)
    angles = synth.beam_angles(181, 180.0)
    flags = unbounded = 0
    for k in range(10):
        ranges = rng.uniform(0.1, 0.5, angles.shape)
        init = np.array([-1.0 + rng.uniform(0.0, 0.3), -2.0 + rng.uniform(0.5, 3.0), np.pi + rng.uniform(-0.3, 0.3)])
        flag, bounded, _, _ = _check(R, refmap, pre, angles, ranges, init, params)
        flags += flag
        unbounded += not bounded
    assert unbounded > 0 and flags >= unbounded


def band_edge_scene(rng, n_matches=6):
    """Scans whose lowest projected cells sit one cell above the band (-lowRes, 0) of coarse indices at the
    lower map edge: row 5 with lowRes 5 and winY 10 (5 - 10 + 5 = 0); every other cell has row and column
    >= 10 in every theta slice.  The row-5 points lie mid-cell in even matches and within 0.3 of their cell's
    lower edge in odd ones, where the +-1 test of near-edge points (edge_eps 0.3) reaches row 4, in the band
(their x fractions stay mid-cell: the +-1 test shifts both axes of a point near an edge on either).
    -> (dense, min_x, min_y, [(angles, ranges, init)], params)."""
    n, mx, my, res = 128, -1.0, -2.0, 0.05
    # the map: strong cells along the lower edge and at the other points of every scan, zero elsewhere, so the
    # scans fit one pose and the pruned sweep of an unflagged match skips most tiles
    ux, uy = rng.uniform(15.0, 100.0, 157), rng.uniform(15.0, 100.0, 157)
    dense = np.zeros((n, n))
    dense[:12, :] = rng.uniform(0.5, 0.99, (12, n))
    dense[uy.astype(int), ux.astype(int)] = 0.9
    params = dict(low_res=5, range_x=1.0, range_y=1.0, range_theta=0.02, scan_range_max=20.0)
    ins = []
    for k in range(n_matches):
        cx, th = 40 + int(rng.integers(-2, 3)), rng.uniform(-0.05, 0.05)
        sx, sy = mx + (cx + 0.5) * res, my + 12.5 * res
        f = 0.5 if k % 2 == 0 else 0.15          # the rotation of the slices moves row-5 points < 0.15 cell
        line = np.stack([mx + (cx + rng.integers(-3, 4, 24) + 0.5) * res, np.full(24, my + (5 + f) * res)], 1)
        upper = np.stack([mx + ux * res, my + uy * res], 1)
        d = np.concatenate([line, upper]) - (sx, sy)
        ins.append((np.arctan2(d[:, 1], d[:, 0]) - th, np.hypot(d[:, 0], d[:, 1]), np.array([sx, sy, th])))
    return dense, mx, my, ins, params


def test_near_edge_points_are_tested_one_cell_either_side():
    """band_edge_scene on the reference's tables: the plain flag never fires; with edge_eps 0.3 the +-1 test
    of near-edge points flags exactly the scans whose row-5 points lie near their cells' lower edge, and with
    a zero band it adds nothing.  Every match the extended flag leaves unflagged has bounded coarse scores."""
    from oracle import backend
    R = backend()
    dense, mx, my, ins, params = band_edge_scene(np.random.default_rng(21))
    refmap = R.RefMap.from_dense(dense, mx, my)
    pre = refmap.precompute(5)
    nx, ny = refmap.geometry()[:2]
    for k, (angles, ranges, init) in enumerate(ins):
        flag, bounded, _, _ = _check(R, refmap, pre, angles, ranges, init, params)
        assert not flag and bounded
        ref = R.rtcsm_match(refmap, angles, ranges, init, pre=pre, **params)
        _, idx, cnt = R.rtcsm_score_table(refmap, pre, False, 5, params["scan_range_max"], init, angles, ranges,
                                          ref.stepT, ref.winT, -ref.winX, 25, -ref.winY, 25, want_table=False)
        cells = idx[:, :cnt[0]]
        assert (cells[..., 1] == 5).any(-1).all()                       # row-5 points in every slice
        assert ((cells[..., 1] == 5) | (cells[..., 1] >= 10)).all() and (cells[..., 0] >= 10).all()
        geo = (ref.winX, ref.winY, 25, 25, 5, nx, ny)
        for eps, want in ((0.3, k % 2 == 1), (0.0, False)):
            edge = near_edge(init, angles, ranges, ref.stepT, ref.winT, mx, my, 0.05, eps)
            assert flagged(cells, *geo, edge) == want, (k, eps)


def test_model_ties_keep_the_first_visit():
    """Equal fine maxima in different blocks and slices, coarse scores equal to them: the keep rule's '>='
    keeps every tied block and the selection returns the first visit, as the CPU's pruned loop does."""
    L = 5
    rng = np.random.default_rng(1)
    fine = rng.uniform(0.0, 1.0, (5, 15, 15)).round(2)
    for t, y, x in ((1, 12, 3), (1, 2, 11), (3, 0, 0), (4, 7, 7)):
        fine[t, y, x] = 2.0
    coarse = np.zeros_like(fine)
    F, C, _ = _blocks(fine, np.zeros_like(fine), L)
    coarse[:, ::L, ::L] = F.transpose(0, 2, 1)               # C = F: every coarse score is tight
    F, C, _ = _blocks(fine, coarse, L)
    thr = 0.5
    found, ix, iy, it, score, n, _ = model_select(fine, coarse, L, thr, False)
    ref = _select(fine, coarse, L, thr)
    assert (found, ix, iy, it, score) == ref[:5] == (1, 3, 12, 1, 2.0)
    # the CPU loop itself: `if (C > best && F > best)` in visit order
    best, win = thr, None
    for t in range(5):
        for bx in range(3):
            for by in range(3):
                if C[t, bx, by] > best and F[t, bx, by] > best:
                    best, win = F[t, bx, by], (t, bx, by)
    assert win == (1, 0, 2) and best == 2.0
    bound, keep = prune(F, C, thr)
    assert bound == 2.0 and keep.sum() == 4 and n == 4    # tiles: slices 0-1 row groups 0 and 2, 2-3, 4


def test_c2_prune_fraction():
    """The bench's C2 workload: fraction of fine blocks, block rows and warp tiles the pruned sweep scores."""
    import bench
    from oracle import backend
    R = backend()
    C2 = bench.C2
    traj, map_scans, angles, ranges, inits = bench.c2_workload(12, seed=1)
    builder = R.RefBuilder()
    for p, r in zip(traj, map_scans):
        builder.append_scan(p, angles, r)
    refmap = builder.latest_map()
    pre = refmap.precompute(5)
    blocks = kept = rows = rows_all = n_tiles = n_all = 0
    for r, init in zip(ranges, inits):
        flag, bounded, n, t = _check(R, refmap, pre, angles, r, init, C2)
        assert not flag and bounded
        n_tiles, n_all = n_tiles + n, n_all + t
        ref = R.rtcsm_match(refmap, angles, r, init, pre=pre, **C2)
        args = (5, C2["scan_range_max"], init, angles, r, ref.stepT, ref.winT, -ref.winX, 25, -ref.winY, 25)
        F, C, _ = _blocks(R.rtcsm_score_table(refmap, pre, False, *args)[0],
                          R.rtcsm_score_table(refmap, pre, True, *args)[0], 5)
        _, keep = prune(F, C, float(np.finfo(np.float64).tiny) * len(r))
        blocks, kept = blocks + keep.size, kept + keep.sum()
        rows, rows_all = rows + keep.any(axis=1).sum(), rows_all + keep.shape[0] * keep.shape[2]
    print(f"C2: fine blocks kept {kept / blocks:.4f}, block rows {rows / rows_all:.4f}, "
          f"warp tiles {n_tiles / n_all:.4f} of the exhaustive sweep")
    assert n_tiles < 0.1 * n_all
