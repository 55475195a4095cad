"""CPU model of the theta-grouped row sweep's load plan (csm_sweep_rows_kernel, csrc/lgs_csm.cu).

A thread owns ROWS window rows of TG consecutive theta slices.  Per kept beam it holds the TG offsets o[t] of
the group (a slice past the match's nT repeats the last valid slice).  Slice 0 loads its ROWS rows; slice t
then decides from o[t] - o[t - 1] alone:

  * 0: the same cell, every row is already held;
  * +pitch / -pitch: the cell above / below, the held rows shift by one and one row is loaded;
  * anything else: all ROWS rows are loaded.

The model replays that plan with registers (values held per lane), accumulates in beam order and compares
with direct gathers bit for bit; on the C2 workload it reports the fraction of the ungrouped sweep's loads
the plan issues."""
import os
import re

import numpy as np

from my_lidar_graph_slam_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROWS = 5


def _kernel_group_size():
    src = open(os.path.join(ROOT, "my_lidar_graph_slam_b200", "csrc", "lgs_csm.cu")).read()
    return int(re.search(r"constexpr int kThetaGroup = (\d+);", src).group(1))


TG = _kernel_group_size()


def group_offsets(offs, t0, tg):
    """offs[nT][nB] -> the [tg][nB] offsets a block stages for slices t0 .. t0 + tg (tail repeats)."""
    return offs[np.minimum(np.arange(t0, t0 + tg), offs.shape[0] - 1)]


def load_plan(o, pitch, rows=ROWS, shifts=True):
    """One beam's offsets of one group -> (addresses loaded, per slice the register index of each row)."""
    o = [int(x) for x in o]
    loads = [o[0] + k * pitch for k in range(rows)]
    held = list(range(rows))                      # register index of row k of the current slice
    picks = [held]
    for t in range(1, len(o)):
        d = o[t] - o[t - 1]
        if d == 0:
            pass
        elif shifts and d == pitch:
            held = held[1:] + [len(loads)]
            loads.append(o[t] + (rows - 1) * pitch)
        elif shifts and d == -pitch:
            held = [len(loads)] + held[:-1]
            loads.append(o[t])
        else:
            held = list(range(len(loads), len(loads) + rows))
            loads += [o[t] + k * pitch for k in range(rows)]
        picks.append(held)
    return loads, picks


def planned_loads(offs, pitch, tg=TG, rows=ROWS, shifts=True):
    """Rows gathered by the plan over a whole match (vectorised; equals summing load_plan)."""
    nT = offs.shape[0]
    g = np.stack([group_offsets(offs, t0, tg) for t0 in range(0, nT, tg)])     # [groups][tg][nB]
    d = g[:, 1:] - g[:, :-1]
    per_step = np.where(d == 0, 0, np.where(shifts & (np.abs(d) == pitch), 1, rows))
    return int(rows * g.shape[0] * g.shape[2] + per_step.sum())


def _sweep(grid, bases, offs, pitch, tg, planned):
    """Scores [nT][ROWS][lanes] of hypotheses at bases (one per lane), beams in order."""
    nT, nB = offs.shape
    acc = np.zeros((nT, ROWS, len(bases)))
    for t0 in range(0, nT, tg):
        g = group_offsets(offs, t0, tg)
        a = np.zeros((tg, ROWS, len(bases)))
        for i in range(nB):
            if planned:
                loads, picks = load_plan(g[:, i], pitch)
                regs = [grid[bases + x] for x in loads]
                for t in range(tg):
                    for k in range(ROWS):
                        a[t, k] = a[t, k] + regs[picks[t][k]]
            else:
                for t in range(tg):
                    for k in range(ROWS):
                        a[t, k] = a[t, k] + grid[bases + g[t, i] + k * pitch]
        n = min(tg, nT - t0)
        acc[t0:t0 + n] = a[:n]
    return acc


def _random_offsets(rng, nT, nB, pitch, sentinel):
    """Offsets with runs of equal values, +-pitch steps, column changes, jumps and clamped sentinels."""
    offs = np.empty((nT, nB), dtype=np.int64)
    for i in range(nB):
        if rng.random() < 0.1:
            offs[:, i] = sentinel                      # padding beam / clamped point
            continue
        x = int(rng.integers(15 * pitch, 18 * pitch))
        for t in range(nT):
            offs[t, i] = x
            u = rng.random()
            if u < 0.45:
                pass
            elif u < 0.65:
                x += pitch
            elif u < 0.8:
                x -= pitch
            elif u < 0.9:
                x += int(rng.choice([-1, 1]))
            elif u < 0.95:
                x = int(rng.integers(15 * pitch, 18 * pitch))
            else:
                x = sentinel
    return offs


def test_plan_accumulates_the_direct_gathers_bit_for_bit():
    rng = np.random.default_rng(11)
    pitch = 37
    grid = rng.standard_normal(40 * pitch) * 10.0 ** rng.integers(-8, 8, 40 * pitch)
    bases = np.arange(0, 2 * pitch, 5)[:8] + pitch          # lanes at different (row, x) hypotheses
    for nT, nB in ((9, 40), (7, 33), (TG, 50), (1, 12), (3 * TG + 1, 25)):
        offs = _random_offsets(rng, nT, nB, pitch, sentinel=0)
        ref = _sweep(grid, bases, offs, pitch, TG, planned=False)
        got = _sweep(grid, bases, offs, pitch, TG, planned=True)
        assert np.array_equal(ref.view(np.int64), got.view(np.int64))
        # the direct gather is the per-slice loop of the ungrouped kernel
        flat = _sweep(grid, bases, offs, pitch, 1, planned=False)
        assert np.array_equal(ref.view(np.int64), flat.view(np.int64))
        count = sum(len(load_plan(group_offsets(offs, t0, TG)[:, i], pitch)[0])
                    for t0 in range(0, nT, TG) for i in range(nB))
        assert count == planned_loads(offs, pitch)


def test_plan_cases():
    p = 100
    # same cell in every slice: one run of ROWS rows
    loads, picks = load_plan([500, 500, 500, 500][:TG], p)
    assert len(loads) == ROWS and all(pk == list(range(ROWS)) for pk in picks)
    # one row up, then back down: one extra row per step, the held rows shift
    o = [500, 600, 500, 400, 400, 500, 600, 600]
    loads, picks = load_plan(o, p)
    assert len(loads) == ROWS + 5
    for t in range(len(o)):
        assert [loads[j] for j in picks[t]] == [o[t] + k * p for k in range(ROWS)]
    # a column change reloads every row
    o = [500, 501, 501, 501]
    loads, picks = load_plan(o, p)
    assert len(loads) == 2 * ROWS
    for t in range(len(o)):
        assert [loads[j] for j in picks[t]] == [o[t] + k * p for k in range(ROWS)]


def _c2_offsets(n_matches):
    """Projected, clamped offsets of C2 matches on the bench's map geometry (host steps of its map build)."""
    import bench
    C2 = bench.C2
    traj, map_scans, angles, ranges, inits = bench.c2_workload(n_matches, seed=1)
    geo = capi.Geometry(0, 0, float(traj[0][0]), float(traj[0][1]), 0.05, 64)
    for p, r in zip(traj, map_scans):
        _, bbox = capi.scan_hit_points(p, angles, r, 0.02, 20.0)
        geo, _, _, _ = capi.geometry_expand(geo, bbox)
    nx, ny, min_x, min_y, res = geo.as_tuple()
    pitch = nx + 2 * 32                                     # apron of the bench's map
    win = int(np.ceil(0.5 * C2["range_x"] / res))
    nw = ((2 * win) // C2["low_res"] + 1) * C2["low_res"]
    lo, hi = -win, -win + nw - 1
    for r, init in zip(ranges, inits):
        keep = r < C2["scan_range_max"]
        max_range = min(r.max(), C2["scan_range_max"])
        step = np.arccos(1.0 - 0.5 * (res / max_range) ** 2)
        win_t = int(np.ceil(0.5 * C2["range_theta"] / step))
        th = init[2] + step * (np.arange(2 * win_t + 1) - win_t)
        a = th[:, None] + angles[keep][None, :]
        cx = np.floor((init[0] + r[keep] * np.cos(a) - min_x) / res).astype(np.int64)
        cy = np.floor((init[1] + r[keep] * np.sin(a) - min_y) / res).astype(np.int64)
        offs = np.clip(cy, -hi - 1, ny - lo) * pitch + np.clip(cx, -hi - 1, nx - lo)
        yield offs, pitch


def test_c2_load_fraction():
    fracs = {}
    for tg in (2, 4, 8):
        loads = base = same_only = 0
        for offs, pitch in _c2_offsets(60):
            nT, nB = offs.shape
            base += nT * nB * ROWS
            loads += planned_loads(offs, pitch, tg=tg)
            same_only += planned_loads(offs, pitch, tg=tg, shifts=False)    # reuse of equal offsets only
        fracs[tg] = (loads / base, same_only / base)
        print(f"C2: TG={tg} loads issued {loads / base:.3f} of the ungrouped sweep "
              f"(equal offsets only: {same_only / base:.3f})")
    assert all(f < s for f, s in fracs.values())
    assert fracs[2][0] > fracs[4][0] > fracs[8][0]
    assert 0.6 < fracs[2][0] < 0.75 and 0.45 < fracs[4][0] < 0.6
