"""CPU model of the interval argument of lgs_grid_construct_many (DESIGN.md section 3.4).

The device projects every beam with its own sincos, which may differ from glibc's in the last ulps.  It evaluates the
CPU's hit expression sx + r * cos(st + a), in the CPU's operation order, at the two ends of cos +- U ulps (U = 8) and
keeps [lo, hi] = the smaller and larger result.  Every operation is monotone, so glibc's hit lies in [lo, hi]:
  * equal floors of (lo - min) / res and (hi - min) / res are glibc's cell;
  * with D = max over beams of lo (and the sensor positions and the DBL_MIN seed), the beams with hi >= D hold
    glibc's maximum; likewise for the three other sides.
Here math.cos / math.sin are glibc, a device value is glibc's moved by up to 2 ulps, and Python floats are IEEE
doubles rounded to nearest without contraction, as the device code is compiled (-fmad=false)."""
import math

import numpy as np

U = 8
EPS = 2.220446049250313e-16
TRUE_MIN = 5e-324
TINY = float(np.finfo(np.float64).tiny)


def _device(v, rng):
    """glibc's value moved by -2 .. 2 ulps: a stand-in for CUDA's sincos."""
    for _ in range(abs(k := int(rng.integers(-2, 3)))):
        v = math.nextafter(v, math.inf if k > 0 else -math.inf)
    return v


def _interval(p, r, trig):
    w = abs(trig) * (U * EPS) + TRUE_MIN
    e0, e1 = p + r * (trig - w), p + r * (trig + w)
    return min(e0, e1), max(e0, e1)


def _scan(rng, n):
    pose = (rng.uniform(-50, 50), rng.uniform(-50, 50), rng.uniform(-math.pi, math.pi))
    angles = np.linspace(-2.36, 2.36, n)
    ranges = rng.uniform(-1.0, 25.0, n)
    # some exact cell-edge hits: axis-aligned beams of whole-cell ranges from a sensor on a cell corner
    if rng.random() < 0.3:
        pose = (float(rng.integers(-20, 20)), float(rng.integers(-20, 20)), 0.0)
        angles = np.resize([0.0, math.pi / 2, math.pi, -math.pi / 2], n)
        ranges = 0.25 * rng.integers(1, 60, n)
    return pose, angles, ranges


def test_candidates_hold_the_glibc_extreme_and_equal_floors_give_the_glibc_cell():
    rng = np.random.default_rng(2024)
    res_choices = (0.25, 0.05, 0.1)
    edges = decided = 0
    for trial in range(40):
        res = res_choices[trial % 3]
        rmin, rmax = (-0.5 if trial % 5 == 0 else 0.02), 20.0
        scans = [_scan(rng, 181) for _ in range(int(rng.integers(1, 6)))]
        hits = []          # (glibc x, glibc y, (lo x, hi x), (lo y, hi y))
        sensors = []
        for (sx, sy, st), angles, ranges in scans:
            sensors.append((sx, sy))
            for a, r in zip(angles, ranges):
                r = float(r)
                if r >= rmax or r <= rmin:
                    continue
                t = st + float(a)
                c, s = math.cos(t), math.sin(t)
                hits.append((sx + r * c, sy + r * s, _interval(sx, r, _device(c, rng)), _interval(sy, r, _device(s, rng))))
        # bbox sides: the candidates' glibc values, the sensors and the seed give the exact extreme
        for axis in (0, 1):
            want_max = max([TINY] + [p[axis] for p in sensors] + [h[axis] for h in hits])
            want_min = min([1.7976931348623157e308] + [p[axis] for p in sensors] + [h[axis] for h in hits])
            d_max = max([TINY] + [p[axis] for p in sensors] + [h[2 + axis][0] for h in hits])
            d_min = min([1.7976931348623157e308] + [p[axis] for p in sensors] + [h[2 + axis][1] for h in hits])
            cand_max = [h[axis] for h in hits if h[2 + axis][1] >= d_max]
            cand_min = [h[axis] for h in hits if h[2 + axis][0] <= d_min]
            assert max([TINY] + [p[axis] for p in sensors] + cand_max) == want_max
            assert min([1.7976931348623157e308] + [p[axis] for p in sensors] + cand_min) == want_min
        # cells against a patch-aligned origin
        mn = (math.floor(min(h[0] for h in hits) / (64 * res)) * 64 * res if hits else 0.0,
              math.floor(min(h[1] for h in hits) / (64 * res)) * 64 * res if hits else 0.0)
        for h in hits:
            for axis in (0, 1):
                lo, hi = h[2 + axis]
                c_lo, c_hi = math.floor((lo - mn[axis]) / res), math.floor((hi - mn[axis]) / res)
                if c_lo == c_hi:
                    decided += 1
                    assert c_lo == math.floor((h[axis] - mn[axis]) / res)
                else:
                    edges += 1
    assert decided > 10000 and edges > 0          # the axis-aligned scans put hits exactly on cell edges
