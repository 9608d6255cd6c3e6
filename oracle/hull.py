"""Oracle (test infrastructure): per-ring convex hull, solidity and orientation, exact.

Cell 18 of hovernet_tile_inference.ipynb:2415-2456 asks regionprops_table for ``solidity`` and ``orientation``; this is
their polygon counterpart, the reference for pg_ring_hull_* (K14).

* Every coordinate is a binary float, so ``x = X / D`` with integers X and D a power of two (``float.as_integer_ratio``).
  The hull (Andrew's monotone chain over the points sorted by (x, y)), the ring's shoelace area and its area moments
  are computed in Python integers on the scaled coordinates - exact for any input - and rounded to float64 once.
* ``convex_area`` = hull area, ``solidity`` = |shoelace area| / ``convex_area`` (the exact ratio rounded once).
* ``orientation`` is skimage's, the expression of oracle/raster.py: with x = column and y = row, the frame
  ``instance_polygons`` emits, ``(a, b, c) = (mu_xx, -mu_xy, mu_yy)`` (each rounded once) and
  ``0.5 * atan2(-2b, c - a)``, or +-pi/4 when ``a == c``.
* NaN rules of pg_map_morph's ``ok`` / ``good``: fewer than 3 vertices -> NaN for all three; zero area -> NaN
  solidity and orientation; zero convex area -> convex_area 0 and NaN solidity.

Being exact, a ring closed (first vertex repeated) or open, clockwise or counter-clockwise, gives identical results.
"""
from __future__ import annotations

import math
from fractions import Fraction

import numpy as np

NAN = float("nan")


def _scaled(points):
    """[(x, y)] floats -> ([(X, Y)] ints, D) with x = X / D exactly."""
    ratios = [(float(x).as_integer_ratio(), float(y).as_integer_ratio()) for x, y in points]
    d = max(max(rx[1], ry[1]) for rx, ry in ratios)
    return [(rx[0] * (d // rx[1]), ry[0] * (d // ry[1])) for rx, ry in ratios], d


def _cross(o, a, b):
    return (a[0] - o[0]) * (b[1] - o[1]) - (a[1] - o[1]) * (b[0] - o[0])


def hull_area2(points) -> int:
    """Twice the area of the convex hull of integer points (monotone chain, collinear points dropped)."""
    pts = sorted(set(points))
    if len(pts) < 3:
        return 0
    lower, upper = [], []
    for p in pts:
        while len(lower) >= 2 and _cross(lower[-2], lower[-1], p) <= 0:
            lower.pop()
        lower.append(p)
    for p in reversed(pts):
        while len(upper) >= 2 and _cross(upper[-2], upper[-1], p) <= 0:
            upper.pop()
        upper.append(p)
    hull = lower[:-1] + upper[:-1]
    return sum(hull[i][0] * hull[(i + 1) % len(hull)][1] - hull[(i + 1) % len(hull)][0] * hull[i][1]
               for i in range(len(hull)))


def ring_hull_one(poly):
    """(convex_area, solidity, orientation) of one ring (sequence of [x, y]; closing vertex optional)."""
    pts = [(float(x), float(y)) for x, y in poly]
    if len(pts) < 3:
        return NAN, NAN, NAN
    p, d = _scaled(pts)
    h2 = hull_area2(p)
    convex_area = float(Fraction(h2, 2 * d * d))
    x0, y0 = p[0]
    s = sx = sy = ixx = iyy = ixy = 0
    n = len(p)
    for i in range(n):
        xa, ya = p[i][0] - x0, p[i][1] - y0
        xb, yb = p[(i + 1) % n][0] - x0, p[(i + 1) % n][1] - y0
        a = xa * yb - xb * ya
        s += a
        sx += (xa + xb) * a
        sy += (ya + yb) * a
        ixx += (ya * ya + ya * yb + yb * yb) * a
        iyy += (xa * xa + xa * xb + xb * xb) * a
        ixy += (xa * yb + 2 * xa * ya + 2 * xb * yb + xb * ya) * a
    if s == 0:
        return convex_area, NAN, NAN
    solidity = float(Fraction(abs(s), h2)) if h2 else NAN
    # central moments of the region (area-normalised), in units of 1 / D^2: cx = Sx / (6 A) with A = S / 2
    cx, cy = Fraction(sx, 3 * s), Fraction(sy, 3 * s)
    d2 = d * d
    mu_xx = float((Fraction(iyy, 6 * s) - cx * cx) / d2)
    mu_yy = float((Fraction(ixx, 6 * s) - cy * cy) / d2)
    mu_xy = float((Fraction(ixy, 12 * s) - cx * cy) / d2)
    ta, tb, tc = mu_xx, -mu_xy, mu_yy
    if ta - tc == 0:
        orientation = math.pi / 4 if tb < 0 else -math.pi / 4
    else:
        orientation = 0.5 * math.atan2(-2 * tb, tc - ta)
    return convex_area, solidity, orientation


def ring_hull_csr(poly_off, poly_xy):
    """convex_area, solidity, orientation (float64 [N] each) over CSR rings."""
    off = np.asarray(poly_off, dtype=np.int64)
    xy = np.asarray(poly_xy).reshape(-1, 2)
    n = len(off) - 1
    out = {k: np.full(n, np.nan) for k in ("convex_area", "solidity", "orientation")}
    for i in range(n):
        ca, so, orient = ring_hull_one(xy[off[i]:off[i + 1]].tolist())
        out["convex_area"][i], out["solidity"][i], out["orientation"][i] = ca, so, orient
    return out
