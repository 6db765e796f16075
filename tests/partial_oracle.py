"""f64 restatement of the partial cost (include/mmrs_b200.h "partial cost"), the reference for the partial tests.

The transform is tests/rigid_oracle.py's (the rotation of the oracle's cost closures, then + (tx, ty), every operation
one IEEE f64 rounding); the directed value is the (q + 1)-th largest row minimum instead of the largest, with
K(n) = max(1, ceil(f n)) and q(n) = n - K(n) over the finite points of each set."""
from __future__ import annotations

import math

import numpy as np

from oracle import oracle_py as ora


def k_of(n, f):
    """K(n) = max(1, ceil(f n)) in f64, as written (0 for an empty set)."""
    return 0 if n <= 0 else max(1, math.ceil(f * n))


def q_of(n, f):
    return 0 if n <= 0 else n - k_of(n, f)


def _finite(a):
    a = np.asarray(a, dtype=np.float64).reshape(-1, 2)
    return a[np.isfinite(a).all(axis=1)]


def _kth(mn, q):
    """(q + 1)-th largest of the row minima (duplicates counted; a non-finite minimum counts as 0)."""
    v = np.where(np.isfinite(mn), mn, 0.0)
    return np.sort(v)[len(v) - 1 - q]


def _directed(rows, pts, q):
    dx = rows[:, None, 0] - pts[None, :, 0]
    dy = rows[:, None, 1] - pts[None, :, 1]
    return np.sqrt(_kth((dx * dx + dy * dy).min(axis=1), q))


def transformed(test, centre, mode, angle, t=(0.0, 0.0)):
    """The rigid oracle's transform of the (finite) test points: rotation of the batch's mode, then + t."""
    t_ = _finite(test)
    if mode == 0 and angle == 0.0:
        rx, ry = t_[:, 0].copy(), t_[:, 1].copy()
    else:
        c, s = math.cos(angle), math.sin(angle)
        x, y = t_[:, 0] - centre[0], t_[:, 1] - centre[1]
        rx = (x * c - y * s) + centre[0]
        ry = (x * s + y * c) + centre[1]
    return np.stack([rx + t[0], ry + t[1]], axis=1)


def cost(test, ref, centre, mode, angle, t, f):
    """f64 partial cost of one candidate (angle, t)."""
    r = _finite(ref)
    moved = transformed(test, centre, mode, angle, t)
    if len(moved) == 0 or len(r) == 0:
        return 0.0
    fwd = _directed(r, moved, q_of(len(r), f))        # reference -> transformed, q = q(m)
    bwd = _directed(moved, r, q_of(len(moved), f))    # transformed -> reference, q = q(n)
    return float(np.fmax(fwd, bwd))


def search(test, ref, centre, mode, angles, offsets, f):
    """Brute force over angles x offsets (flattened c = i T + j). Returns (leftmost arg-min, costs (C, T))."""
    offsets = np.asarray(offsets, dtype=np.float64).reshape(-1, 2)
    costs = np.array([[cost(test, ref, centre, mode, a, t, f) for t in offsets] for a in angles]).reshape(len(angles),
                                                                                                      len(offsets))
    flat = costs.reshape(-1)
    return (int(np.argmin(flat)) if len(flat) else -1), costs


def coarse_to_fine(test, ref, centre, mode, step_deg, range_deg, offsets, f, bruteforce=False):
    """tests/rigid_oracle.rigid_coarse_to_fine with the partial cost. Returns (angle, j, tx, ty, distance)."""
    offsets = np.asarray(offsets, dtype=np.float64).reshape(-1, 2)

    def sr(step, rng, center):
        grid, fb = ora.search_grid(step, rng, center, range_deg)
        if grid is None or len(grid) == 0:
            return fb, -1, 0.0
        best = None
        for a in grid:
            c = np.array([cost(test, ref, centre, mode, a, t, f) for t in offsets])
            j = int(np.argmin(c))
            if best is None or c[j] < best[2]:
                best = (float(a), j, float(c[j]))
        return best

    if bruteforce or step_deg >= 1.0:
        a, j, d = sr(step_deg, range_deg, None)
    elif 0.1 <= step_deg < 1.0:
        a0 = sr(1.0, range_deg, None)[0]
        a, j, d = sr(step_deg, 5.0 if range_deg > 5.0 else range_deg, a0)
    elif 0.01 <= step_deg < 0.1:
        a0 = sr(1.0, range_deg, None)[0]
        a1 = sr(0.1, 5.0 if range_deg > 5.0 else range_deg, a0)[0]
        a, j, d = sr(step_deg, 10.0 * step_deg if range_deg > 10.0 * step_deg else range_deg, a1)
    else:
        a0 = sr(1.0, range_deg, None)[0]
        a1 = sr(0.1, 5.0 if range_deg > 5.0 else range_deg, a0)[0]
        a2 = sr(0.01, 0.1 if range_deg > 0.1 else range_deg, a1)[0]
        a, j, d = sr(step_deg, 10.0 * step_deg if range_deg > 10.0 * step_deg else range_deg, a2)
    tx, ty = (offsets[j] if j >= 0 else (0.0, 0.0))
    return a, j, float(tx), float(ty), d
