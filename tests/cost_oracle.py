"""f64 restatement of the sweep costs, the reference for the rigid, partial and mean-cost tests.

A candidate (angle, t) moves the finite test points by the rotation of the oracle's cost closures (mode 0:
align_within.rs:99-105 with the angle == 0.0 identity, mode 1: align_between.rs:189-216), then + (tx, ty), every
operation one IEEE f64 rounding (numpy elementwise, no fused multiply-add; cos / sin from the C library like the
oracle's). Each direction reduces its row minima of dx * dx + dy * dy to one value; the cost is the larger direction
(0 when either finite set is empty). The reference project has no translation search, so parity is defined here.

cost names the reduction (include/mmrs_b200.h):
- "full" ("rigid candidates"): hausdorff_distance (process_utils.rs:78-121), sqrt of the largest row minimum; an
  overflowed (inf) minimum stays inf.
- "partial" ("partial cost"): sqrt of the (q + 1)-th largest row minimum, duplicates counted and a non-finite minimum
  counted as 0, with K(n) = max(1, ceil(f n)) and q(n) = n - K(n) over the finite points of the set.
- "mean" ("mean cost"): the row values sqrt(minimum) (a non-finite minimum counts as 0) summed sequentially in point
  order (np.cumsum, never np.sum, which sums pairwise), then divided once by the count.

Every function takes a batch of translations at once: elementwise arithmetic, min, np.sort and np.cumsum along the
last axis give the same bits as the one-candidate 1-D forms."""
from __future__ import annotations

import math

import numpy as np

from oracle import oracle_py as ora


def finite(a):
    a = np.asarray(a, dtype=np.float64).reshape(-1, 2)
    return a[np.isfinite(a).all(axis=1)]


def tgrid_offsets(t0x, t0y, step, half_n):
    """Translation j = jy (2 half_n + 1) + jx: (t0x + (jx - half_n) step, t0y + (jy - half_n) step)."""
    w = 2 * half_n + 1
    out = np.empty((w * w, 2))
    for j in range(w * w):
        jy, jx = divmod(j, w)
        out[j] = (t0x + float(jx - half_n) * step, t0y + float(jy - half_n) * step)
    return out


def offsets_of(tg):
    """tgrid_offsets of an mmrs_tgrid mirror (multimodars._native.TGrid)."""
    return tgrid_offsets(tg.t0x, tg.t0y, tg.step, tg.half_n)


def k_of(n, f):
    """K(n) = max(1, ceil(f n)) in f64, as written (0 for an empty set)."""
    return 0 if n <= 0 else max(1, math.ceil(f * n))


def q_of(n, f):
    return 0 if n <= 0 else n - k_of(n, f)


def transformed(test, centre, mode, angle, t=(0.0, 0.0)):
    """The finite test points rotated by the batch's mode, then + t: (n, 2) for one t, (T, n, 2) for t of shape
    (T, 1, 2)."""
    p = finite(test)
    if mode == 0 and angle == 0.0:
        rx, ry = p[:, 0], p[:, 1]
    else:
        c, s = math.cos(angle), math.sin(angle)
        x, y = p[:, 0] - centre[0], p[:, 1] - centre[1]
        rx = (x * c - y * s) + centre[0]
        ry = (x * s + y * c) + centre[1]
    return np.stack([rx, ry], axis=1) + np.asarray(t, dtype=np.float64)


def row_minima(rows, pts):
    """min over pts of dx * dx + dy * dy for every row point: rows (..., n, 2), pts (..., m, 2) -> (..., n)."""
    d2 = rows[..., :, None, 0] - pts[..., None, :, 0]
    dy = rows[..., :, None, 1] - pts[..., None, :, 1]
    d2 *= d2                                  # in place: the (T, n, m) temporaries dominate the oracle's time
    dy *= dy
    d2 += dy
    return d2.min(axis=-1)


def row_values(rows, pts):
    """The mean cost's terms: sqrt of every row minimum (a non-finite minimum counts as 0)."""
    mn = row_minima(rows, pts)
    ok = np.isfinite(mn)
    return np.where(ok, np.sqrt(np.where(ok, mn, 0.0)), 0.0)


def directed(rows, pts, cost, f=1.0):
    """One direction's value, rows (..., n, 2) onto pts (..., m, 2) -> (...)."""
    if cost == "mean":
        return np.cumsum(row_values(rows, pts), axis=-1)[..., -1] / rows.shape[-2]
    mn = row_minima(rows, pts)
    if cost == "full":
        return np.sqrt(np.maximum(mn, 0.0).max(axis=-1))
    if cost == "partial":
        n = mn.shape[-1]
        return np.sqrt(np.sort(np.where(np.isfinite(mn), mn, 0.0), axis=-1)[..., n - 1 - q_of(n, f)])
    raise ValueError(f"unknown cost {cost!r}")


def directions(test, ref, centre, mode, angle, offsets, cost, f=1.0):
    """(fwd, bwd), one value per translation in offsets: reference -> transformed test set and transformed test set ->
    reference (both 0 when either finite set is empty)."""
    off = np.asarray(offsets, dtype=np.float64).reshape(-1, 2)
    r, moved = finite(ref), transformed(test, centre, mode, angle, off[:, None, :])
    if moved.shape[1] == 0 or len(r) == 0:
        return np.zeros(len(off)), np.zeros(len(off))
    return directed(r, moved, cost, f), directed(moved, r, cost, f)


def costs_at_angle(test, ref, centre, mode, angle, offsets, cost, f=1.0):
    """f64 cost of (angle, offsets[k]) for every k."""
    return np.fmax(*directions(test, ref, centre, mode, angle, offsets, cost, f))


def candidate_cost(test, ref, centre, mode, angle, t, cost, f=1.0):
    """f64 cost of one candidate (angle, t)."""
    return float(costs_at_angle(test, ref, centre, mode, angle, [t], cost, f)[0])


def search(test, ref, centre, mode, angles, offsets, cost, f=1.0):
    """Brute force over angles x offsets (flattened c = i T + j). Returns (leftmost arg-min, costs (C, T))."""
    off = np.asarray(offsets, dtype=np.float64).reshape(-1, 2)
    costs = np.array([costs_at_angle(test, ref, centre, mode, a, off, cost, f) for a in angles]).reshape(len(angles),
                                                                                                        len(off))
    flat = costs.reshape(-1)
    return (int(np.argmin(flat)) if len(flat) else -1), costs     # argmin: first occurrence = leftmost


def coarse_to_fine(test, ref, centre, mode, step_deg, range_deg, offsets, cost, f=1.0, bruteforce=False):
    """coarse_to_fine (align_within.rs:208-246) over cost(angle) = min_j cost(angle, t_j); the leftmost flattened
    arg-min of a stage is its leftmost angle of least cost, then the leftmost j at that angle.
    Returns (angle, j, tx, ty, distance) of the last stage."""
    off = np.asarray(offsets, dtype=np.float64).reshape(-1, 2)

    def search_range(step, rng, center):
        grid, fb = ora.search_grid(step, rng, center, range_deg)
        if grid is None or len(grid) == 0:
            return fb, -1, 0.0
        best = None
        for a in grid:
            c = costs_at_angle(test, ref, centre, mode, a, off, cost, f)
            j = int(np.argmin(c))
            if best is None or c[j] < best[2]:
                best = (float(a), j, float(c[j]))
        return best

    def window(w):
        return w if range_deg > w else range_deg

    if bruteforce or step_deg >= 1.0:
        stages = [(step_deg, range_deg)]
    elif step_deg >= 0.1:
        stages = [(1.0, range_deg), (step_deg, window(5.0))]
    elif step_deg >= 0.01:
        stages = [(1.0, range_deg), (0.1, window(5.0)), (step_deg, window(10.0 * step_deg))]
    else:
        stages = [(1.0, range_deg), (0.1, window(5.0)), (0.01, window(0.1)), (step_deg, window(10.0 * step_deg))]
    a, j, d = None, -1, 0.0
    for step, rng in stages:                      # each stage after the first is centred on the previous stage's angle
        a, j, d = search_range(step, rng, a)
    tx, ty = (off[j] if j >= 0 else (0.0, 0.0))
    return a, j, float(tx), float(ty), d


def crafted_order_case():
    """A test set whose backward row values are 1 followed by twenty values of 2^-53 (one reference point at the
    origin): summed left to right, each tiny term rounds away against 1; summed pairwise (np.sum), they do not."""
    xs = np.concatenate([[1.0], np.full(20, 2.0 ** -53)])
    return np.stack([xs, np.zeros_like(xs)], axis=1), np.zeros((1, 2))
