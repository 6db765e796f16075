"""f64 restatement of rigid candidates (include/mmrs_b200.h "rigid candidates"), the reference for the rigid tests.

The reference project has no translation search, so parity is defined by this restatement: the rotation of the
oracle's cost closures (mode 0: align_within.rs:99-105 with the angle == 0.0 identity, mode 1:
align_between.rs:189-216), then + (tx, ty), then hausdorff_distance (process_utils.rs:78-121), every operation one
IEEE f64 rounding (numpy elementwise, no fused multiply-add; cos / sin from the C library like the oracle's)."""
from __future__ import annotations

import math

import numpy as np

from oracle import oracle_py as ora


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


def _finite(a):
    a = np.asarray(a, dtype=np.float64).reshape(-1, 2)
    return a[np.isfinite(a).all(axis=1)]


def _directed(a, b):
    """directed_hausdorff (process_utils.rs:84-121) of every translated copy a[k] (K, N, 2) onto b (M, 2)."""
    dx = a[:, :, None, 0] - b[None, None, :, 0]
    dy = a[:, :, None, 1] - b[None, None, :, 1]
    d2 = dx * dx + dy * dy
    mn = d2.min(axis=2)                                   # (K, N): finite for finite points
    return np.sqrt(np.maximum(mn, 0.0).max(axis=1))


def costs_at_angle(test, ref, centre, mode, angle, offsets):
    """f64 cost of (angle, offsets[k]) for every k."""
    t, r = _finite(test), _finite(ref)
    if len(t) == 0 or len(r) == 0:
        return np.zeros(len(offsets))
    if mode == 0 and angle == 0.0:
        rx, ry = t[:, 0].copy(), t[:, 1].copy()
    else:
        c, s = math.cos(angle), math.sin(angle)
        x, y = t[:, 0] - centre[0], t[:, 1] - centre[1]
        rx = (x * c - y * s) + centre[0]
        ry = (x * s + y * c) + centre[1]
    off = np.asarray(offsets, dtype=np.float64).reshape(-1, 2)
    moved = np.stack([rx[None, :] + off[:, 0:1], ry[None, :] + off[:, 1:2]], axis=2)   # (K, N, 2)
    fwd = np.array([_directed(r[None], m)[0] for m in moved])                         # reference -> moved
    bwd = _directed(moved, r)                                                          # moved -> reference
    return np.fmax(fwd, bwd)


def rigid_search(test, ref, centre, mode, angles, offsets):
    """Brute force over angles x offsets. Returns (flattened index, costs (C, T))."""
    costs = np.stack([costs_at_angle(test, ref, centre, mode, a, offsets) for a in angles]) if len(angles) else \
        np.zeros((0, len(offsets)))
    flat = costs.reshape(-1)
    return (int(np.argmin(flat)) if len(flat) else -1), costs     # argmin: first occurrence = leftmost


def _search_range(test, ref, centre, mode, offsets, step, rng, center, limes):
    """search_range with cost(angle) = min_j H(angle, t_j): (angle, j, cost)."""
    grid, fb = ora.search_grid(step, rng, center, limes)
    if grid is None or len(grid) == 0:
        return fb, -1, 0.0
    best = None
    for a in grid:
        c = costs_at_angle(test, ref, centre, mode, a, offsets)
        j = int(np.argmin(c))
        if best is None or c[j] < best[2]:
            best = (float(a), j, float(c[j]))
    return best


def rigid_coarse_to_fine(test, ref, centre, mode, step_deg, range_deg, offsets, bruteforce=False):
    """coarse_to_fine (align_within.rs:208-246) over cost(angle) = min_j H(angle, t_j); the leftmost flattened
    arg-min of a stage is its leftmost angle of least cost, then the leftmost j at that angle.
    Returns (angle, j, tx, ty, distance) of the last stage."""
    def sr(step, rng, center):
        return _search_range(test, ref, centre, mode, offsets, step, rng, center, range_deg)

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
