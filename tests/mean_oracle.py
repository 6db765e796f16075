"""f64 restatement of the mean cost (include/mmrs_b200.h "mean cost"), the reference for the mean-cost tests.

The transform is the rigid oracle's (tests/partial_oracle.transformed: the rotation of the oracle's cost closures,
then + (tx, ty), every operation one IEEE f64 rounding). A point's row value is sqrt of its minimum squared distance
to the other set (a non-finite minimum counts as 0); each direction sums its row values sequentially in point order
(np.cumsum, never np.sum, which sums pairwise) and divides once by the count; the cost is the larger direction."""
from __future__ import annotations

import numpy as np

from oracle import oracle_py as ora
from tests.partial_oracle import _finite, transformed


def row_values(rows, pts):
    """sqrt(min over pts of dx * dx + dy * dy) for every row point (unfused; a non-finite minimum counts as 0)."""
    dx = rows[:, None, 0] - pts[None, :, 0]
    dy = rows[:, None, 1] - pts[None, :, 1]
    mn = (dx * dx + dy * dy).min(axis=1)
    return np.where(np.isfinite(mn), np.sqrt(np.where(np.isfinite(mn), mn, 0.0)), 0.0)


def seq_mean(v):
    """Sequential left-to-right f64 sum in point order, then one division."""
    return float(np.cumsum(v)[-1]) / len(v)


def directions(test, ref, centre, mode, angle, t=(0.0, 0.0)):
    """(fwd, bwd): reference -> transformed test set, transformed test set -> reference (0, 0 for an empty set)."""
    r = _finite(ref)
    moved = transformed(test, centre, mode, angle, t)
    if len(moved) == 0 or len(r) == 0:
        return 0.0, 0.0
    return seq_mean(row_values(r, moved)), seq_mean(row_values(moved, r))


def cost(test, ref, centre, mode, angle, t=(0.0, 0.0)):
    """f64 mean cost of one candidate (angle, t)."""
    return float(np.fmax(*directions(test, ref, centre, mode, angle, t)))


def search(test, ref, centre, mode, angles, offsets):
    """Brute force over angles x offsets (flattened c = i T + j). Returns (leftmost arg-min, costs (C, T))."""
    offsets = np.asarray(offsets, dtype=np.float64).reshape(-1, 2)
    costs = np.array([[cost(test, ref, centre, mode, a, t) for t in offsets] for a in angles]).reshape(len(angles),
                                                                                                     len(offsets))
    flat = costs.reshape(-1)
    return (int(np.argmin(flat)) if len(flat) else -1), costs


def coarse_to_fine(test, ref, centre, mode, step_deg, range_deg, offsets, bruteforce=False):
    """tests/rigid_oracle.rigid_coarse_to_fine with the mean cost. Returns (angle, j, tx, ty, distance)."""
    offsets = np.asarray(offsets, dtype=np.float64).reshape(-1, 2)

    def sr(step, rng, center):
        grid, fb = ora.search_grid(step, rng, center, range_deg)
        if grid is None or len(grid) == 0:
            return fb, -1, 0.0
        best = None
        for a in grid:
            c = np.array([cost(test, ref, centre, mode, a, t) for t in offsets])
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


def crafted_order_case():
    """A test set whose backward row values are 1 followed by twenty values of 2^-53 (one reference point at the
    origin): summed left to right, each tiny term rounds away against 1; summed pairwise (np.sum), they do not."""
    xs = np.concatenate([[1.0], np.full(20, 2.0 ** -53)])
    return np.stack([xs, np.zeros_like(xs)], axis=1), np.zeros((1, 2))
