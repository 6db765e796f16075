"""Rigid Hausdorff registration: the best rotation AND translation of one point set onto another.

The reference aligns centroids and then searches the rotation only (align_within.rs:84-90, align_between.rs:33-40).
A side branch, a calcification or a catheter artefact moves a centroid, so the Hausdorff-optimal rotation is then
found about the wrong offset. `find_best_rigid_transform` searches a translation grid alongside the rotation sweep:
every candidate (theta, tx, ty) is scored by the symmetric Hausdorff distance on the GPU (mmrs_rigid_sweep_*,
include/mmrs_b200.h "rigid candidates"). This has no reference counterpart; tests/rigid_oracle.py restates it."""
from __future__ import annotations

import math
import numbers

import numpy as np

from . import _native as nat

RIGID_TRANSFORM_DTYPE = np.dtype([("angle_rad", "<f8"), ("rotation_deg", "<f8"), ("tx", "<f8"), ("ty", "<f8"),
                                  ("distance", "<f8"), ("n_ties", "<i4")])


def _as_sets(x, name):
    """One (N, >=2) array or a sequence of them -> list of (N, 2) float64 arrays."""
    if isinstance(x, np.ndarray) and x.ndim == 2:
        sets = [x]
    elif isinstance(x, np.ndarray) and x.ndim == 3:
        sets = list(x)
    elif isinstance(x, (list, tuple)):
        sets = list(x)
    else:
        raise TypeError(f"{name} must be an (N, >=2) array or a sequence of them")
    out = []
    for s in sets:
        a = np.asarray(s, dtype=np.float64)
        if a.ndim != 2 or a.shape[1] < 2:
            raise ValueError(f"{name}: every point set must have shape (N, >=2), got {a.shape}")
        out.append(np.ascontiguousarray(a[:, :2]))
    return out


def _global_centroid(a):
    """align_between.rs:260-271: sequential sums of x and y over the points, divided by n."""
    if len(a) == 0:
        return 0.0, 0.0
    n = float(len(a))
    return float(np.cumsum(a[:, 0])[-1]) / n, float(np.cumsum(a[:, 1])[-1]) / n


def _finite_number(v, name):
    try:
        f = float(v)
    except (TypeError, ValueError):
        raise TypeError(f"{name} must be a number") from None
    if not math.isfinite(f):
        raise ValueError(f"{name} must be finite")
    return f


def find_best_rigid_transform(test, reference, step_rotation_deg=0.5, range_rotation_deg=90.0, step_translation=0.05,
                              range_translation=0.25, centre=None, bruteforce=False, inlier_fraction=1.0,
                              cost="hausdorff"):
    """Best rigid transform (rotation about `centre`, then translation) of `test` onto `reference`.

    Candidates: rotations on the grid of the rotation sweep (coarse-to-fine like find_best_rotation, or one stage
    with `bruteforce`), each combined with every translation (jx, jy) * step_translation, |jx|, |jy| <= half_n,
    half_n = floor(range_translation / step_translation). Every stage searches the full translation grid around
    (0, 0). Cost: the inter-pullback closure (rotation about `centre`, default the reference set's mean), plus the
    translation, scored by the symmetric Hausdorff distance in f64; the leftmost arg-min over (angle, ty, tx) wins.

    test, reference: one (N, >=2) array each (only x, y are used), or equal-length sequences of them; all pairs run
    as one batched sweep per stage. `centre`: one (x, y) for every pair, or one per pair.
    inlier_fraction: f < 1 scores the partial (rank-K) Hausdorff distance instead (include/mmrs_b200.h "partial
    cost"): in each direction the worst n - max(1, ceil(f n)) points of a set do not count, so a few artefact points
    (a side-branch bulge, a calcification) do not decide the transform. 1.0 is the full distance.
    cost: "hausdorff" (the symmetric Hausdorff distance, or its partial form above) or "mean": the modified Hausdorff
    distance (include/mmrs_b200.h "mean cost"), the larger of the two directions' mean closest-point distances, so
    every point counts. "mean" takes inlier_fraction = 1 only. range_translation = 0 searches the rotation only.
    Returns a structured array, one row per pair: angle_rad, rotation_deg, tx, ty, distance, n_ties."""
    tests, refs = _as_sets(test, "test"), _as_sets(reference, "reference")
    if len(tests) != len(refs):
        raise ValueError(f"test and reference hold {len(tests)} and {len(refs)} point sets")
    if len(tests) == 0:
        raise ValueError("no point sets given")
    step_r = _finite_number(step_rotation_deg, "step_rotation_deg")
    range_r = _finite_number(range_rotation_deg, "range_rotation_deg")
    step_t = _finite_number(step_translation, "step_translation")
    range_t = _finite_number(range_translation, "range_translation")
    if step_r <= 0.0:
        raise ValueError("step_rotation_deg must be > 0")
    if range_r <= 0.0:
        raise ValueError("range_rotation_deg must be > 0")
    if step_t <= 0.0:
        raise ValueError("step_translation must be > 0")
    if range_t < 0.0:
        raise ValueError("range_translation must be >= 0")
    if isinstance(inlier_fraction, bool) or not isinstance(inlier_fraction, numbers.Real):
        raise TypeError("inlier_fraction must be a number")
    frac = _finite_number(inlier_fraction, "inlier_fraction")
    if not 0.0 < frac <= 1.0:
        raise ValueError("inlier_fraction must satisfy 0 < inlier_fraction <= 1")
    if not isinstance(cost, str) or cost not in ("hausdorff", "mean"):
        raise ValueError(f"cost must be 'hausdorff' or 'mean', got {cost!r}")
    if cost == "mean" and frac != 1.0:
        raise ValueError("cost='mean' takes inlier_fraction = 1 only (a trimmed mean is not supported)")
    half_n = int(math.floor(range_t / step_t + 1e-9))
    if half_n > 1000:
        raise ValueError(f"range_translation / step_translation = {half_n} translations per side; at most 1000")
    U = len(tests)
    if centre is None:
        cen = np.array([_global_centroid(r) for r in refs], dtype=np.float64).reshape(U, 2)
    else:
        cen = np.asarray(centre, dtype=np.float64)
        if cen.shape == (2,):
            cen = np.tile(cen, (U, 1))
        if cen.shape != (U, 2):
            raise ValueError(f"centre must be one (x, y) or one per pair, got shape {cen.shape}")
    if not np.isfinite(cen).all():
        raise ValueError("centre must be finite")

    stages = [(step_r, range_r)] if bruteforce else nat.stage_plan(step_r, range_r)
    tg = nat.make_tgrid(step_t, half_n)
    test_xy, ref_xy = np.concatenate(tests), np.concatenate(refs)
    test_off = np.concatenate([[0], np.cumsum([len(t) for t in tests])]).astype(np.int64)
    ref_off = np.concatenate([[0], np.cumsum([len(r) for r in refs])]).astype(np.int64)

    from ._processing import get_context   # the process-wide context (created on first use)

    ctx = get_context()
    res = None
    for k, (step, window) in enumerate(stages):
        if k == 0 and cost == "mean":
            ctx.mean_upload(test_xy, test_off, ref_xy, ref_off, cen, [nat.make_grid(step, window, None, range_r)], [tg],
                            mode=1)
        elif k == 0 and frac < 1.0:
            ctx.partial_upload(test_xy, test_off, ref_xy, ref_off, cen, [nat.make_grid(step, window, None, range_r)], [tg],
                               mode=1, inlier_fraction=frac)
        elif k == 0:   # stage 0 centred on 0; stage k > 0 on the previous stage's angle, clipped to +-range_rotation_deg
            ctx.rigid_upload(test_xy, test_off, ref_xy, ref_off, cen, [nat.make_grid(step, window, None, range_r)], [tg],
                             mode=1)
        else:
            grids = [nat.make_grid(step, window, float(a), range_r) for a in res["best_angle"]]
            ctx.rigid_regrid(grids, [tg], grid_of_unit=np.arange(U, dtype=np.int32))
        ctx.sweep_run()
        res = ctx.rigid_download()
    out = np.zeros(U, dtype=RIGID_TRANSFORM_DTYPE)
    out["angle_rad"] = res["best_angle"]
    out["rotation_deg"] = np.degrees(res["best_angle"])
    out["tx"] = res["best_tx"]
    out["ty"] = res["best_ty"]
    out["distance"] = res["best_dist"]
    out["n_ties"] = res["n_ties"]
    return out
