#!/usr/bin/env python
"""Rigid candidates (angle grid x translation grid): device time per sweep, candidate evaluations per second and pair
distances evaluated per candidate, for K1e (default) and K1 (MMRS_EARLY_BREAK=0).

    python scripts/rigid_bench.py [OUT.json]      (default profiles/r04_rigid_bench.json)

(a) the 398 bench units x 361 angles (1 deg over +-180 deg) x 11^2 translations (+-0.25, step 0.05);
(b) a config-3-shaped batch (1 596 units, N = M = 510) through find_best_rigid_transform, coarse-to-fine 0.01 deg over
    +-180 deg, 11^2 translations (wall-clock of the whole call: three stages, uploads and downloads included);
(c) the (a) units with half_n = 0 against the rotation-only sweep on the same grid;
plus the CPU f64 restatement (tests/rigid_oracle.py) on a few candidates as a baseline. Needs a CUDA device."""
from __future__ import annotations

import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "multimoda-rs_b200")]

import bench  # noqa: E402
import multimodars as mm  # noqa: E402
from multimodars import _native as nat  # noqa: E402
from multimodars._processing import get_context  # noqa: E402

REPS = 3


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip()
    return q


def set_eb(flag):
    if flag is None:
        os.environ.pop("MMRS_EARLY_BREAK", None)
    else:
        os.environ["MMRS_EARLY_BREAK"] = flag


def timed_runs(ctx, upload):
    """Uploads once, runs REPS times; median sweep-kernel and whole-run device times (ms) and the K1e counters."""
    upload()
    sweep, total = [], []
    for _ in range(REPS):
        ctx.sweep_run()
        t = ctx.timings()
        sweep.append(t["sweep_ms"])
        total.append(t["total_ms"])
    info = ctx.prefilter_info()
    return float(np.median(sweep)), float(np.median(total)), info


def contour(rng, n, rot=0.0, shift=(0.0, 0.0)):
    phi = np.linspace(0, 2 * np.pi, n, endpoint=False)
    r0, e = rng.uniform(1.5, 3.0), rng.uniform(0.05, 0.35)
    r = r0 * (1 + e * np.cos(2 * phi) + 0.03 * np.cos(3 * phi + 0.4) + 0.02 * np.cos(5 * phi + 1.1))
    return np.stack([r * np.cos(phi + rot) + 4.5 + shift[0], r * np.sin(phi + rot) + 4.5 + shift[1]], 1) + \
        rng.normal(0, 0.005, (n, 2))


def main():
    out_path = Path(sys.argv[1]) if len(sys.argv) > 1 else ROOT / "profiles" / "r04_rigid_bench.json"
    ctx = get_context()
    out = {"gpu": gpu_info(), "reps": REPS, "timing": "CUDA events of mmrs_sweep_run (median of reps)", "cases": []}
    txy, toff, rxy, roff, cen, U, n = bench.make_units(n_pairs=1)
    g = nat.make_grid(1.0, 180.0)
    tg = nat.make_tgrid(0.05, 5)
    T = 121
    # (a) rigid sweep of the bench units
    for flag, kern in (("1", "K1e"), ("0", "K1")):
        set_eb(flag)
        sw, tot, info = timed_runs(ctx, lambda: ctx.rigid_upload(txy, toff, rxy, roff, cen, [g], [tg], mode=0))
        c = U * g.n_cand * T
        out["cases"].append({"case": "a_bench_units_rigid", "kernel": kern, "units": U, "angles": g.n_cand,
                             "translations": T, "candidates": c, "points": [n, n], "sweep_ms": sw, "run_ms": tot,
                             "M_evals_per_s": c / (tot * 1e-3) / 1e6,
                             "pairs_per_candidate": info["eb_pairs"] / info["eb_candidates"] if info["eb_candidates"] else n * n})
        print(out["cases"][-1], flush=True)
    # (c) half_n = 0 against the rotation-only sweep, same units and angles
    z = nat.make_tgrid(0.0, 0)
    for flag, kern in (("1", "K1e"), ("0", "K1")):
        set_eb(flag)
        sw0, tot0, i0 = timed_runs(ctx, lambda: ctx.sweep_upload(txy, toff, rxy, roff, cen, [g], mode=0, prefilter=1,
                                                                 prune=-1))
        sw1, tot1, i1 = timed_runs(ctx, lambda: ctx.rigid_upload(txy, toff, rxy, roff, cen, [g], [z], mode=0))
        out["cases"].append({"case": "c_half_n_0_vs_rotation_only", "kernel": kern, "units": U, "angles": g.n_cand,
                             "rotation_only_sweep_ms": sw0, "rotation_only_run_ms": tot0, "rigid_sweep_ms": sw1,
                             "rigid_run_ms": tot1, "rigid_over_rotation_only": tot1 / tot0})
        print(out["cases"][-1], flush=True)
    # (b) config-3-shaped batch through the public function
    rng = np.random.default_rng(20261020)
    Ub, nb = 1596, 510
    tests = [contour(rng, nb, rot=rng.normal(0, 0.3), shift=rng.normal(0, 0.1, 2)) for _ in range(Ub)]
    refs = [contour(rng, nb) for _ in range(Ub)]
    for flag, kern in (("1", "K1e"), ("0", "K1")):
        set_eb(flag)
        mm.find_best_rigid_transform(tests[:8], refs[:8], step_rotation_deg=0.01, range_rotation_deg=180.0)   # warm-up
        t0 = time.perf_counter()
        res = mm.find_best_rigid_transform(tests, refs, step_rotation_deg=0.01, range_rotation_deg=180.0,
                                           step_translation=0.05, range_translation=0.25)
        wall = time.perf_counter() - t0
        info = ctx.prefilter_info()
        cands = Ub * T * sum(nat.make_grid(s, w).n_cand for s, w in nat.stage_plan(0.01, 180.0))
        out["cases"].append({"case": "b_config3_find_best_rigid_transform", "kernel": kern, "units": Ub, "points": [nb, nb],
                             "stages": nat.stage_plan(0.01, 180.0), "translations": T, "candidates_all_stages": cands,
                             "wall_s": wall, "M_evals_per_s_wall": cands / wall / 1e6,
                             "last_stage_pairs_per_candidate": info["eb_pairs"] / info["eb_candidates"] if info["eb_candidates"] else nb * nb,
                             "mean_distance": float(res["distance"].mean())})
        print(out["cases"][-1], flush=True)
    set_eb(None)
    # CPU baseline: the f64 restatement (numpy, one thread) on a few candidates of two bench units
    from tests import rigid_oracle as ro

    offs = ro.offsets_of(tg)
    t0 = time.perf_counter()
    k = 0
    for u in (0, U // 2):
        for a in (0.1, -0.7):
            ro.costs_at_angle(txy[toff[u]:toff[u + 1]], rxy[roff[u]:roff[u + 1]], cen[u], 0, a, offs)
            k += T
    dt = time.perf_counter() - t0
    out["cpu_oracle"] = {"what": "tests/rigid_oracle.py costs_at_angle (numpy f64, 1 process)", "candidates": k,
                         "s": dt, "evals_per_s": k / dt, "points": [n, n]}
    print(out["cpu_oracle"], flush=True)
    out["gpu_after"] = gpu_info()
    out_path.parent.mkdir(parents=True, exist_ok=True)
    out_path.write_text(json.dumps(out, indent=1))
    print("wrote", out_path)


if __name__ == "__main__":
    main()
