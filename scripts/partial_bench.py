#!/usr/bin/env python
"""Partial cost (rank-K Hausdorff distance): device time per sweep, candidate evaluations per second and pair distances
evaluated per candidate, at inlier_fraction f in {1.0, 0.99, 0.95, 0.9}, early break on (K1e-partial; K1e at f = 1)
and off (MMRS_EARLY_BREAK=0: every row scanned to its end; K1's dense sweep at f = 1).

    python scripts/partial_bench.py [OUT.json]      (default profiles/r05_partial_bench.json)

(a) the 398 bench units x 36 000 angles (0.01 deg over +-180 deg), rotation only;
(b) the 398 bench units x 361 angles x 11^2 translations (+-0.25, step 0.05), rigid;
(c) 16 units of 2 020 points (the chunked size class: 4 warps per CTA), 0.05 deg over +-10 deg;
(d) a config-3-shaped batch (1 596 units, N = M = 510) through find_best_rigid_transform, coarse-to-fine 0.01 deg,
    11^2 translations, wall-clock of the whole call. Early break off is run at f = 1 (K1) and f = 0.95 only: one
    such call evaluates ~5e13 pair distances.
Needs a CUDA device."""
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

FRACTIONS = (1.0, 0.99, 0.95, 0.9)


def gpu_info():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip()


def set_eb(flag):
    os.environ["MMRS_EARLY_BREAK"] = flag


def timed_runs(ctx, upload, reps):
    """Uploads once, runs `reps` times; median sweep-kernel and whole-run device times (ms) and the counters."""
    upload()
    sweep, total = [], []
    for _ in range(reps):
        ctx.sweep_run()
        t = ctx.timings()
        sweep.append(t["sweep_ms"])
        total.append(t["total_ms"])
    return float(np.median(sweep)), float(np.median(total)), ctx.prefilter_info()


def contour(rng, n, rot=0.0, shift=(0.0, 0.0)):
    phi = np.linspace(0, 2 * np.pi, n, endpoint=False)
    r0, e = rng.uniform(1.5, 3.0), rng.uniform(0.05, 0.35)
    r = r0 * (1 + e * np.cos(2 * phi) + 0.03 * np.cos(3 * phi + 0.4) + 0.02 * np.cos(5 * phi + 1.1))
    return np.stack([r * np.cos(phi + rot) + 4.5 + shift[0], r * np.sin(phi + rot) + 4.5 + shift[1]], 1) + \
        rng.normal(0, 0.005, (n, 2))


def kernel_name(f, flag):
    if f == 1.0:
        return "K1e" if flag == "1" else "K1 (dense)"
    return "K1e-partial" if flag == "1" else "K1e-partial, early break off"


def sweep_case(out, ctx, name, upload_of, n_cand, meta):
    for f in FRACTIONS:
        for flag in ("1", "0"):
            set_eb(flag)
            sw, tot, info = timed_runs(ctx, lambda: upload_of(f), 3 if flag == "1" else 1)
            ppc = info["eb_pairs"] / info["eb_candidates"] if info["eb_candidates"] else None
            kern = kernel_name(f, flag) if ppc is not None or flag == "0" else "K1 (K1e does not fit)"
            out["cases"].append(dict(case=name, inlier_fraction=f, early_break=flag == "1", kernel=kern,
                                     candidates=n_cand, sweep_ms=sw, run_ms=tot, M_evals_per_s=n_cand / (tot * 1e-3) / 1e6,
                                     pairs_per_candidate=ppc, **meta))
            print(out["cases"][-1], flush=True)


def main():
    out_path = Path(sys.argv[1]) if len(sys.argv) > 1 else ROOT / "profiles" / "r05_partial_bench.json"
    ctx = get_context()
    out = {"gpu": gpu_info(), "timing": "CUDA events of mmrs_sweep_run (median of 3 runs with early break on, 1 off)",
           "cases": []}
    txy, toff, rxy, roff, cen, U, n = bench.make_units(n_pairs=1)
    # (a) rotation only, 0.01 deg
    g = nat.make_grid(bench.STEP_DEG, bench.RANGE_DEG)
    sweep_case(out, ctx, "a_bench_units_rotation",
               lambda f: ctx.partial_upload(txy, toff, rxy, roff, cen, [g], mode=0, inlier_fraction=f, prefilter=1, prune=-1),
               U * g.n_cand, dict(units=U, angles=g.n_cand, points=[n, n]))
    # (b) rigid: 361 angles x 121 translations
    g1, tg = nat.make_grid(1.0, 180.0), nat.make_tgrid(0.05, 5)
    sweep_case(out, ctx, "b_bench_units_rigid",
               lambda f: ctx.partial_upload(txy, toff, rxy, roff, cen, [g1], [tg], mode=0, inlier_fraction=f),
               U * g1.n_cand * 121, dict(units=U, angles=g1.n_cand, translations=121, points=[n, n]))
    # (c) 2 020-point units
    rng = np.random.default_rng(20261021)
    tc = [contour(rng, 2020, rot=rng.normal(0, 0.1)) for _ in range(16)]
    rc = [contour(rng, 2020) for _ in range(16)]
    off_c = np.arange(17) * 2020
    g2 = nat.make_grid(0.05, 10.0)
    sweep_case(out, ctx, "c_2020_point_units",
               lambda f: ctx.partial_upload(np.concatenate(tc), off_c, np.concatenate(rc), off_c, np.full((16, 2), 4.5), [g2],
                                            mode=0, inlier_fraction=f, prefilter=1, prune=-1),
               16 * g2.n_cand, dict(units=16, angles=g2.n_cand, points=[2020, 2020]))
    # (d) config-3-shaped batch through the public function
    Ub, nb = 1596, 510
    tests = [contour(rng, nb, rot=rng.normal(0, 0.3), shift=rng.normal(0, 0.1, 2)) for _ in range(Ub)]
    refs = [contour(rng, nb) for _ in range(Ub)]
    cands = Ub * 121 * sum(nat.make_grid(s, w).n_cand for s, w in nat.stage_plan(0.01, 180.0))
    for f in FRACTIONS:
        for flag in ("1", "0"):
            if flag == "0" and f not in (1.0, 0.95):
                continue
            set_eb(flag)
            mm.find_best_rigid_transform(tests[:8], refs[:8], step_rotation_deg=0.01, range_rotation_deg=180.0,
                                         inlier_fraction=f)   # warm-up
            t0 = time.perf_counter()
            res = mm.find_best_rigid_transform(tests, refs, step_rotation_deg=0.01, range_rotation_deg=180.0,
                                               step_translation=0.05, range_translation=0.25, inlier_fraction=f)
            wall = time.perf_counter() - t0
            info = ctx.prefilter_info()
            out["cases"].append(dict(case="d_config3_find_best_rigid_transform", inlier_fraction=f, early_break=flag == "1",
                                     kernel=kernel_name(f, flag), units=Ub, points=[nb, nb], translations=121,
                                     candidates_all_stages=cands, wall_s=wall, M_evals_per_s_wall=cands / wall / 1e6,
                                     last_stage_pairs_per_candidate=info["eb_pairs"] / info["eb_candidates"]
                                     if info["eb_candidates"] else None,
                                     mean_distance=float(res["distance"].mean())))
            print(out["cases"][-1], flush=True)
    os.environ.pop("MMRS_EARLY_BREAK", None)
    out["gpu_after"] = gpu_info()
    out_path.parent.mkdir(parents=True, exist_ok=True)
    out_path.write_text(json.dumps(out, indent=1))
    print("wrote", out_path)


if __name__ == "__main__":
    main()
