#!/usr/bin/env python
"""Mean cost (modified Hausdorff distance): sweep-kernel device time of the mean form of K1 against K1 with the full
cost (MMRS_EARLY_BREAK=0) and K1e, on the same batches.

    python scripts/mean_bench.py [OUT.json]      (default profiles/r06_mean_bench.json)

(a) the 398 bench units x 36 000 angles (0.01 deg over +-180 deg), rotation only;
(b) the same units x 3 600 angles (0.1 deg);
(c) the same units x 361 angles x 11^2 translations (+-0.25, step 0.05), rigid;
(d) 8 units of N = M = 2 020 points (the chunked size class; K1e does not fit it), 0.05 deg over +-180 deg.
The kernels are timed in rounds that alternate mean / K1 / K1e; every number is the median over the rounds of the
sweep phase of mmrs_sweep_run (CUDA events, mmrs_last_timings), whose launches are one per size class.
Needs a CUDA device."""
from __future__ import annotations

import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "multimoda-rs_b200")]

import bench  # noqa: E402
from multimodars import _native as nat  # noqa: E402

ROUNDS = 5
KERNELS = (("mean K1", "mean", None), ("K1 (full cost)", "full", "0"), ("K1e (full cost)", "full", "1"))


def gpu_info():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip()


def contour(rng, n, rot=0.0):
    phi = np.linspace(0, 2 * np.pi, n, endpoint=False)
    r0, e = rng.uniform(1.5, 3.0), rng.uniform(0.05, 0.35)
    r = r0 * (1 + e * np.cos(2 * phi) + 0.03 * np.cos(3 * phi + 0.4) + 0.02 * np.cos(5 * phi + 1.1))
    return np.stack([r * np.cos(phi + rot) + 4.5, r * np.sin(phi + rot) + 4.5], 1) + rng.normal(0, 0.005, (n, 2))


def case(out, ctx, name, batch, grid, tg, n_cand, meta):
    txy, toff, rxy, roff, cen = batch
    times = {k: [] for k, *_ in KERNELS}
    launches = {}
    for _ in range(ROUNDS):
        for label, cost, eb in KERNELS:
            if eb is None:
                os.environ.pop("MMRS_EARLY_BREAK", None)
            else:
                os.environ["MMRS_EARLY_BREAK"] = eb
            tgs = None if tg is None else [tg]
            if cost == "mean":
                ctx.mean_upload(txy, toff, rxy, roff, cen, [grid], tgs, mode=0)
            elif tg is None:
                ctx.sweep_upload(txy, toff, rxy, roff, cen, [grid], mode=0, prefilter=1, prune=-1)
            else:
                ctx.rigid_upload(txy, toff, rxy, roff, cen, [grid], tgs, mode=0)
            ctx.sweep_run()   # warm-up of this upload
            ctx.sweep_run()
            t = ctx.timings()
            times[label].append(t["sweep_ms"])
            info = ctx.prefilter_info()
            launches[label] = dict(size_classes=ctx.plan()["size_classes"], run_launches=t["launches"],
                                   eb_candidates=info["eb_candidates"])
    os.environ.pop("MMRS_EARLY_BREAK", None)
    k1 = float(np.median(times["K1 (full cost)"]))
    for label, *_ in KERNELS:
        ms = float(np.median(times[label]))
        out["cases"].append(dict(case=name, kernel=label, candidates=n_cand, sweep_ms=ms, sweep_ms_rounds=times[label],
                                 M_evals_per_s=n_cand / (ms * 1e-3) / 1e6, vs_K1_full=ms / k1, **launches[label], **meta))
        print(out["cases"][-1], flush=True)


def main():
    out_path = Path(sys.argv[1]) if len(sys.argv) > 1 else ROOT / "profiles" / "r06_mean_bench.json"
    ctx = nat.Context(0)
    out = {"gpu": gpu_info(), "timing": f"CUDA events of the sweep phase of mmrs_sweep_run, median of {ROUNDS} rounds "
                                        "alternating mean / K1 / K1e", "cases": []}
    txy, toff, rxy, roff, cen, U, n = bench.make_units(n_pairs=1)
    units = (txy, toff, rxy, roff, cen)
    for name, step in (("a_bench_units_0.01deg", 0.01), ("b_bench_units_0.1deg", 0.1)):
        g = nat.make_grid(step, 180.0)
        case(out, ctx, name, units, g, None, U * g.n_cand, dict(units=U, angles=g.n_cand, points=[n, n]))
    g1, tg = nat.make_grid(1.0, 180.0), nat.make_tgrid(0.05, 5)
    case(out, ctx, "c_bench_units_rigid", units, g1, tg, U * g1.n_cand * 121,
         dict(units=U, angles=g1.n_cand, translations=121, points=[n, n]))
    rng = np.random.default_rng(20261021)
    tc = [contour(rng, 2020, rot=rng.normal(0, 0.1)) for _ in range(8)]
    rc = [contour(rng, 2020) for _ in range(8)]
    off_c = np.arange(9) * 2020
    g2 = nat.make_grid(0.05, 180.0)
    case(out, ctx, "d_2020_point_units", (np.concatenate(tc), off_c, np.concatenate(rc), off_c, np.full((8, 2), 4.5)),
         g2, None, 8 * g2.n_cand, dict(units=8, angles=g2.n_cand, points=[2020, 2020]))
    out["gpu_after"] = gpu_info()
    ctx.close()
    out_path.parent.mkdir(parents=True, exist_ok=True)
    out_path.write_text(json.dumps(out, indent=1))
    print("wrote", out_path)


if __name__ == "__main__":
    main()
