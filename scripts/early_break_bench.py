#!/usr/bin/env python
"""K1 (k_sweep) against K1e (k_sweep_eb, early-break directed passes) per workload class: sweep-kernel device time,
pair distances evaluated per candidate, and which kernel the per-class rule picks on its own.

    python scripts/early_break_bench.py [OUT.json]

Each case is uploaded once per MMRS_EARLY_BREAK setting (0 = K1, 1 = K1e wherever it fits, unset = the rule) and run
REPS times; the median of the sweep-kernel event times is reported. Needs a CUDA device."""
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

REPS = 5


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except OSError:
        q = None
    return q


def contour(rng, n, rot=0.0):
    phi = np.linspace(0, 2 * np.pi, n, endpoint=False)
    r0, e = rng.uniform(1.5, 3.0), rng.uniform(0.05, 0.35)
    r = r0 * (1 + e * np.cos(2 * phi) + 0.03 * np.cos(3 * phi + 0.4) + 0.02 * np.cos(5 * phi + 1.1))
    return np.stack([r * np.cos(phi + rot), r * np.sin(phi + rot)], 1) + rng.normal(0, 0.005, (n, 2))


def pack(tests, refs):
    toff = np.concatenate([[0], np.cumsum([len(t) for t in tests])])
    roff = np.concatenate([[0], np.cumsum([len(r) for r in refs])])
    return np.concatenate(tests), toff, np.concatenate(refs), roff, np.zeros((len(tests), 2))


def run_case(ctx, name, batch, grid, n, m):
    out = {"case": name, "units": len(batch[1]) - 1, "candidates_per_unit": int(grid.n_cand), "points": [n, m]}
    res = {}
    for flag in ("0", "1", None):
        if flag is None:
            os.environ.pop("MMRS_EARLY_BREAK", None)
        else:
            os.environ["MMRS_EARLY_BREAK"] = flag
        ctx.sweep_upload(*batch, [grid], mode=0, prefilter=1, prune=-1)
        ms = []
        for _ in range(REPS):
            ctx.sweep_run()
            r = ctx.sweep_download()
            ms.append(ctx.timings()["sweep_ms"])
        info = ctx.prefilter_info()
        key = {"0": "k1", "1": "k1e", None: "rule"}[flag]
        res[key] = r
        cands = info["eb_candidates"]
        out[key] = {"sweep_ms": float(np.median(ms)), "sweep_ms_min": float(np.min(ms)), "sweep_ms_max": float(np.max(ms)),
                    "k1e_candidates": cands,
                    "pairs_per_candidate": (info["eb_pairs"] / cands) if cands else float(n * m),
                    "pair_fraction_of_nm": (info["eb_pairs"] / cands / (n * m)) if cands else 1.0}
    os.environ.pop("MMRS_EARLY_BREAK", None)
    out["rule_picks"] = "K1e" if out["rule"]["k1e_candidates"] else "K1"
    out["k1e_speedup"] = out["k1"]["sweep_ms"] / out["k1e"]["sweep_ms"]
    out["identical_results"] = all(np.array_equal(res["k1"][f], res[k][f]) for k in ("k1e", "rule")
                                   for f in res["k1"].dtype.names)
    print(json.dumps(out), flush=True)
    return out


def main():
    out_path = Path(sys.argv[1]) if len(sys.argv) > 1 else None
    ctx = nat.Context(0)
    txy, toff, rxy, roff, cen, U, n = bench.make_units(n_pairs=1)   # pair 0: 398 frame pairs, N = M = 520
    bench_batch = (txy, toff, rxy, roff, cen)
    rng = np.random.default_rng(2026)
    rand = [contour(rng, 520, rng.normal(0, 0.3)) for _ in range(2 * 398)]
    phi = np.linspace(0, 2 * np.pi, 520, endpoint=False)
    circ = np.stack([2.0 * np.cos(phi), 2.0 * np.sin(phi)], 1)
    cfg4 = bench.synthetic_pullback(9, 2000, bench.SEED + 40)
    cfg4 = [np.concatenate([f, f[:20]]) - f.mean(0) for f in cfg4]   # N = M = 2 020
    cases = [
        ("bench units, 0.01 deg over +-180", bench_batch, nat.make_grid(0.01, 180.0), 520, 520),
        ("398 random contour pairs, 0.01 deg over +-180", pack(rand[::2], rand[1::2]), nat.make_grid(0.01, 180.0), 520, 520),
        ("circle on circle x 64, 0.01 deg over +-180", pack([circ] * 64, [circ] * 64), nat.make_grid(0.01, 180.0), 520, 520),
        ("bench units, 0.1 deg over +-180", bench_batch, nat.make_grid(0.1, 180.0), 520, 520),
        ("bench units, 0.5 deg over +-90", bench_batch, nat.make_grid(0.5, 90.0), 520, 520),
        ("bench units, 1 deg over +-180", bench_batch, nat.make_grid(1.0, 180.0), 520, 520),
        ("bench units, 40 candidates (between-pullback shape)", bench_batch, nat.make_grid(0.5, 10.0), 520, 520),
        ("config-4 size, 8 frame pairs, 0.05 deg over +-180", pack(cfg4[1:], cfg4[:-1]), nat.make_grid(0.05, 180.0), 2020, 2020),
    ]
    rows = [run_case(ctx, *c) for c in cases]
    doc = {"gpu": gpu_info(), "reps": REPS, "timing": "sweep-kernel device time (CUDA events), median of the reps",
           "rows": rows}
    if out_path:
        out_path.parent.mkdir(parents=True, exist_ok=True)
        out_path.write_text(json.dumps(doc, indent=1) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
