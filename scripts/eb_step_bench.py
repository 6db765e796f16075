#!/usr/bin/env python
"""Early-break sweep kernel time of several builds of the library, alternated in rounds on one GPU.

    python scripts/eb_step_bench.py OUT.json NAME=LIB.so [NAME=LIB.so ...] [--rounds R]

Each round runs every library once, in the order given, each in a fresh process (MMRS_B200_LIB). A run times, with
early break on (MMRS_EARLY_BREAK=1) and the sweep-kernel CUDA events (median of REPS runs per case):
  * every case of scripts/early_break_bench.py (K1e);
  * rigid_bench.py (a): the 398 bench units x 361 angles x 11^2 translations (K1e, RIGID);
  * partial_bench.py (a) and (b) at f in {1, 0.99, 0.95, 0.9} (K1e-partial; K1e at f = 1);
and records the pair distances evaluated per candidate (eb_pairs) and a digest of every result. The card's name, power
limit and max SM clock are read in the same call. Needs a CUDA device."""
from __future__ import annotations

import hashlib
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
REPS = 5


def one():
    sys.path[:0] = [str(ROOT), str(ROOT / "multimoda-rs_b200"), str(ROOT / "scripts")]
    import bench
    import early_break_bench as ebb
    from multimodars import _native as nat

    os.environ["MMRS_EARLY_BREAK"] = "1"
    ctx = nat.Context(0)
    rows = []

    def timed(name, upload, n_cand):
        upload()
        ms = []
        for _ in range(REPS):
            ctx.sweep_run()
            ms.append(ctx.timings()["sweep_ms"])
        r = ctx.sweep_download()
        info = ctx.prefilter_info()
        digest = hashlib.sha256(b"".join(np.ascontiguousarray(r[f]).tobytes() for f in r.dtype.names)).hexdigest()[:16]
        rows.append({"case": name, "sweep_ms": float(np.median(ms)), "sweep_ms_min": float(np.min(ms)),
                     "sweep_ms_max": float(np.max(ms)), "k1e_candidates": info["eb_candidates"],
                     "eb_pairs": info["eb_pairs"], "candidates": n_cand, "result_sha256_16": digest})

    txy, toff, rxy, roff, cen, U, n = bench.make_units(n_pairs=1)
    for name, batch, g, _, _ in ebb.make_cases():
        timed(name, lambda: ctx.sweep_upload(*batch, [g], mode=0, prefilter=1, prune=-1), (len(batch[1]) - 1) * g.n_cand)
    g1, tg = nat.make_grid(1.0, 180.0), nat.make_tgrid(0.05, 5)
    timed("rigid (a): bench units x 361 angles x 121 translations",
          lambda: ctx.rigid_upload(txy, toff, rxy, roff, cen, [g1], [tg], mode=0), U * g1.n_cand * 121)
    g = nat.make_grid(bench.STEP_DEG, bench.RANGE_DEG)
    for f in (1.0, 0.99, 0.95, 0.9):
        timed(f"partial (a) f={f}: bench units, 0.01 deg",
              lambda: ctx.partial_upload(txy, toff, rxy, roff, cen, [g], mode=0, inlier_fraction=f, prefilter=1, prune=-1),
              U * g.n_cand)
    for f in (1.0, 0.99, 0.95, 0.9):
        timed(f"partial (b) f={f}: bench units x 361 angles x 121 translations",
              lambda: ctx.partial_upload(txy, toff, rxy, roff, cen, [g1], [tg], mode=0, inlier_fraction=f),
              U * g1.n_cand * 121)
    ctx.close()
    print(json.dumps(rows))


def main():
    args = sys.argv[1:]
    rounds = 3
    if "--rounds" in args:
        k = args.index("--rounds")
        rounds = int(args[k + 1])
        del args[k:k + 2]
    out_path, libs = Path(args[0]), [a.split("=", 1) for a in args[1:]]
    q = ["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"]
    doc = {"gpu": subprocess.run(q, capture_output=True, text=True, timeout=30).stdout.strip(), "reps": REPS,
           "timing": "sweep-kernel CUDA events, median of the reps; libraries alternated per round",
           "runs": {name: [] for name, _ in libs}}
    for r in range(rounds):
        for name, lib in libs:
            env = dict(os.environ, MMRS_B200_LIB=str(Path(lib).resolve()))
            p = subprocess.run([sys.executable, __file__, "--one"], env=env, capture_output=True, text=True, check=True)
            rows = json.loads(p.stdout.strip().splitlines()[-1])
            doc["runs"][name].append(rows)
            print(f"round {r} {name}: " + ", ".join(f"{x['sweep_ms']:.2f}" for x in rows), flush=True)
    names = [n for n, _ in libs]
    doc["summary"] = []
    for i, row in enumerate(doc["runs"][names[0]][0]):
        s = {"case": row["case"]}
        for name in names:
            ms = [run[i]["sweep_ms"] for run in doc["runs"][name]]
            last = doc["runs"][name][-1][i]
            s[name] = {"sweep_ms_median": float(np.median(ms)), "sweep_ms_runs": ms,
                       "pairs_per_candidate": last["eb_pairs"] / last["k1e_candidates"] if last["k1e_candidates"] else None,
                       "eb_pairs": last["eb_pairs"], "result_sha256_16": last["result_sha256_16"]}
        doc["summary"].append(s)
        print(json.dumps(s), flush=True)
    doc["gpu_after"] = subprocess.run(q, capture_output=True, text=True, timeout=30).stdout.strip()
    out_path.parent.mkdir(parents=True, exist_ok=True)
    out_path.write_text(json.dumps(doc, indent=1) + "\n")


if __name__ == "__main__":
    if sys.argv[1:2] == ["--one"]:
        one()
    else:
        main()
