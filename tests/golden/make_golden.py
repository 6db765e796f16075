"""Generates tests/golden/*.npz. Run with a checkout of the reference:

    python tests/golden/make_golden.py <reference checkout>

Inputs: the reference's example / fixture pullbacks, re-encoded as (N,4) [frame, x, y, z]
arrays (+ reference point, + records) so the tests run without the
reference. Outputs: what the CPU ORACLE (oracle/, a restatement pinned on
the reference's Rust KATs — the reference itself cannot be built here) returns for the
reference's own configurations. These are oracle-generated goldens, not reference-generated."""
import hashlib
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path[:0] = [str(ROOT)]
from oracle import oracle_py as ora  # noqa: E402

REF = Path(sys.argv[1])
OUT = Path(__file__).resolve().parent


def _load(p):
    first = open(p).readline()
    delim = "\t" if first.count("\t") > first.count(",") else ","   # io/input.rs:149-170
    return np.loadtxt(p, delimiter=delim, ndmin=2)


def load_dir(d):
    d = Path(d)
    out = {}
    for phase in ("diastolic", "systolic"):
        out[f"{phase}_lumen"] = _load(d / f"{phase}_contours.csv")[:, :4]
        out[f"{phase}_ref"] = _load(d / f"{phase}_reference_points.csv")[0, :4]
        for pre, key in (("eem", "eem"), ("calcium", "calc"), ("branch", "side")):
            p = d / f"{pre}_{phase}_contours.csv"
            if p.exists():
                out[f"{phase}_{key}"] = _load(p)[:, :4]
    rec = d / "combined_sorted_manual.csv"
    if rec.exists():
        import csv

        rows = []
        with open(rec) as f:
            for r in csv.DictReader(f):
                def num(s):
                    try:
                        return float(s)
                    except ValueError:
                        return np.nan
                rows.append([float(r["frame"]), 1.0 if r["phase"] == "D" else 0.0, num(r["measurement_1"]),
                             num(r["measurement_2"])])
        out["records"] = np.array(rows)
    return out


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.float64).tobytes()).hexdigest()


def main():
    pack = {}
    for name, d in (("rest", REF / "examples/data/ivus_rest"), ("stress", REF / "examples/data/ivus_stress"),
                    ("ideal", REF / "data/fixtures/idealized_geometry")):
        for k, v in load_dir(d).items():
            pack[f"{name}__{k}"] = v
    np.savez_compressed(OUT / "inputs.npz", **pack)

    gold = {}
    # config 1: from_file_full(ivus_rest, ivus_stress), defaults except write_obj/postprocessing
    blobs = [ora.build_geometry_from_dir(REF / "examples/data" / d, d, dia) for d in ("ivus_rest", "ivus_stress")
             for dia in (True, False)]
    for i, b in enumerate(blobs):
        gold[f"cfg1_in_sha_{i}"] = np.array(sha(b))
    for tag, kw in (("default", dict(step=0.5, rng=90.0, brute=False, smooth=True)),
                    ("brute0p5", dict(step=0.5, rng=90.0, brute=True, smooth=False)),
                    ("hier0p05", dict(step=0.05, rng=90.0, brute=False, smooth=False))):
        outs, logs = ora.process(4, blobs, kw["step"], kw["rng"], kw["smooth"], kw["brute"], 500, threads=8)
        for i, l in enumerate(logs):
            gold[f"cfg1_{tag}_logs_{i}"] = l
        for i, o in enumerate(outs):
            gold[f"cfg1_{tag}_out_sha_{i}"] = np.array(sha(o))
    # align_within.rs:855-887 / align_between.rs:305-373 on the idealized fixture
    ideal = ora.build_geometry_from_dir(REF / "data/fixtures/idealized_geometry", "stress", True)
    out, logs, an = ora.align_within(ideal, 0.01, 20.0, True, False, 200)
    gold["ideal_within_logs"] = logs
    gold["ideal_within_anomalous"] = np.array(an)
    gold["ideal_within_out_sha"] = np.array(sha(out))
    np.savez_compressed(OUT / "oracle_outputs.npz", **gold)
    print("wrote", OUT / "inputs.npz", OUT / "oracle_outputs.npz")
    for k in sorted(gold):
        if "logs" in k:
            print(k, gold[k].shape, gold[k][:2, 2])


if __name__ == "__main__":
    main()
