"""Helpers shared by the golden-fixture tests: load tests/golden/inputs.npz into the arguments the
oracle and the product take, and write a pullback back to the reference's CSV directory layout."""
import hashlib
from pathlib import Path

import numpy as np

GOLD = Path(__file__).resolve().parent / "golden"


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.float64).tobytes()).hexdigest()


def inputs():
    return np.load(GOLD / "inputs.npz")


def oracle_outputs():
    return np.load(GOLD / "oracle_outputs.npz")


def phase_arrays(pack, name, diastole):
    ph = "diastolic" if diastole else "systolic"
    g = lambda k: pack[f"{name}__{ph}_{k}"] if f"{name}__{ph}_{k}" in pack else None  # noqa: E731
    rec = pack[f"{name}__records"] if f"{name}__records" in pack else None
    return dict(lumen=g("lumen"), ref_point=g("ref"), eem=g("eem"), calc=g("calc"), side=g("side"), records=rec)


def write_dir(pack, name, dst):
    """Re-creates the reference's input directory (tab-separated, no header; io/input.rs:62-147)."""
    dst = Path(dst)
    dst.mkdir(parents=True, exist_ok=True)
    for dia in (True, False):
        ph = "diastolic" if dia else "systolic"
        a = phase_arrays(pack, name, dia)

        def dump(arr, fname):
            with open(dst / fname, "w") as f:
                for r in np.asarray(arr).reshape(-1, 4):
                    f.write(f"{int(r[0])}\t{float(r[1])!r}\t{float(r[2])!r}\t{float(r[3])!r}\n")

        dump(a["lumen"], f"{ph}_contours.csv")
        dump(a["ref_point"], f"{ph}_reference_points.csv")
        for key, pre in (("eem", "eem"), ("calc", "calcium"), ("side", "branch")):
            if a[key] is not None:
                dump(a[key], f"{pre}_{ph}_contours.csv")
    rec = phase_arrays(pack, name, True)["records"]
    if rec is not None:
        with open(dst / "combined_sorted_manual.csv", "w") as f:
            f.write("frame,position,phase,measurement_1,measurement_2\n")
            for r in rec:
                m1 = "" if np.isnan(r[2]) else repr(float(r[2]))
                m2 = "" if np.isnan(r[3]) else repr(float(r[3]))
                f.write(f"{int(r[0])},0,{'D' if r[1] else 'S'},{m1},{m2}\n")
    return dst


def py_input(mm, pack, name, diastole, label):
    a = phase_arrays(pack, name, diastole)
    rec = None
    if a["records"] is not None:
        rec = np.array([[int(r[0]), "D" if r[1] else "S", None if np.isnan(r[2]) else float(r[2]),
                         None if np.isnan(r[3]) else float(r[3])] for r in a["records"]], dtype=object)
    return mm.numpy_to_inputdata(a["lumen"], a["ref_point"], diastole, record=rec, eem_arr=a["eem"],
                                 calcification=a["calc"], sidebranch=a["side"], label=label)
