"""The reference's own ingest known-answer tests, held against the PRODUCT's host ingest (mmrs_geometry_from_dir in
libmmrs_b200.so, no GPU involved): io/build.rs:244-400, processing/preprocessing.rs:242-262. The input directories are
written from the committed pullbacks of tests/golden/inputs.npz (the reference's ivus_rest and ivus_stress examples);
the layered directory of build.rs:244-337 is ivus_rest with an EEM contour added to every frame."""
import numpy as np
import pytest

import multimodars as mm
from multimodars import _native as nat
from tests import golden_io as gio


@pytest.fixture(scope="module")
def fix(tmp_path_factory):
    root = tmp_path_factory.mktemp("fixtures")
    pack = gio.inputs()
    gio.write_dir(pack, "rest", root / "ivus_rest")
    gio.write_dir(pack, "stress", root / "ivus_stress")
    full = {k: pack[k] for k in pack.files if k.startswith("rest__")}
    for ph in ("diastolic", "systolic"):
        lum = full[f"rest__{ph}_lumen"]
        eem = lum.copy()
        for f in np.unique(lum[:, 0]):
            m = lum[:, 0] == f
            c = lum[m, 1:3].mean(axis=0)
            eem[m, 1:3] = c + 1.3 * (lum[m, 1:3] - c)       # the vessel wall outside the lumen, same frame and z
        full[f"rest__{ph}_eem"] = eem
    gio.write_dir(full, "rest", root / "ivus_full")
    return root


def build(fix, name, label, diastole=True, n_cath=20):
    return mm.PyGeometry.from_blob(nat.geometry_from_dir(fix / name, label, diastole, (4.5, 4.5), 0.5, n_cath), label)


def test_rest_directory_first_frame(fix):  # build.rs:339-370
    g = build(fix, "ivus_rest", "full")
    lum = g.frames[0].lumen
    (_, _), long_axis = lum.find_farthest_points()
    (_, _), short_axis = lum.find_closest_opposite()
    assert lum.original_frame == 385
    assert lum.get_area() == pytest.approx(5.42, abs=0.1)
    assert long_axis == pytest.approx(5.2, abs=0.1) and short_axis == pytest.approx(1.15, abs=0.1)
    assert lum.get_elliptic_ratio() == pytest.approx(4.52, abs=0.1)
    assert lum.aortic_thickness == 0.96 and lum.pulmonary_thickness == 1.68
    assert g.frames[0].reference_point.frame_index == lum.original_frame


def test_catheter_contours(fix):  # build.rs:372-400
    g = build(fix, "ivus_rest", "test")
    assert g.label == "test" and len(g.frames) > 0
    for f in g.frames:
        cath = f.extras["Catheter"] if "Catheter" in f.extras else f.extras[mm.PyContourType.Catheter]
        assert len(cath) == 20
        assert cath.centroid[2] == pytest.approx(f.lumen.centroid[2], abs=1e-6)
    assert all(len((f.extras.get("Catheter") or f.extras.get(mm.PyContourType.Catheter))) == 7
               for f in build(fix, "ivus_rest", "t", n_cath=7).frames)


def test_full_directory_layers_agree_on_ids(fix):  # build.rs:244-337
    g = build(fix, "ivus_full", "full")
    assert len(g.frames) > 0
    for f in g.frames:
        kinds = {str(k): c for k, c in f.extras.items()}
        assert "Eem" in kinds and "Catheter" in kinds
        for c in kinds.values():
            assert (c.id, c.original_frame) == (f.lumen.id, f.lumen.original_frame)
    assert [f.id for f in g.frames] == list(range(len(g.frames)))            # integrity_check.rs: consecutive ids


def test_stress_directory_first_frame(fix):  # preprocessing.rs:242-262
    g = build(fix, "ivus_stress", "stress")
    assert g.frames[0].lumen.original_frame == 314 and g.frames[0].reference_point is not None
    sys_ = build(fix, "ivus_stress", "stress", diastole=False)               # :264-283 reads both phases of one directory
    assert len(sys_.frames) > 0 and sys_.frames[0].reference_point is not None
