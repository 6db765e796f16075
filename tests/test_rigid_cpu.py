"""CPU checks of rigid candidates: the f64 restatement against scipy, the translation-grid formula, the ctypes mirrors
of the header structs, and argument validation of find_best_rigid_transform (which raises before any device call)."""
import ctypes as C
import math
import re
from pathlib import Path

import numpy as np
import pytest
from scipy.spatial.distance import directed_hausdorff

import multimodars as mm
from multimodars import _native as nat
from tests import rigid_oracle as ro

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.parametrize("mode", [0, 1])
def test_rigid_search_against_scipy(mode):
    rng = np.random.default_rng(3 + mode)
    test, ref = rng.normal(0, 1, (23, 2)), rng.normal(0.1, 1.1, (19, 2))
    centre = (0.2, -0.1)
    angles = [0.0, 0.3, -1.2]
    offs = ro.tgrid_offsets(0.05, -0.02, 0.1, 2)
    idx, costs = ro.rigid_search(test, ref, centre, mode, angles, offs)
    want = np.empty_like(costs)
    for i, a in enumerate(angles):
        for j, (tx, ty) in enumerate(offs):
            if mode == 0 and a == 0.0:
                m = test + (tx, ty)
            else:
                c, s = math.cos(a), math.sin(a)
                x, y = test[:, 0] - centre[0], test[:, 1] - centre[1]
                m = np.stack([x * c - y * s + centre[0] + tx, x * s + y * c + centre[1] + ty], 1)
            want[i, j] = max(directed_hausdorff(m, ref)[0], directed_hausdorff(ref, m)[0])
    assert np.allclose(costs, want, rtol=1e-13, atol=1e-13)
    assert idx == int(np.argmin(want.reshape(-1)))


def test_rigid_search_empty_and_non_finite():
    offs = ro.tgrid_offsets(0.0, 0.0, 0.1, 1)
    idx, costs = ro.rigid_search(np.zeros((0, 2)), np.ones((3, 2)), (0, 0), 1, [0.1, 0.2], offs)
    assert idx == 0 and (costs == 0.0).all()
    rng = np.random.default_rng(9)
    a, b = rng.normal(size=(10, 2)), rng.normal(size=(8, 2))
    a_nan = np.concatenate([a, [[np.nan, 1.0], [np.inf, 0.0]]])
    assert np.array_equal(ro.rigid_search(a_nan, b, (0, 0), 1, [0.4], offs)[1], ro.rigid_search(a, b, (0, 0), 1, [0.4], offs)[1])


def test_translation_grid_formula():
    tg = nat.make_tgrid(0.07, 3, t0=(0.3, -0.2))
    offs = ro.offsets_of(tg)
    assert offs.shape == (49, 2)
    for j in (0, 5, 7, 24, 48):
        jy, jx = divmod(j, 7)
        assert offs[j, 0] == 0.3 + float(jx - 3) * 0.07 and offs[j, 1] == -0.2 + float(jy - 3) * 0.07
    assert np.array_equal(ro.offsets_of(nat.make_tgrid(0.5, 0)), [[0.0, 0.0]])   # half_n = 0: c == i


def test_struct_mirrors_match_header():
    hdr = (ROOT / "include" / "mmrs_b200.h").read_text()
    assert C.sizeof(nat.TGrid) == 32
    assert C.sizeof(nat.RigidResult) == 40 + 8 + 8 + 16
    assert nat.RIGID_RESULT_DTYPE.itemsize == C.sizeof(nat.RigidResult)
    for f, _ in nat.RigidResult._fields_:
        assert nat.RIGID_RESULT_DTYPE.fields.get(f) or f == "r"
        assert re.search(rf"\b{f}\b", hdr), f
    for f, _ in nat.TGrid._fields_:
        assert re.search(rf"\b{f}\b", hdr), f
    body = hdr[hdr.index("typedef struct mmrs_rigid_result"):hdr.index("} mmrs_rigid_result;")]
    assert [m for m in re.findall(r"\b(r|angle_idx|trans_idx|pad|best_tx|best_ty)\b", re.sub(r"/\*.*?\*/", "", body, flags=re.S))] == \
        ["r", "angle_idx", "trans_idx", "pad", "best_tx", "best_ty"]
    off = {f: getattr(nat.RigidResult, f).offset for f, _ in nat.RigidResult._fields_}
    assert off == {"r": 0, "angle_idx": 40, "trans_idx": 48, "pad": 52, "best_tx": 56, "best_ty": 64}


def test_public_function_is_exported():
    assert "find_best_rigid_transform" in mm.__all__


@pytest.mark.parametrize("kw,exc,msg", [
    (dict(step_rotation_deg=0.0), ValueError, "step_rotation_deg"),
    (dict(step_rotation_deg=float("nan")), ValueError, "step_rotation_deg"),
    (dict(range_rotation_deg=-1.0), ValueError, "range_rotation_deg"),
    (dict(step_translation=0.0), ValueError, "step_translation"),
    (dict(step_translation=-0.1), ValueError, "step_translation"),
    (dict(range_translation=-0.1), ValueError, "range_translation"),
    (dict(range_translation=float("inf")), ValueError, "range_translation"),
    (dict(step_translation=1e-6, range_translation=1.0), ValueError, "at most 1000"),
    (dict(centre=(np.nan, 0.0)), ValueError, "centre"),
    (dict(centre=[(0.0, 0.0)] * 3), ValueError, "centre"),
    (dict(step_rotation_deg="x"), TypeError, "step_rotation_deg"),
])
def test_find_best_rigid_transform_validates_before_any_device_call(monkeypatch, kw, exc, msg):
    import multimodars._processing as proc

    monkeypatch.setattr(proc, "get_context", lambda *a, **k: pytest.fail("device reached"))
    rng = np.random.default_rng(0)
    a, b = rng.normal(size=(20, 3)), rng.normal(size=(25, 2))
    with pytest.raises(exc, match=msg):
        mm.find_best_rigid_transform(a, b, **kw)


@pytest.mark.parametrize("test,ref,msg", [
    ([np.zeros((5, 2))] * 2, [np.zeros((5, 2))], "2 and 1 point sets"),
    (np.zeros((5, 1)), np.zeros((5, 2)), "shape"),
    ([], [], "no point sets"),
    ("abc", np.zeros((5, 2)), "array"),
])
def test_find_best_rigid_transform_rejects_bad_sets(monkeypatch, test, ref, msg):
    import multimodars._processing as proc

    monkeypatch.setattr(proc, "get_context", lambda *a, **k: pytest.fail("device reached"))
    with pytest.raises((ValueError, TypeError), match=msg):
        mm.find_best_rigid_transform(test, ref)
