"""The partial cost of the f64 oracle (tests/cost_oracle.py) and the argument checks of find_best_rigid_transform's
inlier_fraction, on the CPU."""
import math

import numpy as np
import pytest
from scipy.spatial.distance import cdist

import multimodars as mm
from tests import cost_oracle as co


def _brute(test, ref, centre, mode, angle, t, f):
    """cdist + np.partition: the (q + 1)-th largest row minimum per direction, then the larger square root."""
    moved = co.transformed(test, centre, mode, angle, t)
    r = np.asarray(ref, dtype=np.float64)
    d2 = cdist(r, moved, "sqeuclidean")
    fwd_rows, bwd_rows = d2.min(axis=1), d2.min(axis=0)
    out = []
    for v in (fwd_rows, bwd_rows):
        k = max(1, math.ceil(f * len(v)))
        out.append(np.sqrt(np.partition(v, k - 1)[k - 1]))   # the K-th smallest = the (n - K + 1)-th largest
    return max(out)


@pytest.mark.parametrize("f", [1.0, 0.99, 0.95, 0.9, 0.5, 1e-9])
def test_oracle_against_cdist_partition(f):
    rng = np.random.default_rng(11)
    test, ref = rng.normal(0, 1, (57, 2)), rng.normal(0, 1.2, (43, 2))
    for mode in (0, 1):
        for angle, t in [(0.0, (0.0, 0.0)), (0.3, (0.1, -0.2)), (-1.1, (0.0, 0.05))]:
            want = _brute(test, ref, (0.1, -0.1), mode, angle, t, f)
            got = co.candidate_cost(test, ref, (0.1, -0.1), mode, angle, t, "partial", f)
            assert got == pytest.approx(want, rel=1e-12, abs=1e-15)


def test_full_fraction_is_the_rigid_oracle_bit_for_bit():
    rng = np.random.default_rng(12)
    test, ref = rng.normal(0, 1, (40, 2)), rng.normal(0, 1, (35, 2))
    test[5] = np.nan
    offs = co.tgrid_offsets(0.02, -0.01, 0.05, 2)
    for mode in (0, 1):
        for a in (0.0, 0.2, -2.5):
            want = co.costs_at_angle(test, ref, (0.3, 0.2), mode, a, offs, "full")
            got = np.array([co.candidate_cost(test, ref, (0.3, 0.2), mode, a, t, "partial", 1.0) for t in offs])
            assert np.array_equal(got, want)


def test_k_formula_boundaries():
    assert co.k_of(100, 0.95) == 95 and co.q_of(100, 0.95) == 5          # f n exactly an integer
    assert co.k_of(520, 0.95) == math.ceil(0.95 * 520) == 494
    assert co.k_of(1, 0.5) == 1 and co.q_of(1, 0.5) == 0                  # n = 1
    assert co.k_of(6, 1e-12) == 1 and co.q_of(6, 1e-12) == 5              # f tiny: one point counts
    assert co.k_of(10, 1.0) == 10 and co.q_of(10, 1.0) == 0
    assert co.k_of(0, 0.5) == 0 and co.q_of(0, 0.5) == 0
    assert co.k_of(3, 0.7) == math.ceil(0.7 * 3)                          # 0.7 * 3 = 2.0999999999999996 -> 3
    assert co.q_of(3, 0.7) == 0


def test_non_finite_points_do_not_count_in_k():
    rng = np.random.default_rng(13)
    test, ref = rng.normal(0, 1, (20, 2)), rng.normal(0, 1, (20, 2))
    noisy = np.concatenate([test, np.full((7, 2), np.nan)])
    for f in (0.9, 0.6):
        assert co.candidate_cost(noisy, ref, (0, 0), 1, 0.4, (0, 0), "partial", f) == \
            co.candidate_cost(test, ref, (0, 0), 1, 0.4, (0, 0), "partial", f)


@pytest.mark.parametrize("bad", [0.0, -0.5, 1.0000001, 2.0, float("nan"), float("inf")])
def test_find_best_rigid_transform_rejects_bad_fractions(bad):
    a = np.zeros((10, 2))
    with pytest.raises(ValueError, match="inlier_fraction"):
        mm.find_best_rigid_transform(a, a, inlier_fraction=bad)


@pytest.mark.parametrize("bad", ["0.9", None, [0.9], True])
def test_find_best_rigid_transform_rejects_non_numbers(bad):
    a = np.zeros((10, 2))
    with pytest.raises(TypeError, match="inlier_fraction"):
        mm.find_best_rigid_transform(a, a, inlier_fraction=bad)
