"""The mean cost of the f64 oracle (tests/cost_oracle.py) and the argument checks of find_best_rigid_transform's
cost, on the CPU."""
import numpy as np
import pytest
from scipy.spatial.distance import cdist

import multimodars as mm
from tests import cost_oracle as co


def mean(test, ref, centre, mode, angle, t=(0.0, 0.0)):
    return co.candidate_cost(test, ref, centre, mode, angle, t, "mean")


def _brute(test, ref, centre, mode, angle, t):
    """cdist: per direction the mean of the row minima of the distance matrix, then the larger direction."""
    moved = co.transformed(test, centre, mode, angle, t)
    d = cdist(np.asarray(ref, dtype=np.float64), moved)
    return max(d.min(axis=1).mean(), d.min(axis=0).mean())


def test_oracle_against_cdist():
    rng = np.random.default_rng(31)
    test, ref = rng.normal(0, 1, (57, 2)), rng.normal(0, 1.2, (43, 2))
    for mode in (0, 1):
        for angle, t in [(0.0, (0.0, 0.0)), (0.3, (0.1, -0.2)), (-1.1, (0.0, 0.05))]:
            want = _brute(test, ref, (0.1, -0.1), mode, angle, t)
            got = mean(test, ref, (0.1, -0.1), mode, angle, t)
            assert got == pytest.approx(want, rel=1e-12, abs=1e-15)


def test_summation_order_is_pinned():
    test, ref = co.crafted_order_case()
    v = co.row_values(co.transformed(test, (0, 0), 0, 0.0), ref)
    assert v[0] == 1.0 and (v[1:] == 2.0 ** -53).all()
    assert float(np.cumsum(v)[-1]) == 1.0 and float(np.sum(v)) != 1.0     # the two orders differ here
    (fwd,), (bwd,) = co.directions(test, ref, (0, 0), 0, 0.0, [(0.0, 0.0)], "mean")
    assert bwd == 1.0 / len(v) and fwd == 2.0 ** -53
    assert mean(test, ref, (0, 0), 0, 0.0) == 1.0 / len(v)


def test_empty_and_one_point_sets():
    a = np.array([[1.0, 2.0], [3.0, -1.0]])
    assert mean(a, np.zeros((0, 2)), (0, 0), 0, 0.3) == 0.0
    assert mean(np.zeros((0, 2)), a, (0, 0), 1, 0.3) == 0.0
    assert mean(np.full((3, 2), np.nan), a, (0, 0), 1, 0.3) == 0.0     # only non-finite points: empty
    p, q = np.array([[3.0, 0.0]]), np.array([[0.0, 4.0]])
    assert mean(p, q, (0, 0), 0, 0.0) == 5.0
    # one point against two: fwd averages two distances, bwd is the one nearest distance
    two = np.array([[0.0, 4.0], [3.0, 1.0]])
    (fwd,), (bwd,) = co.directions(p, two, (0, 0), 0, 0.0, [(0.0, 0.0)], "mean")
    assert bwd == 1.0 and fwd == (5.0 + 1.0) / 2
    # non-finite points are dropped
    noisy = np.concatenate([a, [[np.nan, 1.0], [np.inf, 0.0]]])
    assert mean(noisy, two, (0.5, 0.5), 1, 0.7, (0.1, 0.0)) == mean(a, two, (0.5, 0.5), 1, 0.7, (0.1, 0.0))


@pytest.mark.parametrize("bad", ["max", "Mean", "", None, 1])
def test_find_best_rigid_transform_rejects_unknown_costs(bad):
    a = np.zeros((10, 2))
    with pytest.raises(ValueError, match="cost"):
        mm.find_best_rigid_transform(a, a, cost=bad)


@pytest.mark.parametrize("f", [0.9, 0.5])
def test_find_best_rigid_transform_rejects_a_trimmed_mean(f):
    a = np.zeros((10, 2))
    with pytest.raises(ValueError, match="inlier_fraction"):
        mm.find_best_rigid_transform(a, a, cost="mean", inlier_fraction=f)
