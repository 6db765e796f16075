"""The mean-cost oracle (tests/mean_oracle.py) and the argument checks of find_best_rigid_transform's cost, on the
CPU."""
import numpy as np
import pytest
from scipy.spatial.distance import cdist

import multimodars as mm
from tests import mean_oracle as mo
from tests import partial_oracle as po


def _brute(test, ref, centre, mode, angle, t):
    """cdist: per direction the mean of the row minima of the distance matrix, then the larger direction."""
    moved = po.transformed(test, centre, mode, angle, t)
    d = cdist(np.asarray(ref, dtype=np.float64), moved)
    return max(d.min(axis=1).mean(), d.min(axis=0).mean())


def test_oracle_against_cdist():
    rng = np.random.default_rng(31)
    test, ref = rng.normal(0, 1, (57, 2)), rng.normal(0, 1.2, (43, 2))
    for mode in (0, 1):
        for angle, t in [(0.0, (0.0, 0.0)), (0.3, (0.1, -0.2)), (-1.1, (0.0, 0.05))]:
            want = _brute(test, ref, (0.1, -0.1), mode, angle, t)
            got = mo.cost(test, ref, (0.1, -0.1), mode, angle, t)
            assert got == pytest.approx(want, rel=1e-12, abs=1e-15)


def test_summation_order_is_pinned():
    test, ref = mo.crafted_order_case()
    v = mo.row_values(po.transformed(test, (0, 0), 0, 0.0), ref)
    assert v[0] == 1.0 and (v[1:] == 2.0 ** -53).all()
    assert float(np.cumsum(v)[-1]) == 1.0 and float(np.sum(v)) != 1.0     # the two orders differ here
    fwd, bwd = mo.directions(test, ref, (0, 0), 0, 0.0)
    assert bwd == 1.0 / len(v) and fwd == 2.0 ** -53
    assert mo.cost(test, ref, (0, 0), 0, 0.0) == 1.0 / len(v)


def test_empty_and_one_point_sets():
    a = np.array([[1.0, 2.0], [3.0, -1.0]])
    assert mo.cost(a, np.zeros((0, 2)), (0, 0), 0, 0.3) == 0.0
    assert mo.cost(np.zeros((0, 2)), a, (0, 0), 1, 0.3) == 0.0
    assert mo.cost(np.full((3, 2), np.nan), a, (0, 0), 1, 0.3) == 0.0     # only non-finite points: empty
    p, q = np.array([[3.0, 0.0]]), np.array([[0.0, 4.0]])
    assert mo.cost(p, q, (0, 0), 0, 0.0) == 5.0
    # one point against two: fwd averages two distances, bwd is the one nearest distance
    two = np.array([[0.0, 4.0], [3.0, 1.0]])
    fwd, bwd = mo.directions(p, two, (0, 0), 0, 0.0)
    assert bwd == 1.0 and fwd == (5.0 + 1.0) / 2
    # non-finite points are dropped
    noisy = np.concatenate([a, [[np.nan, 1.0], [np.inf, 0.0]]])
    assert mo.cost(noisy, two, (0.5, 0.5), 1, 0.7, (0.1, 0.0)) == mo.cost(a, two, (0.5, 0.5), 1, 0.7, (0.1, 0.0))


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
