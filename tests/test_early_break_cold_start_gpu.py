"""The first candidate of each K1e warp run (k_sweep_eb) takes its hints from a subsample of the other set.

A run starts anywhere in the angle range, where a point's index-diagonal neighbour is rarely near it; the subsample's
nearest point is. Pair counts on the bench units show the saving. The hints only order the scans, so K1e must still give
every candidate's FP32 distance bit for bit as K1 does (and K1e-partial as its early-break-off form), including at set
sizes around the subsample stride, N != M, non-finite points and rigid runs, on grids whose runs start far from angle 0."""
import numpy as np
import pytest

import bench
from multimodars import _native as nat
from tests.test_early_break_gpu import assert_identical, both, ctx  # noqa: F401  (ctx: the module fixture)
from tests.test_partial_gpu import on_vs_off
from tests.test_rigid_gpu import k1_vs_k1e
from tests.test_sweep_gpu import make_units

pytestmark = pytest.mark.gpu


def far_grids():
    """A full-range grid, and a fine grid centred at 137 deg: every run of the second starts far from angle 0."""
    return [nat.make_grid(0.5, 180.0), nat.make_grid(0.05, 10.0, center=2.4, limes_deg=180.0)]


def far(ctx, monkeypatch, tests, refs, cents):  # noqa: F811
    gou = np.arange(len(tests)) % 2
    return assert_identical(both(ctx, monkeypatch, tests, refs, cents, far_grids(), grid_of_unit=gou))


def pairs_per_candidate(ctx, monkeypatch, step_deg):  # noqa: F811
    txy, toff, rxy, roff, cen, U, n = bench.make_units(n_pairs=1)
    g = nat.make_grid(step_deg, 180.0)
    monkeypatch.setenv("MMRS_EARLY_BREAK", "1")
    ctx.sweep_batched(txy, toff, rxy, roff, cen, [g], mode=0, prefilter=1, prune=-1)
    monkeypatch.delenv("MMRS_EARLY_BREAK")
    info = ctx.prefilter_info()
    assert info["eb_candidates"] == U * g.n_cand
    return info["eb_pairs"] / info["eb_candidates"]


@pytest.mark.parametrize("step_deg,limit", [(0.01, 2000), (1.0, 8000)])
def test_bench_units_pairs_per_candidate(ctx, monkeypatch, step_deg, limit):  # noqa: F811
    """The 398 bench units over +-180 deg: 2 494 (0.01 deg) and 15 113 (1 deg) pairs per candidate with index-diagonal
    first hints."""
    per_cand = pairs_per_candidate(ctx, monkeypatch, step_deg)
    print(f"{step_deg} deg: {per_cand:.0f} pairs per candidate")
    assert per_cand < limit, per_cand


def test_unequal_sets(ctx, monkeypatch):  # noqa: F811
    rng = np.random.default_rng(301)
    tests, refs, cents, *_ = make_units(rng, [(520, 300), (300, 520), (97, 411), (411, 97)])
    far(ctx, monkeypatch, tests, refs, cents)


@pytest.mark.parametrize("k", [1, 2, 3, 15, 16, 17, 33])
def test_sets_around_the_stride(ctx, monkeypatch, k):  # noqa: F811
    rng = np.random.default_rng(310 + k)
    tests, refs, cents, *_ = make_units(rng, [(k, 520), (520, k), (k, k), (k, 17), (33, k)])
    far(ctx, monkeypatch, tests, refs, cents)


def test_non_finite_points(ctx, monkeypatch):  # noqa: F811
    """NaN and inf at indices that are multiples of the stride and elsewhere; the sets that remain are of 2 to 520
    points."""
    rng = np.random.default_rng(320)
    tests, refs, cents, *_ = make_units(rng, [(520, 520), (200, 180), (17, 16), (40, 3)])
    tests[0][[0, 16, 203]] = np.nan
    refs[0][[0, 32]] = np.inf
    refs[1][[0, 5]] = -np.inf
    refs[2][::2] = np.nan
    tests[3][0] = np.inf
    refs[3][0] = np.nan
    far(ctx, monkeypatch, tests, refs, cents)


def test_rigid_batch(ctx, monkeypatch):  # noqa: F811
    rng = np.random.default_rng(330)
    tests, refs, cents, *_ = make_units(rng, [(520, 520), (300, 411), (16, 33), (3, 17)])
    k1_vs_k1e(ctx, monkeypatch, tests, refs, cents, far_grids()[1:], [nat.make_tgrid(0.05, 2, t0=(0.02, -0.03))])


def test_partial_on_off(ctx, monkeypatch):  # noqa: F811
    rng = np.random.default_rng(340)
    tests, refs, cents, *_ = make_units(rng, [(520, 520), (300, 411), (411, 300), (33, 17), (17, 520)])
    tests[1][[0, 16]] = np.nan
    for g in far_grids():
        on_vs_off(ctx, monkeypatch, tests, refs, cents, [g], 0.95)
