"""The early-break dense sweep (K1e, k_sweep_eb) against the full dense sweep (K1, k_sweep).

Every case runs twice on one context, MMRS_EARLY_BREAK=0 (K1 everywhere) and =1 (K1e wherever it fits). K1e must give
the same FP32 distance for every candidate, bit for bit, and therefore the same result in every field."""
import numpy as np
import pytest

import bench
from multimodars import _native as nat
from tests.test_sweep_gpu import check_against_oracle, contour, make_units

pytestmark = pytest.mark.gpu

FIELDS = ("best_idx", "best_angle", "best_dist", "best_dist_f32", "n_shortlist", "n_ties", "flags")


@pytest.fixture(scope="module")
def ctx():
    c = nat.Context(0)
    yield c
    c.close()


def both(ctx, monkeypatch, tests, refs, cents, grids, grid_of_unit=None, mode=0):
    """Results, dist32 rows and the K1e counters of the two runs."""
    txy, rxy = np.concatenate(tests), np.concatenate(refs)
    toff = np.concatenate([[0], np.cumsum([len(t) for t in tests])])
    roff = np.concatenate([[0], np.cumsum([len(r) for r in refs])])
    gou = np.zeros(len(tests), dtype=np.int32) if grid_of_unit is None else np.asarray(grid_of_unit, dtype=np.int32)
    out = []
    for flag in ("0", "1"):
        monkeypatch.setenv("MMRS_EARLY_BREAK", flag)
        res = ctx.sweep_batched(txy, toff, rxy, roff, cents, grids, grid_of_unit=gou, mode=mode, keep_dist32=True)
        d32 = [ctx.dist32(u, int(grids[gou[u]].n_cand)) if len(tests[u]) and len(refs[u]) else None
               for u in range(len(tests))]
        out.append((res, d32, ctx.prefilter_info()))
    monkeypatch.delenv("MMRS_EARLY_BREAK")
    return out


def assert_identical(runs):
    (r0, d0, i0), (r1, d1, i1) = runs
    assert i0["eb_candidates"] == 0, "MMRS_EARLY_BREAK=0 must run K1"
    assert i1["eb_candidates"] > 0, "MMRS_EARLY_BREAK=1 must run K1e"
    for u, (a, b) in enumerate(zip(d0, d1)):
        if a is not None:
            bad = np.flatnonzero(a.view(np.uint32) != b.view(np.uint32))
            assert bad.size == 0, (u, bad[:8], a[bad[:8]], b[bad[:8]])
    for f in FIELDS:
        assert np.array_equal(r0[f], r1[f]), f
    return i1


def test_bench_units_bit_identical_and_few_pairs(ctx, monkeypatch):
    """64 units spread over the bench batch, full 36 000-candidate grid; K1e must evaluate < 5 % of N M pairs."""
    txy, toff, rxy, roff, cen, U, n = bench.make_units()
    pick = np.linspace(0, U - 1, 64).astype(int)
    tests = [txy[toff[u]:toff[u + 1]] for u in pick]
    refs = [rxy[roff[u]:roff[u + 1]] for u in pick]
    g = nat.make_grid(bench.STEP_DEG, bench.RANGE_DEG)
    info = assert_identical(both(ctx, monkeypatch, tests, refs, cen[pick], [g]))
    per_cand = info["eb_pairs"] / info["eb_candidates"]
    assert info["eb_candidates"] == 64 * g.n_cand
    assert per_cand < 0.05 * n * n, per_cand


def test_auto_rule_picks_k1e_for_the_bench_shape(ctx):
    txy, toff, rxy, roff, cen, U, n = bench.make_units(n_pairs=1)
    g = nat.make_grid(bench.STEP_DEG, bench.RANGE_DEG)
    ctx.sweep_batched(txy[:8 * n], toff[:9], rxy[:8 * n], roff[:9], cen[:8], [g], mode=0, prefilter=1, prune=-1)
    assert ctx.prefilter_info()["eb_candidates"] == 8 * g.n_cand


def test_random_clouds(ctx, monkeypatch):
    rng = np.random.default_rng(41)
    tests = [rng.normal(0, s, (k, 2)) for k, s in ((520, 1.0), (300, 2.0), (97, 0.3), (64, 5.0))]
    refs = [rng.normal(0, s, (k, 2)) for k, s in ((520, 1.0), (411, 1.5), (250, 0.3), (64, 5.0))]
    assert_identical(both(ctx, monkeypatch, tests, refs, np.zeros((4, 2)), [nat.make_grid(0.05, 180.0)]))


def test_circle_on_circle_every_candidate_ties(ctx, monkeypatch):
    phi = np.linspace(0, 2 * np.pi, 360, endpoint=False)
    circ = np.stack([2.0 * np.cos(phi), 2.0 * np.sin(phi)], 1)
    runs = both(ctx, monkeypatch, [circ, circ[::2]], [circ, circ], np.zeros((2, 2)), [nat.make_grid(0.1, 180.0)])
    assert_identical(runs)


def test_contour_against_itself(ctx, monkeypatch):
    rng = np.random.default_rng(5)
    c = contour(rng, 520)
    runs = both(ctx, monkeypatch, [c, c[:333]], [c.copy(), c.copy()], np.array([[4.5, 4.5], [4.5, 4.5]]),
                [nat.make_grid(0.01, 180.0)])
    assert_identical(runs)


def test_unequal_tiny_and_duplicated_sets(ctx, monkeypatch):
    rng = np.random.default_rng(8)
    sizes = [(520, 300), (300, 520), (33, 257), (6, 6), (1, 5), (5, 1), (31, 40), (544, 520)]
    tests, refs, cents, *_ = make_units(rng, sizes)
    tests[3] = np.repeat(tests[3][:2], 3, axis=0)          # duplicated points
    refs[3] = np.concatenate([refs[3][:3], refs[3][:3]])
    assert_identical(both(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(0.05, 180.0)]))


def test_non_finite_points(ctx, monkeypatch):
    rng = np.random.default_rng(13)
    tests, refs, cents, *_ = make_units(rng, [(520, 520), (200, 180)])
    tests[0][[3, 200]] = np.nan
    refs[0][17] = np.inf
    refs[1][[0, 5]] = -np.inf
    assert_identical(both(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(0.05, 180.0)]))


@pytest.mark.parametrize("mode", [0, 1])
def test_modes_and_oracle(ctx, monkeypatch, mode):
    """mode 1 = the between-pullback sweep; the K1e run is also pinned against the CPU oracle."""
    rng = np.random.default_rng(21 + mode)
    tests, refs, cents, *_ = make_units(rng, [(520, 520), (400, 450), (130, 64)])
    runs = both(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(0.1, 180.0)], mode=mode)
    assert_identical(runs)
    check_against_oracle(ctx, tests, refs, cents, runs[1][0], 0.1, 180.0, mode)


def test_coarse_grid_and_hierarchical_run(ctx, monkeypatch):
    rng = np.random.default_rng(6)
    tests, refs, cents, *_ = make_units(rng, [(520, 520)] * 6)
    coarse = both(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(1.0, 180.0)])
    assert_identical(coarse)
    centres = coarse[1][0]["best_angle"]
    grids = [nat.make_grid(0.01, 2.0, center=float(c), limes_deg=180.0) for c in centres]
    fine = both(ctx, monkeypatch, tests, refs, cents, grids, grid_of_unit=np.arange(6))
    assert_identical(fine)
    check_against_oracle(ctx, tests, refs, cents, fine[1][0], 0.01, 2.0, 0, center=centres, limes=180.0)
