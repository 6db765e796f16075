"""K1e (k_sweep_eb) seeds each candidate through a uniform grid over the other set instead of scanning all of it.

K0 builds one grid per set and upload: the reference set in its own frame, the test set unrotated. A seed visits only
the cells within a margin of its hint's distance; the points it skips are provably farther than the minimum. So every
candidate's FP32 distance must stay bit for bit K1's (MMRS_EARLY_BREAK=0), on the bench units and on sets chosen to
stress the grid: points on cell boundaries, empty cells, degenerate extents (no grid), coordinates near FP32 overflow,
tiny sets, rigid queries outside the grid's box. The pair count on the bench units shows the saving."""
import numpy as np
import pytest

import bench
from multimodars import _native as nat
from tests.test_early_break_cold_start_gpu import pairs_per_candidate
from tests.test_early_break_gpu import assert_identical, both, ctx  # noqa: F401  (ctx: the module fixture)
from tests.test_rigid_gpu import k1_vs_k1e
from tests.test_sweep_gpu import contour, make_units, pack

pytestmark = pytest.mark.gpu


def grids():
    return [nat.make_grid(0.5, 180.0), nat.make_grid(0.05, 10.0, center=2.4, limes_deg=180.0)]


def check(ctx, monkeypatch, tests, refs, cents, gs=None):  # noqa: F811
    gs = grids() if gs is None else gs
    gou = np.arange(len(tests)) % len(gs)
    return assert_identical(both(ctx, monkeypatch, tests, refs, np.asarray(cents, dtype=float), gs, grid_of_unit=gou))


def pairs_at(ctx, monkeypatch, tests, refs, cents, scale):  # noqa: F811
    """Pairs per candidate of K1e (pinned to K1) on the units scaled by `scale` about the origin."""
    info = check(ctx, monkeypatch, [t * scale for t in tests], [r * scale for r in refs], np.asarray(cents) * scale)
    return info["eb_pairs"] / info["eb_candidates"]


def lattice_units(rng):
    """Lattice coordinates (multiples of 1/8 over an extent of 8, every cell edge of a 16 x 16 grid carries points)."""
    tests, refs = [], []
    for n, m in ((520, 520), (300, 411), (257, 130)):
        tests.append(np.round(contour(rng, n, r0=3.0, centre=(4.0, 4.0)) * 8) / 8)
        refs.append(np.round(contour(rng, m, r0=3.0, centre=(4.0, 4.0)) * 8) / 8)
    square = np.array([(x, y) for x in np.arange(0, 8.01, 0.5) for y in np.arange(0, 8.01, 0.5)])   # 17 x 17 lattice
    tests.append(square)
    refs.append(square[::-1].copy())
    return tests, refs, [(4.0, 4.0)] * 4


@pytest.mark.parametrize("case", ["contours", "lattice"])
def test_grids_cut_the_seed_pairs(ctx, monkeypatch, case):  # noqa: F811
    """Scaling every coordinate by a power of two changes no FP32 comparison, and beyond 2^60 a set takes no grid. So at
    2^60 K1e counts the pairs of full seed scans of the same geometry; at 1 and 2^57 the grids must visit fewer."""
    rng = np.random.default_rng(590)
    if case == "contours":
        tests, refs, cents, *_ = make_units(rng, [(520, 520), (300, 411), (411, 130)])
    else:
        tests, refs, cents = lattice_units(rng)
    full = pairs_at(ctx, monkeypatch, tests, refs, cents, 2.0 ** 60)
    for scale in (1.0, 2.0 ** 57):
        per_cand = pairs_at(ctx, monkeypatch, tests, refs, cents, scale)
        print(f"{case} x {scale:g}: {per_cand:.0f} pairs per candidate against {full:.0f} with full seed scans")
        assert per_cand < full, (scale, per_cand, full)


@pytest.mark.parametrize("sizes", [[(620, 620)], [(520, 900)], [(605, 605), (520, 520)]], ids=["620", "520x900", "mixed"])
def test_auto_rule_keeps_k1e_where_a_grid_does_not_fit(ctx, monkeypatch, sizes):  # noqa: F811
    """Units whose K1e shared memory is just under the 3-CTAs-per-SM rule without the grid block run K1e in auto mode
    (MMRS_EARLY_BREAK unset) as before, seeding by full scans, and still give K1's distances bit for bit, also beside a
    520-point unit that takes a grid."""
    rng = np.random.default_rng(600 + len(sizes))
    tests, refs, cents, *_ = make_units(rng, sizes)
    txy, toff, rxy, roff = pack(tests, refs)
    g = nat.make_grid(0.5, 180.0)
    runs = []
    for flag in (None, "0"):
        if flag is None:
            monkeypatch.delenv("MMRS_EARLY_BREAK", raising=False)
        else:
            monkeypatch.setenv("MMRS_EARLY_BREAK", flag)
        res = ctx.sweep_batched(txy, toff, rxy, roff, cents, [g], mode=0, prefilter=1, prune=-1, keep_dist32=True)
        runs.append((res, [ctx.dist32(u, int(g.n_cand)) for u in range(len(tests))], ctx.prefilter_info()))
    monkeypatch.delenv("MMRS_EARLY_BREAK")
    assert runs[0][2]["eb_candidates"] == len(sizes) * g.n_cand, runs[0][2]
    assert_identical(runs[::-1])


def test_bench_units_pairs_per_candidate(ctx, monkeypatch):  # noqa: F811
    """The 398 bench units over +-180 deg at 0.01 deg: 1 731 pairs per candidate with full seed scans, 1 352 through the
    grids (B200)."""
    per_cand = pairs_per_candidate(ctx, monkeypatch, 0.01)
    print(f"0.01 deg: {per_cand:.0f} pairs per candidate")
    assert per_cand < 1450, per_cand


@pytest.mark.parametrize("step_deg", [0.1, 1.0])
def test_bench_units_bit_identical(ctx, monkeypatch, step_deg):  # noqa: F811
    txy, toff, rxy, roff, cen, U, n = bench.make_units(n_pairs=1)
    tests = [txy[toff[u]:toff[u + 1]] for u in range(U)]
    refs = [rxy[roff[u]:roff[u + 1]] for u in range(U)]
    info = check(ctx, monkeypatch, tests, refs, cen, [nat.make_grid(step_deg, 180.0)])
    assert info["eb_candidates"] == U * nat.make_grid(step_deg, 180.0).n_cand


def test_points_on_cell_boundaries(ctx, monkeypatch):  # noqa: F811
    check(ctx, monkeypatch, *lattice_units(np.random.default_rng(500)))


def test_degenerate_sets(ctx, monkeypatch):  # noqa: F811
    """All points identical, collinear along an axis (zero extent: no grid) and along a diagonal (most cells empty)."""
    rng = np.random.default_rng(510)
    c = contour(rng, 300)
    same = np.full((200, 2), 4.7)
    t = np.linspace(-2, 2, 300)
    horiz = np.stack([t + 4.5, np.full_like(t, 4.5)], 1)
    diag = np.stack([t + 4.5, 0.5 * t + 4.5], 1)
    tests = [same, c, horiz, c, diag, diag]
    refs = [c, same, c, horiz, c, diag[::-1].copy()]
    check(ctx, monkeypatch, tests, refs, [(4.5, 4.5)] * 6)


def test_far_outlier(ctx, monkeypatch):  # noqa: F811
    """One point far from the rest: the grid's box is set by it and nearly every cell is empty."""
    rng = np.random.default_rng(520)
    tests, refs, cents, *_ = make_units(rng, [(520, 520), (300, 300), (520, 97)])
    refs[0][100] = (400.0, -300.0)
    tests[1][7] = (-250.0, 90.0)
    refs[2][0] = (1e4, 1e4)
    tests[2][519] = (-1e4, 3.0)
    check(ctx, monkeypatch, tests, refs, cents)


def test_non_finite_points(ctx, monkeypatch):  # noqa: F811
    """The host drops points with a NaN or infinite coordinate before staging, so K0 builds the grids over the finite rest
    (a coordinate that is finite in f64 but not in FP32 would turn its set's grid off instead)."""
    rng = np.random.default_rng(530)
    tests, refs, cents, *_ = make_units(rng, [(520, 520), (300, 200)])
    tests[0][[0, 64, 300]] = np.nan
    refs[0][5] = (np.inf, 1.0)
    refs[1][[1, 2]] = -np.inf
    check(ctx, monkeypatch, tests, refs, cents)


@pytest.mark.parametrize("scale", [1e16, 2e17, 5e18])
def test_coordinates_near_overflow(ctx, monkeypatch, scale):  # noqa: F811
    """Grids at 1e16 and 2e17 (d^2 stays finite); at 5e18 the coordinates pass 2^60, the units take no grid and some d^2 overflow FP32."""
    rng = np.random.default_rng(540)
    tests, refs, cents, *_ = make_units(rng, [(520, 520), (300, 257)])
    tests = [t * scale for t in tests]
    refs = [r * scale for r in refs]
    check(ctx, monkeypatch, tests, refs, np.asarray(cents) * scale)


def test_unequal_sets(ctx, monkeypatch):  # noqa: F811
    rng = np.random.default_rng(550)
    tests, refs, cents, *_ = make_units(rng, [(520, 130), (130, 520), (1100, 300), (255, 256), (1023, 1024)])
    check(ctx, monkeypatch, tests, refs, cents)


@pytest.mark.parametrize("k", [1, 2, 5, 31, 32, 33, 63, 64, 65, 70])
def test_small_sets(ctx, monkeypatch, k):  # noqa: F811
    """Around the smallest set that takes a grid (64 points)."""
    rng = np.random.default_rng(560 + k)
    tests, refs, cents, *_ = make_units(rng, [(k, 520), (520, k), (k, k), (k, 70), (64, k)])
    check(ctx, monkeypatch, tests, refs, cents)


def test_rigid_queries_outside_the_grid(ctx, monkeypatch):  # noqa: F811
    """Translations larger than the sets: column queries R(-theta)(b - t) and rotated rows fall outside the grids' boxes."""
    rng = np.random.default_rng(570)
    tests, refs, cents, *_ = make_units(rng, [(520, 520), (300, 411), (130, 64)])
    k1_vs_k1e(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(2.0, 180.0)], [nat.make_tgrid(3.0, 2, t0=(0.5, -1.0))])


def test_one_degree_grid(ctx, monkeypatch):  # noqa: F811
    rng = np.random.default_rng(580)
    tests, refs, cents, *_ = make_units(rng, [(520, 520)] * 4 + [(411, 300)])
    check(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(1.0, 180.0)])
