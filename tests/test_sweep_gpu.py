"""GPU parity of the batched sweep (through the C ABI) against the CPU oracle.

Bars (BASELINE.json north_star): selected candidate index / angle identical to
the reference semantics; f64 Hausdorff of the selection bit-identical to the
oracle; FP32 sweep distances within 1e-5 relative of the oracle's f64 values."""
import math

import numpy as np
import pytest

from multimodars import _native as nat
from oracle import oracle_py as ora

pytestmark = pytest.mark.gpu

REL_TOL_FP32 = 1e-5  # north_star: "Hausdorff values must match within 1e-5 relative in FP32"


@pytest.fixture(scope="module")
def ctx():
    c = nat.Context(0)
    yield c
    c.close()


def contour(rng, n, r0=2.5, e=0.2, rot=0.0, centre=(4.5, 4.5), noise=0.005):
    phi = np.linspace(0, 2 * np.pi, n, endpoint=False)
    r = r0 * (1 + e * np.cos(2 * phi) + 0.03 * np.cos(3 * phi + 0.4) + 0.02 * np.cos(5 * phi + 1.1))
    x = r * np.cos(phi + rot) + centre[0] + rng.normal(0, noise, n)
    y = r * np.sin(phi + rot) + centre[1] + rng.normal(0, noise, n)
    return np.stack([x, y], axis=1)


def make_units(rng, sizes, centre=(4.5, 4.5)):
    tests, refs, cents = [], [], []
    for (n, m) in sizes:
        rot = rng.normal(0, 0.2)
        refs.append(contour(rng, m, r0=rng.uniform(1.5, 3.0), e=rng.uniform(0.05, 0.35)))
        tests.append(contour(rng, n, r0=rng.uniform(1.5, 3.0), e=rng.uniform(0.05, 0.35), rot=rot))
        cents.append(np.array(centre) + rng.normal(0, 0.05, 2))
    return (tests, refs, np.array(cents), *pack(tests, refs))


def pack(tests, refs):
    """Per-unit point sets -> (test_xy, test_off, ref_xy, ref_off) of one batch."""
    toff = np.concatenate([[0], np.cumsum([len(t) for t in tests])])
    roff = np.concatenate([[0], np.cumsum([len(r) for r in refs])])
    return np.concatenate(tests), toff, np.concatenate(refs), roff


def same_bits(a, b, what):
    """Per-unit FP32 distance arrays equal bit for bit (None: a unit without distances)."""
    for u, (x, y) in enumerate(zip(a, b)):
        if x is not None:
            bad = np.flatnonzero(x.view(np.uint32) != y.view(np.uint32))
            assert bad.size == 0, (what, u, bad[:8], x[bad[:8]], y[bad[:8]])


def check_against_oracle(ctx, tests, refs, cents, res, step, rng_deg, mode, center=None, limes=None, check_dist32=True):
    for u, (t, r, c) in enumerate(zip(tests, refs, cents)):
        o = ora.sweep(t, r, c, mode, step, rng_deg, center=None if center is None else center[u], limes_deg=limes)
        assert res["best_idx"][u] == o["index"], (u, res[u], o["index"], o["cost"])
        assert res["best_angle"][u] == o["angle"]                      # bit-exact f64
        assert res["best_dist"][u] == o["cost"]                        # bit-exact f64
        if check_dist32:
            d32 = ctx.dist32(u, len(o["costs"]))
            rel = np.abs(d32.astype(np.float64) - o["costs"]) / np.maximum(o["costs"], 1e-30)
            assert rel.max() <= REL_TOL_FP32, (u, rel.max())


# ---- the reference's Hausdorff KATs, through the exact device path -----------------
@pytest.mark.parametrize("a,b,want", [
    ([(0, 0), (1, 0), (0, 1)], [(0, 0), (1, 0), (0, 1)], 0.0),           # process_utils.rs:215-245
    ([(0, 0), (1, 0)], [(2, 0), (3, 0)], 2.0),                           # :248-293
    ([(0, 0), (3, 0)], [(1, 0), (2, 0), (4, 0)], 1.0),                   # :296-353
    ([(0, 0), (2, 0), (2, 2), (0, 2)], [(1, 0), (2, 1), (1, 2), (0, 1)], 1.0),  # :379-457
    ([(float(i), 0.0) for i in range(100)], [(i + 0.5, 0.0) for i in range(100)], 0.5),  # :517-547
])
def test_hausdorff_kats_on_device(ctx, a, b, want):
    d = ctx.eval_exact(a, b, (0.0, 0.0), 1, [0.0])[0]
    assert d == pytest.approx(want, abs=1e-10)
    assert d == ora.hausdorff(b, a)


def test_hausdorff_empty_sets_on_device(ctx):  # process_utils.rs:356-376
    e = np.zeros((0, 2))
    assert ctx.eval_exact(e, [(1, 1)], (0, 0), 1, [0.0, 0.3]).tolist() == [0.0, 0.0]
    assert ctx.eval_exact([(1, 1)], e, (0, 0), 1, [0.1]).tolist() == [0.0]


def test_eval_exact_matches_oracle_closures(ctx):
    rng = np.random.default_rng(3)
    t, r = contour(rng, 137), contour(rng, 211, rot=0.3)
    angles = np.concatenate([[0.0, -0.0, math.pi, -math.pi], rng.uniform(-3.1, 3.1, 40)])
    for mode in (0, 1):
        got = ctx.eval_exact(t, r, (4.4, 4.6), mode, angles)
        want = ora.costs(t, r, (4.4, 4.6), mode, angles)
        assert (got == want).all()


# ---- batched sweep vs oracle -----------------------------------------------------------
@pytest.mark.parametrize("mode", [0, 1])
def test_sweep_small_units_brute(ctx, mode):
    rng = np.random.default_rng(11 + mode)
    sizes = [(64, 64), (100, 90), (33, 257), (520, 520), (6, 6), (1, 5), (5, 1), (130, 64)]
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, sizes)
    g = nat.make_grid(0.5, 90.0)
    res = ctx.sweep_batched(txy, toff, rxy, roff, cents, [g], mode=mode, keep_dist32=True)
    check_against_oracle(ctx, tests, refs, cents, res, 0.5, 90.0, mode)
    assert (res["n_shortlist"] >= 1).all()


def test_sweep_default_step_config1_shape(ctx):
    """N=M=520, +-90 deg, 1 deg coarse + 0.5 deg fine (config 1's two stages)."""
    rng = np.random.default_rng(5)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(520, 520)] * 6)
    g = nat.make_grid(1.0, 90.0)
    res = ctx.sweep_batched(txy, toff, rxy, roff, cents, [g], mode=0, keep_dist32=True)
    check_against_oracle(ctx, tests, refs, cents, res, 1.0, 90.0, 0)
    coarse = res["best_angle"]
    grids = [nat.make_grid(0.5, 5.0, center=float(c), limes_deg=90.0) for c in coarse]
    res2 = ctx.sweep_batched(txy, toff, rxy, roff, cents, grids, grid_of_unit=np.arange(6), mode=0, keep_dist32=True)
    check_against_oracle(ctx, tests, refs, cents, res2, 0.5, 5.0, 0, center=coarse, limes=90.0)


def test_sweep_fine_brute_0p01(ctx):
    """Config-2 shaped unit: 36 000 candidates at 0.01 deg over +-180 deg."""
    rng = np.random.default_rng(2)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(520, 520), (500, 520)])
    g = nat.make_grid(0.01, 180.0)
    assert g.n_cand == 36000
    res = ctx.sweep_batched(txy, toff, rxy, roff, cents, [g], mode=0, keep_dist32=True)
    check_against_oracle(ctx, tests, refs, cents, res, 0.01, 180.0, 0)


def test_sweep_multichunk_oct_resolution(ctx):
    """Config-4 shaped unit (N=M=2020 -> 4 register chunks), on a 3 601-candidate grid."""
    rng = np.random.default_rng(9)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(2020, 2020), (2020, 1999), (700, 2020)])
    g = nat.make_grid(0.05, 90.0)
    res = ctx.sweep_batched(txy, toff, rxy, roff, cents, [g], mode=0, keep_dist32=True)
    check_against_oracle(ctx, tests, refs, cents, res, 0.05, 90.0, 0)


def test_zero_angle_shortcut_is_bitwise(ctx):
    """mode 0 must apply ContourPoint::rotate's `angle == 0.0` identity (contour_point.rs:39-41):
    identical sets around an off-grid centre give exactly 0.0 only through the shortcut."""
    rng = np.random.default_rng(4)
    p = contour(rng, 200)
    c = np.array([[4.123456789, 4.987654321]])
    g = nat.make_grid(1.0, 10.0)
    res = ctx.sweep_batched(p, [0, 200], p, [0, 200], c, [g], mode=0)
    assert res["best_dist"][0] == 0.0 and res["best_angle"][0] == 0.0
    o = ora.sweep(p, p, c[0], 0, 1.0, 10.0)
    assert res["best_idx"][0] == o["index"] and o["cost"] == 0.0
    res1 = ctx.sweep_batched(p, [0, 200], p, [0, 200], c, [g], mode=1)
    o1 = ora.sweep(p, p, c[0], 1, 1.0, 10.0)
    assert res1["best_idx"][0] == o1["index"] and res1["best_dist"][0] == o1["cost"]


def test_plateau_ties_resolve_to_lowest_index(ctx):
    """A circle against itself: every angle ties (up to rounding). The reference keeps the
    leftmost minimum (process_utils.rs:69-74); all 181 candidates must be rechecked in f64."""
    n = 180
    phi = np.linspace(0, 2 * np.pi, n, endpoint=False)
    p = np.stack([2.0 * np.cos(phi), 2.0 * np.sin(phi)], axis=1)
    g = nat.make_grid(2.0, 180.0)   # 2-deg steps == the point spacing: every candidate maps the circle onto itself
    res = ctx.sweep_batched(p, [0, n], p, [0, n], [[0.0, 0.0]], [g], mode=0, shortlist_cap=8)
    o = ora.sweep(p, p, (0.0, 0.0), 0, 2.0, 180.0)
    assert res["n_shortlist"][0] == g.n_cand          # one unit may take any share of the recheck pool
    assert res["best_idx"][0] == o["index"]
    assert res["best_dist"][0] == o["cost"]
    idx, d = ctx.shortlist(0)
    order = np.argsort(idx)
    assert (idx[order] == np.arange(g.n_cand)).all() and (d[order] == o["costs"]).all()


def test_recheck_pool_overflow_falls_back_to_full_f64(ctx):
    """72 000 tying candidates exceed the 65 536-item recheck pool: the unit is rechecked over ALL its
    candidates in f64 (MMRS_FLAG_FULL_F64) and must still agree with the oracle bit for bit."""
    n = 72
    phi = np.linspace(0, 2 * np.pi, n, endpoint=False)
    p = np.stack([2.0 * np.cos(phi), 2.0 * np.sin(phi)], axis=1)
    q = np.stack([2.0 * np.cos(phi + 0.01), 2.0 * np.sin(phi + 0.01)], axis=1)
    g = nat.make_grid(0.005, 180.0)
    assert g.n_cand == 72000
    # a huge window makes every candidate a shortlist member
    res = ctx.sweep_batched(np.concatenate([p, q]), [0, n, 2 * n], np.concatenate([p, p]), [0, n, 2 * n],
                            np.zeros((2, 2)), [g], mode=0, shortlist_abs=10.0)
    for u, t in enumerate((p, q)):
        o = ora.sweep(t, p, (0.0, 0.0), 0, 0.005, 180.0, threads=8)
        assert res["best_idx"][u] == o["index"] and res["best_dist"][u] == o["cost"]
    assert (res["flags"] & nat.FLAG_FULL_F64).any()
    idx, d = ctx.shortlist(int(np.argmax(res["flags"] & nat.FLAG_FULL_F64)))
    assert len(idx) == g.n_cand


def test_wrap_duplicates_pick_first(ctx):
    """R=180: candidate 0 and the last candidate can both wrap to -pi; the first must win."""
    rng = np.random.default_rng(8)
    t = contour(rng, 128)
    r = np.stack([-(t[:, 0] - 4.5) + 4.5, -(t[:, 1] - 4.5) + 4.5], axis=1)  # t rotated by pi about (4.5,4.5)
    g = nat.make_grid(1.0, 180.0)
    res = ctx.sweep_batched(t, [0, 128], r, [0, 128], [[4.5, 4.5]], [g], mode=0)
    o = ora.sweep(t, r, (4.5, 4.5), 0, 1.0, 180.0)
    assert res["best_idx"][0] == o["index"] == 0
    assert res["best_angle"][0] == -math.pi


def test_degenerate_and_empty_units(ctx):
    rng = np.random.default_rng(1)
    p = contour(rng, 50)
    e = np.zeros((0, 2))
    g_ok, g_deg = nat.make_grid(1.0, 10.0), nat.make_grid(0.0, 10.0, center=0.25)
    txy = np.concatenate([p, e, p])
    res = ctx.sweep_batched(txy, [0, 50, 50, 100], np.concatenate([p, p, p]), [0, 50, 100, 150],
                            np.zeros((3, 2)) + 4.5, [g_ok, g_deg], grid_of_unit=[0, 0, 1], mode=0)
    assert res["flags"][1] & nat.FLAG_EMPTY and res["best_idx"][1] == 0 and res["best_dist"][1] == 0.0
    assert res["best_angle"][1] == ora.sweep(e, p, (4.5, 4.5), 0, 1.0, 10.0)["angle"]
    assert res["flags"][2] & nat.FLAG_DEGENERATE and res["best_idx"][2] == -1 and res["best_angle"][2] == 0.25
    assert res["best_idx"][0] == ora.sweep(p, p, (4.5, 4.5), 0, 1.0, 10.0)["index"]


@pytest.mark.parametrize("mode", [0, 1])
def test_units_beyond_the_shared_memory_staging(ctx, mode):
    """The reference has no size limit (process_utils.rs:84-121). Units that do not fit K1's shared-memory staging
    (more than ~4 000 points per set) take the blocked kernel K1b (reference set streamed through shared memory in
    blocks, row minima kept across blocks) and the f64 recheck with its rotated points in global memory: N = M = 8 000,
    lopsided sets, next to an ordinary 520-point unit in the same batch — same bars as everywhere else."""
    rng = np.random.default_rng(5 + mode)
    sizes = [(8000, 8000), (520, 520), (5000, 300), (300, 9000), (4500, 4600)]
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, sizes)
    g = nat.make_grid(1.0, 12.0)
    res = ctx.sweep_batched(txy, toff, rxy, roff, cents, [g], mode=mode, keep_dist32=True)
    p = ctx.plan()
    assert p["blocked"] and p["size_classes"] >= 2
    for u, (t, r, c) in enumerate(zip(tests, refs, cents)):
        o = ora.sweep(t, r, c, mode, 1.0, 12.0, threads=16)
        assert res["best_idx"][u] == o["index"] and res["best_angle"][u] == o["angle"], (u, sizes[u])
        assert res["best_dist"][u] == o["cost"], (u, sizes[u])
        d32 = ctx.dist32(u, len(o["costs"])).astype(np.float64)
        assert (np.abs(d32 - o["costs"]) <= REL_TOL_FP32 * o["costs"]).all(), (u, sizes[u])
    # the literal cost closure on oversize sets (rotated points in global scratch)
    ang = np.array([0.0, 0.1, -0.2])
    assert np.array_equal(ctx.eval_exact(tests[0], refs[0], cents[0], mode, ang), ora.costs(tests[0], refs[0], cents[0], mode, ang))
    big = contour(rng, 6000)
    res = ctx.sweep_batched(big, [0, 6000], big, [0, 6000], np.zeros((1, 2)) + 4.5, [nat.make_grid(1.0, 5.0)], mode=0)
    assert res["best_idx"][0] == 5 and res["best_dist"][0] == 0.0          # the identity rotation of a set on itself


def test_three_step_api_and_timings(ctx):
    rng = np.random.default_rng(12)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(256, 256)] * 4)
    g = nat.make_grid(0.1, 30.0)
    ctx.sweep_upload(txy, toff, rxy, roff, cents, [g], mode=0)
    ctx.sweep_run()
    a = ctx.sweep_download()
    ctx.sweep_run()   # idempotent on resident inputs
    b = ctx.sweep_download()
    assert (a == b).all()
    t = ctx.timings()
    assert t["launches"] == 4 and t["sweep_ms"] > 0
    check_against_oracle(ctx, tests, refs, cents, a, 0.1, 30.0, 0, check_dist32=False)


def test_regrid_keeps_points_resident(ctx):
    """mmrs_sweep_regrid: second window of find_best_rotation on the SAME uploaded points must equal a
    fresh upload with those grids; skipped (degenerate-grid) units are reported as such."""
    rng = np.random.default_rng(31)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(300, 280), (520, 520), (128, 128)])
    ctx.sweep_upload(txy, toff, rxy, roff, cents, [nat.make_grid(1.0, 60.0)], mode=0)
    ctx.sweep_run()
    coarse = ctx.sweep_download()
    grids = [nat.make_grid(0.1, 5.0, center=float(c), limes_deg=60.0) for c in coarse["best_angle"]]
    grids[2] = nat.make_grid(0.0, 5.0, center=0.125)          # degenerate: this unit is skipped
    ctx.sweep_regrid(grids, grid_of_unit=[0, 1, 2])
    ctx.sweep_run()
    fine = ctx.sweep_download()
    fresh = ctx.sweep_batched(txy, toff, rxy, roff, cents, grids, grid_of_unit=[0, 1, 2], mode=0)
    assert (fine == fresh).all()
    assert fine["flags"][2] & nat.FLAG_DEGENERATE and fine["best_angle"][2] == 0.125
    for u in range(2):
        o = ora.sweep(tests[u], refs[u], cents[u], 0, 0.1, 5.0, center=float(coarse["best_angle"][u]), limes_deg=60.0)
        assert fine["best_idx"][u] == o["index"] and fine["best_dist"][u] == o["cost"]


def test_rotation_linearity_property_full_size(ctx):
    """Size-independent property at BASELINE sizes: rotating the test contour by a grid angle
    shifts the arg-min by exactly that many candidates (no oracle needed)."""
    rng = np.random.default_rng(21)
    n = 2000
    ref = contour(rng, n, noise=0.0)
    step = 0.05
    g = nat.make_grid(step, 90.0)
    k = 137
    a = -k * step * math.pi / 180.0
    c, s = math.cos(a), math.sin(a)
    q = ref - 4.5
    test = np.stack([q[:, 0] * c - q[:, 1] * s, q[:, 0] * s + q[:, 1] * c], axis=1) + 4.5
    res = ctx.sweep_batched(test, [0, n], ref, [0, n], [[4.5, 4.5]], [g], mode=1)
    mid = (g.n_cand - 1) // 2
    assert abs(int(res["best_idx"][0]) - (mid + k)) <= 1
    assert res["best_dist"][0] < 1e-3


def test_fp32_error_stays_inside_half_the_shortlist_window(ctx):
    """Soundness of the FP32 filter: the f64 arg-min is guaranteed to be rechecked iff
    |d32 - d64| <= window/2 for every candidate, window = 2e-6 * d_min + 2e-6 * Rmax (DESIGN.md §4)."""
    rng = np.random.default_rng(77)
    sizes = [(520, 520), (505, 505), (2020, 2020), (64, 300), (600, 600)]
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, sizes)
    g = nat.make_grid(0.25, 180.0)
    res = ctx.sweep_batched(txy, toff, rxy, roff, cents, [g], mode=0, keep_dist32=True)
    worst = 0.0
    for u, (t, r, c) in enumerate(zip(tests, refs, cents)):
        o = ora.sweep(t, r, c, 0, 0.25, 180.0, threads=8)
        d32 = ctx.dist32(u, g.n_cand).astype(np.float64)
        rmax = max(np.abs(t - c).max(), np.abs(r - c).max())
        half_window = 0.5 * (2e-6 * o["costs"].min() + 2e-6 * rmax)
        err = np.abs(d32 - o["costs"]).max()
        worst = max(worst, err / half_window)
        assert err <= half_window, (u, err, half_window)
        assert res["best_idx"][u] == o["index"]
    assert worst < 1.0


def test_fp32_probe_reports_plausible_peak(ctx):
    tf = ctx.fp32_probe(2048)
    assert 20.0 < tf < 90.0, tf


# ---- exact tiling (tail pass) and size classes -----------------------------------------------------
@pytest.mark.parametrize("mode", [0, 1])
def test_exact_tiling_tail_pass(ctx, mode):
    """Test sets of 32 TA + R points (R = 1 ... 31) take the exact-tiling kernel: 32 TA points in register slots and
    a tail pass over the rest. Odd and even reference counts, reference sets at the edge of the tail pass's
    register budget (M <= 32 (TA + 1)), and the same sizes one point past it (padded slot instead)."""
    rng = np.random.default_rng(21 + mode)
    sizes = [(520, 520), (521, 519), (513, 544), (543, 512), (520, 545), (130, 128), (159, 160), (200, 193), (577, 600)]
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, sizes)
    g = nat.make_grid(0.25, 45.0)
    res = ctx.sweep_batched(txy, toff, rxy, roff, cents, [g], mode=mode, keep_dist32=True)
    assert ctx.plan()["size_classes"] >= 3
    check_against_oracle(ctx, tests, refs, cents, res, 0.25, 45.0, mode)


def test_exact_tiling_is_the_plan_for_520_points(ctx):
    rng = np.random.default_rng(23)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(520, 520)] * 3)
    ctx.sweep_upload(txy, toff, rxy, roff, cents, [nat.make_grid(1.0, 20.0)], mode=0)
    p = ctx.plan()
    assert (p["TA"], p["multi"], p["exact_tiling"], p["size_classes"]) == (16, False, True, 1)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(510, 510)] * 3)
    ctx.sweep_upload(txy, toff, rxy, roff, cents, [nat.make_grid(1.0, 20.0)], mode=0)
    p = ctx.plan()
    assert (p["TA"], p["multi"], p["exact_tiling"]) == (16, False, False)


def test_mixed_size_classes_in_one_batch(ctx):
    """520-point frame pairs next to OCT-resolution (2 020, four register chunks) and small units: one launch per
    size class instead of one register tile for the whole batch; pruned list re-scoring goes through the classes too."""
    rng = np.random.default_rng(29)
    sizes = [(520, 520), (2020, 2020), (300, 310), (520, 520), (1000, 1000), (2020, 2000)]
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, sizes)
    g = nat.make_grid(0.1, 30.0)
    res = ctx.sweep_batched(txy, toff, rxy, roff, cents, [g], mode=0, keep_dist32=True)
    assert ctx.plan()["size_classes"] >= 3
    check_against_oracle(ctx, tests, refs, cents, res, 0.1, 30.0, 0)
    pr = ctx.sweep_batched(txy, toff, rxy, roff, cents, [g], mode=0, prune=1)
    assert ctx.prefilter_info()["kind"] == "lower-bound pruning"
    for k in ("best_idx", "best_angle", "best_dist", "n_ties"):
        assert (pr[k] == res[k]).all(), k


@pytest.mark.parametrize("mode", [0, 1])
def test_chunked_units_with_odd_reference_counts(ctx, mode):
    """The main loop walks four reference points per trip and closes with an odd float4; chunked units keep their
    column minima in a per-warp shared-memory row whose stride is rounded up to 16 bytes. Reference counts of every
    residue mod 4 (and odd), against chunked (N > 576), padded and exact-tiling test sets."""
    rng = np.random.default_rng(31 + mode)
    sizes = [(700, 601), (1301, 1203), (1154, 1150), (640, 77), (900, 3), (2021, 2017), (577, 578), (96, 5), (520, 2)]
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, sizes)
    g = nat.make_grid(0.5, 20.0)
    res = ctx.sweep_batched(txy, toff, rxy, roff, cents, [g], mode=mode, keep_dist32=True)
    check_against_oracle(ctx, tests, refs, cents, res, 0.5, 20.0, mode)


# ---- non-finite coordinates (process_utils.rs:108, :112) -------------------------------------------------
def test_non_finite_points_take_no_part(ctx):
    """A NaN distance never passes `d2 < min_sq` and a non-finite row minimum is skipped (process_utils.rs:104-114), so
    a point with a NaN / infinite coordinate takes part in neither directed pass, in either role. Units with such
    points in the test set, in the reference set, in both, and a set made ONLY of them (every candidate costs 0.0, the
    leftmost wins) must select what the oracle's literal loops select, with bit-equal f64 distances."""
    rng = np.random.default_rng(31)
    sizes = [(200, 200), (520, 520), (130, 140), (64, 64), (300, 300)]
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, sizes)
    nan, inf = float("nan"), float("inf")
    tests[0][7] = (nan, 1.0)
    tests[0][100] = (inf, -inf)
    refs[1][0] = (nan, nan)
    refs[1][519] = (2.0, inf)
    tests[2][5] = (nan, nan)
    refs[2][9] = (-inf, 0.5)
    tests[3][:] = nan                      # all rows non-finite: both directed distances are 0.0 at every angle
    txy, rxy = np.concatenate(tests), np.concatenate(refs)
    g = nat.make_grid(0.5, 60.0)
    for mode in (0, 1):
        res = ctx.sweep_batched(txy, toff, rxy, roff, cents, [g], mode=mode)
        for u, (t, r, c) in enumerate(zip(tests, refs, cents)):
            o = ora.sweep(t, r, c, mode, 0.5, 60.0)
            assert res["best_idx"][u] == o["index"] and res["best_angle"][u] == o["angle"], (mode, u)
            assert res["best_dist"][u] == o["cost"], (mode, u)
        assert res["best_idx"][3] == 0 and res["best_dist"][3] == 0.0
    # the literal cost closure on the device (no filtering in front of it) agrees with the oracle's loops too
    angles = np.array([0.0, 0.3, -1.2])
    for u in (0, 1, 2, 3):
        got = ctx.eval_exact(tests[u], refs[u], cents[u], 0, angles)
        assert np.array_equal(got, ora.costs(tests[u], refs[u], cents[u], 0, angles)), u


def test_contexts_on_several_host_threads_with_different_unit_sizes():
    """Several contexts driven from several host threads on one GPU (the cohort pipeline does this): the dynamic
    shared-memory limit of a kernel is per-function state shared by all of them, so it is raised once to the opt-in
    maximum and never lowered — launches of the same instantiation with different sizes must not disturb each other."""
    import threading

    rng = np.random.default_rng(77)
    jobs = []
    for sizes in ([(520, 520)] * 3, [(700, 650)] * 3, [(300, 310), (2020, 2020)], [(130, 128)] * 4):
        tests, refs, cents, txy, toff, rxy, roff = make_units(rng, sizes)
        want = [ora.sweep(t, r, c, 0, 0.5, 20.0) for t, r, c in zip(tests, refs, cents)]
        jobs.append((txy, toff, rxy, roff, cents, want))
    errs = []

    def run(job):
        txy, toff, rxy, roff, cents, want = job
        try:
            c = nat.Context(0)
            g = nat.make_grid(0.5, 20.0)
            for _ in range(6):
                res = c.sweep_batched(txy, toff, rxy, roff, cents, [g], mode=0)
                for u, o in enumerate(want):
                    assert res["best_idx"][u] == o["index"] and res["best_dist"][u] == o["cost"]
            c.close()
        except Exception as e:  # noqa: BLE001
            errs.append(repr(e))

    threads = [threading.Thread(target=run, args=(j,)) for j in jobs]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errs, errs
