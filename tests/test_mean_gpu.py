"""The mean cost (include/mmrs_b200.h "mean cost") on the GPU.

1. mmrs_eval_exact_mean against the f64 restatement in tests/cost_oracle.py, bit for bit.
2. The sweep against the oracle over every K1 size class (padded odd and even register tiles, exact tiling with even
   and odd tails, n = 32 TA +- 1, odd m, tiny and duplicated sets, the chunked 2 020-point class, rigid batches):
   selection, f64 distance and ties exactly, and every candidate's FP32 value within the documented bound of its f64
   cost (a padding duplicate counted in a sum would move the mean by about d / n, far outside it).
3. Regrids keep the cost, a plain upload clears it. 4. A planted transform is recovered. 5. Launches and tier.
6. find_best_rigid_transform(cost="mean"). 7. Error cases."""
import numpy as np
import pytest

import multimodars as mm
from multimodars import _native as nat
from oracle import oracle_py as ora
from tests import cost_oracle as co
from tests.test_sweep_gpu import contour, make_units, pack

pytestmark = pytest.mark.gpu

FIELDS = ("best_idx", "best_angle", "best_dist", "best_dist_f32", "n_shortlist", "n_ties", "flags")

# the FP32 -> f64 bound of include/mmrs_b200.h "mean cost": 5e-7 R + 3.6e-7 d (R: Rmax, or R_eff for rigid runs)
ABS_BOUND, REL_BOUND = 5e-7, 3.6e-7
WORST = {"ratio": 0.0}   # largest |d32 - d64| / R_eff seen


@pytest.fixture(scope="module")
def ctx():
    c = nat.Context(0)
    yield c
    c.close()
    print(f"\nmean cost: largest |d32 - d64| / R_eff = {WORST['ratio']:.3e}")


def mean_run(ctx, tests, refs, cents, grid, tg=None, mode=0, **opts):
    """One mean sweep with keep_dist32: (results, dist32 per unit (None for an empty set))."""
    txy, toff, rxy, roff = pack(tests, refs)
    ctx.mean_upload(txy, toff, rxy, roff, cents, [grid], None if tg is None else [tg], mode=mode, keep_dist32=True,
                    **opts)
    ctx.sweep_run()
    res = ctx.sweep_download() if tg is None else ctx.rigid_download()
    T = 1 if tg is None else (2 * tg.half_n + 1) ** 2
    d32 = [ctx.dist32(u, grid.n_cand * T) if len(tests[u]) and len(refs[u]) else None for u in range(len(tests))]
    return res, d32


def check_oracle(ctx, tests, refs, cents, res, d32, grid_params, mode, tg=None):
    offs = np.zeros((1, 2)) if tg is None else co.offsets_of(tg)
    T = len(offs)
    angles, _ = ora.search_grid(*grid_params)
    for u in range(len(tests)):
        idx, costs = co.search(tests[u], refs[u], cents[u], mode, angles, offs, "mean")
        flat = costs.reshape(-1)
        assert res["best_idx"][u] == idx, (u, res["best_idx"][u], idx)
        assert res["best_angle"][u] == angles[idx // T]
        assert res["best_dist"][u] == flat[idx], (u, res["best_dist"][u], flat[idx])
        if tg is not None:
            assert res["best_tx"][u] == offs[idx % T, 0] and res["best_ty"][u] == offs[idx % T, 1]
        assert res["n_ties"][u] == int(np.sum(flat == flat[idx]))   # tie_margin 0: equal f64 cost, another transform
        d64 = ctx.eval_exact_mean(tests[u], refs[u], cents[u], mode, np.repeat(angles, T),
                                  None if tg is None else np.tile(offs, (len(angles), 1)))
        assert np.array_equal(d64, flat), u
        if d32[u] is not None:
            pts = np.concatenate([co.finite(tests[u]), co.finite(refs[u])])
            r_eff = np.abs(pts - cents[u]).max() + np.hypot(offs[:, 0], offs[:, 1]).max()
            err = np.abs(d32[u].astype(np.float64) - flat)
            assert (err <= ABS_BOUND * r_eff + REL_BOUND * flat).all(), (u, len(tests[u]), len(refs[u]), err.max(), r_eff)
            WORST["ratio"] = max(WORST["ratio"], float(err.max() / r_eff))


# ---- 1. the f64 evaluation ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [0, 1])
def test_eval_exact_mean_against_oracle(ctx, mode):
    rng = np.random.default_rng(300 + mode)
    a_dup = np.repeat(rng.normal(0, 1, (20, 2)), 3, axis=0)
    nf = contour(rng, 60)
    nf[[2, 30]] = np.nan
    nf_r = contour(rng, 45)
    nf_r[5, 0] = np.inf
    pairs = [(rng.normal(0, 1, (57, 2)), rng.normal(0, 1.2, (43, 2))),     # N != M
             (rng.normal(0, 1, (1, 2)), rng.normal(0, 1, (2, 2))),         # 1-3 points
             (rng.normal(0, 1, (3, 2)), rng.normal(0, 1, (1, 2))),
             (a_dup, rng.normal(0, 1, (30, 2))),                           # duplicated points
             (nf, nf_r),                                                   # non-finite points dropped
             co.crafted_order_case()]                                      # sequential order differs from pairwise
    angles = np.array([0.0, 0.3, -1.1, 2.5])
    txy = np.array([[0.0, 0.0], [0.1, -0.2], [0.0, 0.05], [-0.3, 0.01]])
    for test, ref in pairs:
        cen = (0.1, -0.1)
        got = ctx.eval_exact_mean(test, ref, cen, mode, angles)
        want = np.array([co.candidate_cost(test, ref, cen, mode, a, (0.0, 0.0), "mean") for a in angles])
        assert np.array_equal(got, want), (got, want)
        got = ctx.eval_exact_mean(test, ref, cen, mode, angles, txy)
        want = np.array([co.candidate_cost(test, ref, cen, mode, a, t, "mean") for a, t in zip(angles, txy)])
        assert np.array_equal(got, want), (got, want)
    empty = np.zeros((0, 2))
    assert (ctx.eval_exact_mean(empty, pairs[0][1], (0, 0), mode, angles) == 0.0).all()
    assert (ctx.eval_exact_mean(np.full((4, 2), np.nan), pairs[0][1], (0, 0), mode, angles) == 0.0).all()


# ---- 2. the sweep against the oracle --------------------------------------------------------------------------------
# (n, m): padded even / odd register tiles, n = 32 TA +- 1, odd m, exact tiling (520 = 16 * 32 + 8; 257 = 8 * 32 + 1,
# an odd tail), tiny sets
SHAPES = [(100, 90), (95, 97), (161, 130), (159, 158), (520, 520), (520, 511), (257, 199), (1, 1), (3, 2), (2, 3)]


@pytest.mark.parametrize("mode", [0, 1])
def test_sweep_against_oracle_every_class(ctx, mode):
    rng = np.random.default_rng(310 + mode)
    tests, refs, cents, *_ = make_units(rng, SHAPES)
    tests.append(np.repeat(contour(rng, 40), 3, axis=0))             # duplicated points
    refs.append(np.repeat(contour(rng, 35), 2, axis=0))
    nf_t, nf_r = contour(rng, 200), contour(rng, 180)
    nf_t[[3, 50, 51]] = np.nan
    nf_r[7] = np.inf
    tests += [nf_t, np.zeros((0, 2))]
    refs += [nf_r, contour(rng, 50)]                                   # ... and an empty set
    cents = np.concatenate([cents, [[4.5, 4.5]] * 3])
    g = nat.make_grid(3.0, 30.0)
    res, d32 = mean_run(ctx, tests, refs, cents, g, mode=mode)
    assert res["flags"][-1] & nat.FLAG_EMPTY and res["best_dist"][-1] == 0.0
    check_oracle(ctx, tests[:-1], refs[:-1], cents[:-1], res[:-1], d32[:-1], (3.0, 30.0, None, 30.0), mode)


def test_sweep_against_oracle_chunked_units(ctx):
    rng = np.random.default_rng(320)
    tests, refs, cents, *_ = make_units(rng, [(2020, 2020), (2020, 1901)])
    g = nat.make_grid(0.05, 0.2)
    res, d32 = mean_run(ctx, tests, refs, cents, g, mode=1)
    check_oracle(ctx, tests, refs, cents, res, d32, (0.05, 0.2, None, 0.2), 1)


@pytest.mark.parametrize("mode", [0, 1])
def test_sweep_against_oracle_rigid(ctx, mode):
    rng = np.random.default_rng(330 + mode)
    tests, refs, cents, *_ = make_units(rng, [(100, 90), (95, 97), (520, 520), (257, 199), (3, 2)])
    tg = nat.make_tgrid(0.05, 1, t0=(0.02, -0.01))
    res, d32 = mean_run(ctx, tests, refs, cents, nat.make_grid(4.0, 20.0), tg, mode=mode)
    check_oracle(ctx, tests, refs, cents, res, d32, (4.0, 20.0, None, 20.0), mode, tg)


# ---- 3. regrids keep the cost; a plain upload clears it -------------------------------------------------------------
def test_regrid_keeps_the_cost_and_plain_upload_clears_it(ctx):
    rng = np.random.default_rng(340)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(520, 520), (100, 90), (159, 158)])
    plain0 = ctx.sweep_batched(txy, toff, rxy, roff, cents, [nat.make_grid(1.0, 180.0)], keep_dist32=True)
    ctx.mean_upload(txy, toff, rxy, roff, cents, [nat.make_grid(1.0, 180.0)])
    ctx.sweep_run()
    coarse = ctx.sweep_download()
    grids = [nat.make_grid(0.01, 0.5, center=float(a), limes_deg=180.0) for a in coarse["best_angle"]]
    ctx.sweep_regrid(grids, grid_of_unit=np.arange(3))
    ctx.sweep_run()
    fine = ctx.sweep_download()
    for u in range(3):
        angles, _ = ora.search_grid(0.01, 0.5, float(coarse["best_angle"][u]), 180.0)
        idx, costs = co.search(tests[u], refs[u], cents[u], 0, angles, np.zeros((1, 2)), "mean")
        assert fine["best_idx"][u] == idx and fine["best_dist"][u] == costs.reshape(-1)[idx]
    ctx.sweep_upload(txy, toff, rxy, roff, cents, [nat.make_grid(1.0, 180.0)], keep_dist32=True)
    ctx.sweep_run()
    plain1 = ctx.sweep_download()
    for f in FIELDS:
        assert np.array_equal(plain0[f], plain1[f]), f


# ---- 4. a planted transform -----------------------------------------------------------------------------------------
def test_planted_rotation_and_translation_recovered(ctx):
    rng = np.random.default_rng(350)
    ref = contour(rng, 400)
    cen = ref.mean(axis=0)
    g = nat.make_grid(0.5, 20.0)
    tg = nat.make_tgrid(0.05, 3)
    offs = co.offsets_of(tg)
    i_star, j_star = 23, 3 * 7 + 5
    theta = nat.grid_angle(g, i_star)
    c, s = np.cos(theta), np.sin(theta)
    # test = the reference moved by the inverse of the planted transform, so (theta, t) maps it back onto ref
    x, y = ref[:, 0] - offs[j_star, 0] - cen[0], ref[:, 1] - offs[j_star, 1] - cen[1]
    test = np.stack([x * c + y * s + cen[0], -x * s + y * c + cen[1]], 1)
    res, _ = mean_run(ctx, [test], [ref], cen[None], g, tg, mode=1)
    T = len(offs)
    assert res["best_idx"][0] == i_star * T + j_star
    assert res["best_dist"][0] < 1e-9


# ---- 5. launches and tier -------------------------------------------------------------------------------------------
def test_launches_and_dense_tier(ctx):
    rng = np.random.default_rng(360)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(100, 90), (520, 520), (2020, 2020), (95, 97)])
    ctx.mean_upload(txy, toff, rxy, roff, cents, [nat.make_grid(1.0, 30.0)])
    C = ctx.plan()["size_classes"]
    assert C == 4
    ctx.sweep_run()
    assert ctx.timings()["launches"] == C + 3
    info = ctx.prefilter_info()
    assert not info["ran"] and info["kind"] is None and info["eb_candidates"] == 0
    # MMRS_EARLY_BREAK does not apply: the same run with it on gives the same launches and results
    first = ctx.sweep_download()
    mp = pytest.MonkeyPatch()
    try:
        mp.setenv("MMRS_EARLY_BREAK", "1")
        ctx.mean_upload(txy, toff, rxy, roff, cents, [nat.make_grid(1.0, 30.0)])
        ctx.sweep_run()
    finally:
        mp.undo()
    assert ctx.timings()["launches"] == C + 3 and ctx.prefilter_info()["eb_candidates"] == 0
    again = ctx.sweep_download()
    for f in FIELDS:
        assert np.array_equal(first[f], again[f]), f


# ---- 6. the public function -----------------------------------------------------------------------------------------
def test_find_best_rigid_transform_mean_against_oracle():
    rng = np.random.default_rng(370)
    tests, refs, _, *_ = make_units(rng, [(80, 90), (64, 64)])
    kw = dict(step_rotation_deg=0.5, range_rotation_deg=10.0, step_translation=0.05)
    offs = co.tgrid_offsets(0.0, 0.0, 0.05, 1)
    for brute in (False, True):
        out = mm.find_best_rigid_transform(tests, refs, range_translation=0.05, bruteforce=brute, cost="mean", **kw)
        for u in range(2):
            cen = (np.cumsum(refs[u][:, 0])[-1] / len(refs[u]), np.cumsum(refs[u][:, 1])[-1] / len(refs[u]))
            a, j, tx, ty, d = co.coarse_to_fine(tests[u], refs[u], cen, 1, 0.5, 10.0, offs, "mean", bruteforce=brute)
            assert out["angle_rad"][u] == a and out["tx"][u] == tx and out["ty"][u] == ty and out["distance"][u] == d
    rot = mm.find_best_rigid_transform(tests, refs, range_translation=0.0, cost="mean", **kw)   # rotation only
    for u in range(2):
        cen = (np.cumsum(refs[u][:, 0])[-1] / len(refs[u]), np.cumsum(refs[u][:, 1])[-1] / len(refs[u]))
        a, j, tx, ty, d = co.coarse_to_fine(tests[u], refs[u], cen, 1, 0.5, 10.0, np.zeros((1, 2)), "mean")
        assert rot["angle_rad"][u] == a and rot["tx"][u] == 0.0 and rot["ty"][u] == 0.0 and rot["distance"][u] == d
    same = mm.find_best_rigid_transform(tests, refs, range_translation=0.05, **kw)
    full = mm.find_best_rigid_transform(tests, refs, range_translation=0.05, cost="hausdorff", **kw)
    assert same.tobytes() == full.tobytes()


# ---- 7. errors ------------------------------------------------------------------------------------------------------
def test_error_cases(ctx):
    rng = np.random.default_rng(380)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(300, 300), (40, 40)])
    g = [nat.make_grid(1.0, 10.0)]
    big_t, big_toff, big_r, big_roff = (np.concatenate([txy, contour(rng, 5000)]), np.append(toff, toff[-1] + 5000),
                                        np.concatenate([rxy, contour(rng, 5000)]), np.append(roff, roff[-1] + 5000))
    with pytest.raises(nat.MmrsError, match="mean cost: unit 2 is beyond the shared-memory staging"):
        ctx.mean_upload(big_t, big_toff, big_r, big_roff, np.concatenate([cents, [[4.5, 4.5]]]), g)
    with pytest.raises(nat.MmrsError, match="prune is not supported with the mean cost"):
        ctx.mean_upload(txy, toff, rxy, roff, cents, g, prune=1)
    for pf in (2, 3):
        with pytest.raises(nat.MmrsError, match="prefilter 2 / 3 is not supported with the mean cost"):
            ctx.mean_upload(txy, toff, rxy, roff, cents, g, prefilter=pf)
    ctx.mean_upload(txy, toff, rxy, roff, cents, g)   # the context still works after the errors
    ctx.sweep_run()
    assert (ctx.sweep_download()["best_idx"] >= 0).all()
