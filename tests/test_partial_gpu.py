"""The partial cost (include/mmrs_b200.h "partial cost") on the GPU.

1. inlier_fraction = 1 is the plain rotation-only / rigid sweep, field for field and dist32 bit for bit; in a batch
   with f < 1, units whose q is 0 in both directions match the plain sweep.
2. Early break on (K1e-partial) equals early break off (every row scanned to its end), dist32 bit for bit.
3. Results against the f64 restatement in tests/cost_oracle.py and mmrs_eval_exact_partial.
4. A planted transform is recovered despite a 3-point bulge. 5. find_best_rigid_transform(inlier_fraction=...).
6. Error cases."""
import numpy as np
import pytest

import bench
import multimodars as mm
from multimodars import _native as nat
from oracle import oracle_py as ora
from tests import cost_oracle as co
from tests.test_sweep_gpu import contour, make_units, pack, same_bits

pytestmark = pytest.mark.gpu

FIELDS = ("best_idx", "best_angle", "best_dist", "best_dist_f32", "n_shortlist", "n_ties", "flags")
RIGID_FIELDS = FIELDS + ("angle_idx", "trans_idx", "best_tx", "best_ty")


@pytest.fixture(scope="module")
def ctx():
    c = nat.Context(0)
    yield c
    c.close()


def n_cands(tests, refs, grids, tgrids, gou=None):
    T = 1 if tgrids is None else (2 * tgrids[0].half_n + 1) ** 2
    return [0 if grids[0 if gou is None else gou[u]].degenerate else grids[0 if gou is None else gou[u]].n_cand * T
            for u in range(len(tests))]


def partial(ctx, tests, refs, cents, grids, f, tgrids=None, gou=None, mode=0, **opts):
    """One partial sweep with keep_dist32: (results, dist32 per unit (None for an empty set), prefilter_info)."""
    txy, toff, rxy, roff = pack(tests, refs)
    ctx.partial_upload(txy, toff, rxy, roff, cents, grids, tgrids, grid_of_unit=gou, mode=mode, inlier_fraction=f,
                       keep_dist32=True, **opts)
    ctx.sweep_run()
    res = ctx.sweep_download() if tgrids is None else ctx.rigid_download()
    nc = n_cands(tests, refs, grids, tgrids, gou)
    d32 = [ctx.dist32(u, int(nc[u])) if len(tests[u]) and len(refs[u]) else None for u in range(len(tests))]
    return res, d32, ctx.prefilter_info()


def plain(ctx, tests, refs, cents, grids, tgrids=None, gou=None, mode=0):
    txy, toff, rxy, roff = pack(tests, refs)
    if tgrids is None:
        res = ctx.sweep_batched(txy, toff, rxy, roff, cents, grids, grid_of_unit=gou, mode=mode, keep_dist32=True)
    else:
        res = ctx.rigid_sweep_batched(txy, toff, rxy, roff, cents, grids, tgrids, grid_of_unit=gou, mode=mode,
                                      keep_dist32=True)
    nc = n_cands(tests, refs, grids, tgrids, gou)
    return res, [ctx.dist32(u, int(nc[u])) if len(tests[u]) and len(refs[u]) else None for u in range(len(tests))]


def bench_units(k, rng_deg=None):
    txy, toff, rxy, roff, cen, U, n = bench.make_units()
    pick = np.linspace(0, U - 1, k).astype(int)
    return ([txy[toff[u]:toff[u + 1]] for u in pick], [rxy[roff[u]:roff[u + 1]] for u in pick], cen[pick])


def mixed_shapes(seed):
    """Random clouds (N != M), circle on circle, a contour against itself, tiny, duplicated and non-finite sets."""
    rng = np.random.default_rng(seed)
    tests, refs, cents, *_ = make_units(rng, [(520, 520), (300, 411)])
    tests.append(rng.normal(0, 1.0, (300, 2)))
    refs.append(rng.normal(0, 1.2, (211, 2)))
    phi = np.linspace(0, 2 * np.pi, 360, endpoint=False)
    circ = np.stack([2.0 * np.cos(phi), 2.0 * np.sin(phi)], 1)
    own = contour(rng, 256)
    tests += [circ, own, rng.normal(0, 1, (6, 2)), np.repeat(rng.normal(0, 1, (40, 2)), 3, axis=0)]
    refs += [circ.copy(), own.copy(), rng.normal(0, 1, (6, 2)), np.repeat(rng.normal(0, 1, (30, 2)), 2, axis=0)]
    nf_t, nf_r = contour(rng, 200), contour(rng, 180)
    nf_t[[3, 50, 51]] = np.nan
    nf_r[7] = np.inf
    tests.append(nf_t)
    refs.append(nf_r)
    cents = np.concatenate([cents, np.zeros((2, 2)), [[4.5, 4.5]], np.zeros((2, 2)), [[4.5, 4.5]]])
    return tests, refs, cents


# ---- 1. f = 1 is the plain sweep ---------------------------------------------------------------------------------
@pytest.mark.parametrize("rigid", [False, True])
def test_full_fraction_is_the_plain_sweep(ctx, monkeypatch, rigid):
    tests, refs, cents = mixed_shapes(201)
    grids = [nat.make_grid(1.0, 180.0)]
    tg = [nat.make_tgrid(0.05, 1, t0=(0.01, -0.02))] if rigid else None
    for flag in ("0", "1"):
        monkeypatch.setenv("MMRS_EARLY_BREAK", flag)
        r0, d0 = plain(ctx, tests, refs, cents, grids, tg)
        r1, d1, _ = partial(ctx, tests, refs, cents, grids, 1.0, tg)
        for f in (RIGID_FIELDS if rigid else FIELDS):
            assert np.array_equal(r0[f], r1[f]), (flag, f)
        same_bits(d0, d1, f"f = 1, MMRS_EARLY_BREAK={flag}")
    monkeypatch.delenv("MMRS_EARLY_BREAK")


def test_units_without_outliers_match_the_plain_sweep(ctx, monkeypatch):
    """f = 0.9: units of <= 9 points per set have q = 0 in both directions."""
    rng = np.random.default_rng(203)
    tests, refs, cents, *_ = make_units(rng, [(6, 9), (520, 520), (8, 7), (130, 97), (9, 9)])
    grids = [nat.make_grid(0.5, 180.0)]
    for flag in ("0", "1"):
        monkeypatch.setenv("MMRS_EARLY_BREAK", flag)
        r0, d0 = plain(ctx, tests, refs, cents, grids)
        r1, d1, _ = partial(ctx, tests, refs, cents, grids, 0.9)
        for u in (0, 2, 4):
            for f in FIELDS:
                assert r0[f][u] == r1[f][u], (flag, u, f)
            same_bits([d0[u]], [d1[u]], f"q = 0 unit {u}")
        assert r1["best_dist"][1] < r0["best_dist"][1]
    monkeypatch.delenv("MMRS_EARLY_BREAK")


# ---- 2. early break on == off ------------------------------------------------------------------------------------
def on_vs_off(ctx, monkeypatch, tests, refs, cents, grids, f, tgrids=None, gou=None, mode=0):
    runs = []
    for flag in ("0", "1"):
        monkeypatch.setenv("MMRS_EARLY_BREAK", flag)
        runs.append(partial(ctx, tests, refs, cents, grids, f, tgrids, gou=gou, mode=mode))
    monkeypatch.delenv("MMRS_EARLY_BREAK")
    (r0, d0, i0), (r1, d1, i1) = runs
    assert i0["eb_candidates"] > 0 and i1["eb_candidates"] == i0["eb_candidates"]
    same_bits(d0, d1, f"early break on vs off, f = {f}")
    for f_ in (RIGID_FIELDS if tgrids is not None else FIELDS):
        assert np.array_equal(r0[f_], r1[f_]), f_
    return runs


@pytest.mark.parametrize("f", [0.99, 0.95, 0.9])
def test_on_off_bench_units_fine_grid(ctx, monkeypatch, f):
    tests, refs, cents = bench_units(4)
    (_, _, i0), (_, _, i1) = on_vs_off(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(0.01, 20.0)], f)
    assert i1["eb_pairs"] < i0["eb_pairs"]
    print(f"f = {f}: pairs per candidate {i1['eb_pairs'] / i1['eb_candidates']:.0f} (off: "
          f"{i0['eb_pairs'] / i0['eb_candidates']:.0f})")


@pytest.mark.parametrize("mode,f", [(0, 0.95), (1, 0.9), (0, 0.5)])
def test_on_off_mixed_shapes(ctx, monkeypatch, mode, f):
    tests, refs, cents = mixed_shapes(210 + mode)
    if f == 0.5:   # q(520) = 260 > 255: keep the sets that fit
        tests, refs, cents = tests[1:], refs[1:], cents[1:]
    on_vs_off(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(1.0, 180.0)], f, mode=mode)


def test_on_off_tiny_sets_every_q():
    """n = 6 with q from 0 to 5 (f = 1 / 6 ... 0.99)."""
    c = nat.Context(0)
    mp = pytest.MonkeyPatch()
    try:
        rng = np.random.default_rng(215)
        tests, refs = [rng.normal(0, 1, (6, 2)) for _ in range(3)], [rng.normal(0, 1, (6, 2)) for _ in range(3)]
        for f in (0.99, 0.8, 0.6, 0.5, 0.3, 1e-6):
            on_vs_off(c, mp, tests, refs, np.zeros((3, 2)), [nat.make_grid(2.0, 180.0)], f)
    finally:
        mp.undo()
        c.close()


def test_on_off_rigid_and_hierarchical(ctx, monkeypatch):
    tests, refs, cents = mixed_shapes(220)
    on_vs_off(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(2.0, 180.0)], 0.95,
              tgrids=[nat.make_tgrid(0.07, 2, t0=(0.03, -0.11))])
    # a hierarchical run: the fraction stays with the points across regrids, on and off agree at every stage
    rng = np.random.default_rng(221)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(520, 520)] * 4)
    outs = []
    for flag in ("0", "1"):
        monkeypatch.setenv("MMRS_EARLY_BREAK", flag)
        ctx.partial_upload(txy, toff, rxy, roff, cents, [nat.make_grid(1.0, 180.0)], mode=0, inlier_fraction=0.95,
                           keep_dist32=True)
        ctx.sweep_run()
        coarse = ctx.sweep_download()
        grids = [nat.make_grid(0.01, 2.0, center=float(a), limes_deg=180.0) for a in coarse["best_angle"]]
        ctx.sweep_regrid(grids, grid_of_unit=np.arange(4))
        ctx.sweep_run()
        fine = ctx.sweep_download()
        outs.append((coarse, fine, [ctx.dist32(u, grids[u].n_cand) for u in range(4)]))
    monkeypatch.delenv("MMRS_EARLY_BREAK")
    for f in FIELDS:
        assert np.array_equal(outs[0][0][f], outs[1][0][f]) and np.array_equal(outs[0][1][f], outs[1][1][f]), f
    same_bits(outs[0][2], outs[1][2], "hierarchical")
    # the regridded stage scores the partial cost: compare the fine winner with the oracle
    for u in range(4):
        angles, _ = ora.search_grid(0.01, 2.0, float(coarse["best_angle"][u]), 180.0)
        assert fine["best_dist"][u] == co.candidate_cost(tests[u], refs[u], cents[u], 0, angles[fine["best_idx"][u]],
                                                         (0, 0), "partial", 0.95)


def test_on_off_chunked_units_and_q255(ctx, monkeypatch):
    """2 020-point units (the reduced warps-per-CTA path) and q = 255 in both directions."""
    rng = np.random.default_rng(225)
    tests, refs, cents, *_ = make_units(rng, [(2020, 2020), (2020, 1900)])
    on_vs_off(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(0.05, 2.0)], 0.95)
    t2, r2, c2, *_ = make_units(rng, [(1275, 1275), (600, 1275)])
    f = 1.0 - 255.0 / 1275.0                      # K = ceil(f n) = 1020 -> q = 255 for n = 1275
    assert co.q_of(1275, f) == 255
    on_vs_off(ctx, monkeypatch, t2, r2, c2, [nat.make_grid(1.0, 30.0)], f)


# ---- 3. against the oracle ------------------------------------------------------------------------------------------
def check_oracle(ctx, tests, refs, cents, res, d32, grid_params, f, mode, tg=None):
    offs = np.zeros((1, 2)) if tg is None else co.offsets_of(tg)
    T = len(offs)
    for u in range(len(tests)):
        angles, _ = ora.search_grid(*grid_params)
        idx, costs = co.search(tests[u], refs[u], cents[u], mode, angles, offs, "partial", f)
        flat = costs.reshape(-1)
        assert res["best_idx"][u] == idx, (u, res["best_idx"][u], idx)
        assert res["best_angle"][u] == angles[idx // T]
        assert res["best_dist"][u] == flat[idx]
        if tg is not None:
            assert res["best_tx"][u] == offs[idx % T, 0] and res["best_ty"][u] == offs[idx % T, 1]
        assert res["n_ties"][u] == int(np.sum(flat == flat[idx]))   # tie_margin 0: equal f64 cost, another transform
        aa = np.repeat(angles, T)
        d64 = ctx.eval_exact_partial(tests[u], refs[u], cents[u], mode, aa,
                                     None if tg is None else np.tile(offs, (len(angles), 1)), inlier_fraction=f)
        assert np.array_equal(d64, flat)
        if d32[u] is not None:
            err = np.abs(d32[u].astype(np.float64) - d64)
            assert (err <= 1e-5 * d64 + 1e-12).all(), err.max()


@pytest.mark.parametrize("mode", [0, 1])
def test_against_oracle(ctx, mode):
    rng = np.random.default_rng(230 + mode)
    tests, refs, cents, *_ = make_units(rng, [(120, 130), (64, 97), (40, 40)])
    tests[2][[4, 5]] = np.nan                       # K counts the finite points
    for f in (0.95, 0.8):
        res, d32, _ = partial(ctx, tests, refs, cents, [nat.make_grid(1.0, 30.0)], f, mode=mode)
        check_oracle(ctx, tests, refs, cents, res, d32, (1.0, 30.0, None, 30.0), f, mode)
    tg = nat.make_tgrid(0.05, 1, t0=(0.02, -0.01))
    res, d32, _ = partial(ctx, tests, refs, cents, [nat.make_grid(2.0, 20.0)], 0.9, [tg], mode=mode)
    check_oracle(ctx, tests, refs, cents, res, d32, (2.0, 20.0, None, 20.0), 0.9, mode, tg)


def test_circle_ties_and_self_match(ctx):
    phi = np.linspace(0, 2 * np.pi, 90, endpoint=False)
    circ = np.stack([2.0 * np.cos(phi), 2.0 * np.sin(phi)], 1)
    g = nat.make_grid(4.0, 180.0)                   # every angle maps the circle onto itself
    res, d32, _ = partial(ctx, [circ], [circ.copy()], np.zeros((1, 2)), [g], 0.9, mode=1, tie_margin=1e-9)
    angles, _ = ora.search_grid(4.0, 180.0, None, 180.0)
    idx, costs = co.search(circ, circ, (0.0, 0.0), 1, angles, np.zeros((1, 2)), "partial", 0.9)
    assert res["best_idx"][0] == idx and res["best_dist"][0] == costs.reshape(-1)[idx]
    assert res["n_ties"][0] > 1


# ---- 4. the motivating case ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rigid", [False, True])
def test_bulge_does_not_decide_the_transform(ctx, rigid):
    tests, _, cents = bench_units(1)
    ref = tests[0].copy()
    cen = cents[0]
    g = nat.make_grid(0.5, 20.0)
    tg = nat.make_tgrid(0.05, 3) if rigid else None
    offs = co.offsets_of(tg) if rigid else np.zeros((1, 2))
    i_star, j_star = 17, (3 * 7 + 5 if rigid else 0)
    theta = nat.grid_angle(g, i_star)
    c, s = np.cos(theta), np.sin(theta)
    # test = the reference moved by the inverse of the planted transform, so (theta, t) maps it back onto ref
    x, y = ref[:, 0] - offs[j_star, 0] - cen[0], ref[:, 1] - offs[j_star, 1] - cen[1]
    test = np.stack([x * c + y * s + cen[0], -x * s + y * c + cen[1]], 1)
    k0 = 100                                          # 3 consecutive points pushed 0.5 mm outward
    for k in range(k0, k0 + 3):
        v = test[k] - test.mean(axis=0)
        test[k] += 0.5 * v / np.linalg.norm(v)
    f = 1.0 - 4.0 / len(test)                         # q >= 3 in both directions
    assert co.q_of(len(test), f) >= 3 and co.q_of(len(ref), f) >= 3
    tgs = None if tg is None else [tg]
    res, _, _ = partial(ctx, [test], [ref], cen[None], [g], f, tgs, mode=1)
    full, _, _ = partial(ctx, [test], [ref], cen[None], [g], 1.0, tgs, mode=1)
    T = len(offs)
    assert res["best_idx"][0] == i_star * T + j_star, (res["best_idx"][0], i_star * T + j_star)
    # recorded, not asserted: what the full cost picks on the same input
    print(f"planted {i_star * T + j_star}; partial -> {res['best_idx'][0]} ({res['best_dist'][0]:.4f}); "
          f"full cost -> {full['best_idx'][0]} ({full['best_dist'][0]:.4f})")


# ---- 5. the public function ------------------------------------------------------------------------------------------
def test_find_best_rigid_transform_partial_against_oracle():
    rng = np.random.default_rng(240)
    tests, refs, _, *_ = make_units(rng, [(80, 90), (64, 64)])
    out = mm.find_best_rigid_transform(tests, refs, step_rotation_deg=0.5, range_rotation_deg=10.0,
                                       step_translation=0.05, range_translation=0.05, inlier_fraction=0.95)
    offs = co.tgrid_offsets(0.0, 0.0, 0.05, 1)
    for u in range(2):
        cen = (np.cumsum(refs[u][:, 0])[-1] / len(refs[u]), np.cumsum(refs[u][:, 1])[-1] / len(refs[u]))
        a, j, tx, ty, d = co.coarse_to_fine(tests[u], refs[u], cen, 1, 0.5, 10.0, offs, "partial", 0.95)
        assert out["angle_rad"][u] == a and out["tx"][u] == tx and out["ty"][u] == ty and out["distance"][u] == d
    same = mm.find_best_rigid_transform(tests, refs, step_rotation_deg=0.5, range_rotation_deg=10.0,
                                        step_translation=0.05, range_translation=0.05)
    full = mm.find_best_rigid_transform(tests, refs, step_rotation_deg=0.5, range_rotation_deg=10.0,
                                        step_translation=0.05, range_translation=0.05, inlier_fraction=1.0)
    assert same.tobytes() == full.tobytes()


# ---- 6. errors -------------------------------------------------------------------------------------------------------
def test_error_cases(ctx):
    rng = np.random.default_rng(250)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(300, 300), (40, 40)])
    g = [nat.make_grid(1.0, 10.0)]

    def up(f, t=txy, to=toff, r=rxy, ro_=roff, **opts):
        ctx.partial_upload(t, to, r, ro_, cents, g, inlier_fraction=f, **opts)

    with pytest.raises(nat.MmrsError, match="q = 255"):
        up(1.0 - 256.0 / 300.0 - 1e-9)             # q(300) = 256
    big_t, big_toff, big_r, big_roff = (np.concatenate([txy, contour(rng, 5000)]), np.append(toff, toff[-1] + 5000),
                                        np.concatenate([rxy, contour(rng, 5000)]), np.append(roff, roff[-1] + 5000))
    with pytest.raises(nat.MmrsError, match="beyond the shared-memory staging"):
        ctx.partial_upload(big_t, big_toff, big_r, big_roff, np.concatenate([cents, [[4.5, 4.5]]]), g,
                           inlier_fraction=0.99)
    with pytest.raises(nat.MmrsError, match="prune is not supported with the partial cost"):
        up(0.9, prune=1)
    for pf in (2, 3):
        with pytest.raises(nat.MmrsError, match="prefilter 2 / 3 is not supported with the partial cost"):
            up(0.9, prefilter=pf)
    for bad in (0.0, -0.1, 1.5, float("nan"), float("inf")):
        with pytest.raises(nat.MmrsError, match="inlier_fraction"):
            up(bad)
        with pytest.raises(nat.MmrsError, match="inlier_fraction"):
            ctx.eval_exact_partial(tests[0], refs[0], cents[0], 0, [0.0], inlier_fraction=bad)
    up(0.9)                                        # the context still works after the errors
    ctx.sweep_run()
    assert (ctx.sweep_download()["best_idx"] >= 0).all()
