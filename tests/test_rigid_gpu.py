"""Rigid candidates (angle grid x translation grid, include/mmrs_b200.h "rigid candidates") on the GPU.

1. A zero translation grid is the rotation-only sweep, field for field and dist32 bit for bit, under K1 and K1e.
2. K1e equals K1 on rigid runs, dist32 bit for bit.
3. Results against the f64 restatement in tests/cost_oracle.py; every FP32 distance within 1e-5 relative of
   mmrs_eval_exact_rigid.
4. A known transform is recovered exactly. 5. Ties. 6. find_best_rigid_transform against the oracle's
   coarse-to-fine. 7. Error cases."""
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


@pytest.fixture(scope="module")
def ctx():
    c = nat.Context(0)
    yield c
    c.close()


def _d32(ctx, tests, refs, n_cand):
    return [ctx.dist32(u, int(n_cand[u])) if len(tests[u]) and len(refs[u]) else None for u in range(len(tests))]


def rigid(ctx, tests, refs, cents, grids, tgrids, gou=None, tou=None, mode=0, **opts):
    txy, toff, rxy, roff = pack(tests, refs)
    res = ctx.rigid_sweep_batched(txy, toff, rxy, roff, cents, grids, tgrids, grid_of_unit=gou, tgrid_of_unit=tou,
                                  mode=mode, keep_dist32=True, **opts)
    U = len(tests)
    gi = np.zeros(U, int) if gou is None else np.asarray(gou)
    ti = np.zeros(U, int) if tou is None else np.asarray(tou)
    n_cand = [0 if grids[gi[u]].degenerate else grids[gi[u]].n_cand * (2 * tgrids[ti[u]].half_n + 1) ** 2
              for u in range(U)]
    return res, _d32(ctx, tests, refs, n_cand), ctx.prefilter_info()


# ---- 1. zero translation == the rotation-only sweep -------------------------------------------------------------
def zero_vs_rotation(ctx, monkeypatch, tests, refs, cents, grids, gou=None, mode=0):
    txy, toff, rxy, roff = pack(tests, refs)
    z = nat.make_tgrid(0.0, 0)
    for flag in ("0", "1"):
        monkeypatch.setenv("MMRS_EARLY_BREAK", flag)
        r0 = ctx.sweep_batched(txy, toff, rxy, roff, cents, grids, grid_of_unit=gou, mode=mode, keep_dist32=True)
        n_cand = [grids[0 if gou is None else gou[u]].n_cand for u in range(len(tests))]
        d0 = _d32(ctx, tests, refs, n_cand)
        r1, d1, _ = rigid(ctx, tests, refs, cents, grids, [z], gou=gou, mode=mode)
        for f in FIELDS:
            assert np.array_equal(r0[f], r1[f]), (flag, f, r0[f], r1[f])
        assert (r1["trans_idx"][r1["best_idx"] >= 0] == 0).all()
        assert (r1["best_tx"] == 0.0).all() and (r1["best_ty"] == 0.0).all()
        same_bits(d0, d1, f"MMRS_EARLY_BREAK={flag}")
    monkeypatch.delenv("MMRS_EARLY_BREAK")


def test_zero_translation_bench_units(ctx, monkeypatch):
    txy, toff, rxy, roff, cen, U, n = bench.make_units()
    pick = np.linspace(0, U - 1, 16).astype(int)
    tests = [txy[toff[u]:toff[u + 1]] for u in pick]
    refs = [rxy[roff[u]:roff[u + 1]] for u in pick]
    zero_vs_rotation(ctx, monkeypatch, tests, refs, cen[pick], [nat.make_grid(bench.STEP_DEG, bench.RANGE_DEG)])


@pytest.mark.parametrize("mode", [0, 1])
def test_zero_translation_modes_and_classes(ctx, monkeypatch, mode):
    """mode 0 / 1; an exact-tiling class (N = 520), odd register tiles, and small sets."""
    rng = np.random.default_rng(70 + mode)
    tests, refs, cents, *_ = make_units(rng, [(520, 520), (300, 411), (97, 250), (6, 6)])
    zero_vs_rotation(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(0.05, 180.0)], mode=mode)


def test_zero_translation_chunked_and_oversize(ctx, monkeypatch):
    """A chunked K1 class (N = M = 2 020) and an oversize K1b unit (N = M = 5 000, 41 angles)."""
    rng = np.random.default_rng(77)
    tests, refs, cents, *_ = make_units(rng, [(2020, 2020), (5000, 5000)])
    zero_vs_rotation(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(1.0, 20.0)])


def test_zero_translation_hierarchical_regrid(ctx):
    rng = np.random.default_rng(78)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(520, 520)] * 4)
    z = nat.make_tgrid(0.0, 0)
    ctx.sweep_upload(txy, toff, rxy, roff, cents, [nat.make_grid(1.0, 180.0)], mode=0)
    ctx.sweep_run()
    coarse = ctx.sweep_download()
    grids = [nat.make_grid(0.01, 2.0, center=float(c), limes_deg=180.0) for c in coarse["best_angle"]]
    ctx.sweep_regrid(grids, grid_of_unit=np.arange(4))
    ctx.sweep_run()
    want = ctx.sweep_download()
    ctx.rigid_upload(txy, toff, rxy, roff, cents, [nat.make_grid(1.0, 180.0)], [z], mode=0)
    ctx.sweep_run()
    rc = ctx.rigid_download()
    assert np.array_equal(rc["best_idx"], coarse["best_idx"]) and np.array_equal(rc["best_dist"], coarse["best_dist"])
    ctx.rigid_regrid(grids, [z], grid_of_unit=np.arange(4))
    ctx.sweep_run()
    got = ctx.rigid_download()
    for f in FIELDS:
        assert np.array_equal(want[f], got[f]), f


# ---- 2. K1e == K1 on rigid runs ------------------------------------------------------------------------------------
def k1_vs_k1e(ctx, monkeypatch, tests, refs, cents, grids, tgrids, mode=0):
    runs = []
    for flag in ("0", "1"):
        monkeypatch.setenv("MMRS_EARLY_BREAK", flag)
        runs.append(rigid(ctx, tests, refs, cents, grids, tgrids, mode=mode))
    monkeypatch.delenv("MMRS_EARLY_BREAK")
    (r0, d0, i0), (r1, d1, i1) = runs
    assert i0["eb_candidates"] == 0 and i1["eb_candidates"] > 0
    same_bits(d0, d1, "K1 vs K1e")
    for f in RIGID_FIELDS:
        assert np.array_equal(r0[f], r1[f]), f
    return runs


RIGID_FIELDS = FIELDS + ("angle_idx", "trans_idx", "best_tx", "best_ty")


@pytest.mark.parametrize("half_n", [1, 3, 5])
def test_k1e_equals_k1_rigid(ctx, monkeypatch, half_n):
    rng = np.random.default_rng(80 + half_n)
    tests, refs, cents, *_ = make_units(rng, [(520, 520), (400, 333), (130, 64)])
    tests.append(rng.normal(0, 1.0, (300, 2)))                                  # random clouds, N != M
    refs.append(rng.normal(0, 1.2, (211, 2)))
    phi = np.linspace(0, 2 * np.pi, 360, endpoint=False)
    circ = np.stack([2.0 * np.cos(phi), 2.0 * np.sin(phi)], 1)
    tests += [circ, np.repeat(rng.normal(0, 1, (2, 2)), 3, axis=0), rng.normal(0, 1, (5, 2))]   # circle, duplicated, tiny
    refs += [circ.copy(), np.concatenate([refs[0][:3], refs[0][:3]]) - 4.5, rng.normal(0, 1, (1, 2))]
    nf_t, nf_r = contour(rng, 200), contour(rng, 180)                           # non-finite points
    nf_t[[3, 50]] = np.nan
    nf_r[7] = np.inf
    tests.append(nf_t)
    refs.append(nf_r)
    cents = np.concatenate([cents, np.zeros((4, 2)), [[4.5, 4.5]]])
    tg = nat.make_tgrid(0.07, half_n, t0=(0.03, -0.11))
    k1_vs_k1e(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(1.0, 180.0)], [tg])


# ---- 3. against the oracle -----------------------------------------------------------------------------------------
def check_oracle(ctx, tests, refs, cents, res, d32, grid_params, tg, mode):
    offs = co.offsets_of(tg)
    worst = 0.0
    for u in range(len(tests)):
        angles, fb = ora.search_grid(*grid_params)
        idx, costs = co.search(tests[u], refs[u], cents[u], mode, angles, offs, "full")
        T = len(offs)
        assert res["best_idx"][u] == idx
        assert res["angle_idx"][u] == idx // T and res["trans_idx"][u] == idx % T
        assert res["best_angle"][u] == angles[idx // T]
        assert res["best_tx"][u] == offs[idx % T, 0] and res["best_ty"][u] == offs[idx % T, 1]
        assert res["best_dist"][u] == costs.reshape(-1)[idx]
        if d32[u] is None:
            continue
        aa = np.repeat(angles, T)
        tt = np.tile(offs, (len(angles), 1))
        d64 = ctx.eval_exact_rigid(tests[u], refs[u], cents[u], mode, aa, tt)
        assert np.array_equal(d64, costs.reshape(-1))
        err = np.abs(d32[u].astype(np.float64) - d64)
        assert (err <= 1e-5 * d64 + 1e-12).all(), err.max()
        pts = np.concatenate([tests[u], refs[u]]) - cents[u]
        r_eff = np.abs(pts).max() + np.hypot(offs[:, 0], offs[:, 1]).max()
        worst = max(worst, float((err / r_eff).max()))
    print(f"largest |d32 - d64| / R_eff: {worst:.3e}")
    return worst


@pytest.mark.parametrize("mode", [0, 1])
def test_against_oracle(ctx, mode):
    rng = np.random.default_rng(90 + mode)
    tests, refs, cents, *_ = make_units(rng, [(120, 130), (64, 97), (40, 40)])
    tg = nat.make_tgrid(0.05, 2, t0=(0.02, -0.01))
    res, d32, _ = rigid(ctx, tests, refs, cents, [nat.make_grid(1.0, 30.0)], [tg], mode=mode)
    check_oracle(ctx, tests, refs, cents, res, d32, (1.0, 30.0, None, 30.0), tg, mode)


def test_empty_set_and_degenerate_grid(ctx):
    rng = np.random.default_rng(95)
    tests, refs, cents, *_ = make_units(rng, [(50, 60), (0, 40), (50, 60)])
    tg = nat.make_tgrid(0.1, 1, t0=(0.5, -0.25))
    grids = [nat.make_grid(2.0, 10.0), nat.make_grid(0.0, 10.0, center=0.3)]
    res, d32, _ = rigid(ctx, tests, refs, cents, grids, [tg], gou=np.array([0, 0, 1], np.int32))
    assert res["best_idx"][1] == 0 and res["best_dist"][1] == 0.0 and res["flags"][1] & nat.FLAG_EMPTY
    offs = co.offsets_of(tg)
    assert res["trans_idx"][1] == 0 and res["best_tx"][1] == offs[0, 0] and res["best_ty"][1] == offs[0, 1]
    assert res["best_idx"][2] == -1 and res["best_angle"][2] == 0.3 and res["flags"][2] & nat.FLAG_DEGENERATE
    assert res["angle_idx"][2] == -1 and res["trans_idx"][2] == -1
    assert res["best_tx"][2] == 0.5 and res["best_ty"][2] == -0.25
    check_oracle(ctx, tests[:1], refs[:1], cents[:1], res[:1], d32[:1], (2.0, 10.0, None, 10.0), tg, 0)


# ---- 4. known answer -----------------------------------------------------------------------------------------------
def test_known_transform_is_recovered(ctx):
    rng = np.random.default_rng(97)
    test = contour(rng, 300, noise=0.0)
    cen = np.array([4.5, 4.5])
    g = nat.make_grid(1.0, 30.0)
    tg = nat.make_tgrid(0.05, 5)
    offs = co.offsets_of(tg)
    i_star, j_star = 37, 7 * 11 + 2
    theta = nat.grid_angle(g, i_star)
    c, s = np.cos(theta), np.sin(theta)
    x, y = test[:, 0] - cen[0], test[:, 1] - cen[1]
    ref = np.stack([x * c - y * s + cen[0] + offs[j_star, 0], x * s + y * c + cen[1] + offs[j_star, 1]], 1)
    res, _, _ = rigid(ctx, [test], [ref], cen[None], [g], [tg], mode=1)
    assert res["angle_idx"][0] == i_star and res["trans_idx"][0] == j_star
    assert res["best_dist"][0] <= 1e-12 * np.abs(ref - cen).max()
    rot = ctx.sweep_batched(test, [0, len(test)], ref, [0, len(ref)], cen[None], [g], mode=1)
    assert rot["best_dist"][0] > res["best_dist"][0]


# ---- 5. ties -------------------------------------------------------------------------------------------------------
def test_circle_ties_pick_the_lowest_flattened_index(ctx):
    phi = np.linspace(0, 2 * np.pi, 90, endpoint=False)
    circ = np.stack([2.0 * np.cos(phi), 2.0 * np.sin(phi)], 1)
    g = nat.make_grid(4.0, 180.0)           # multiples of the 4 deg point spacing: every angle maps the circle onto itself
    tg = nat.make_tgrid(0.1, 1)
    res, _, _ = rigid(ctx, [circ], [circ.copy()], np.zeros((1, 2)), [g], [tg], mode=1, tie_margin=1e-9)
    angles, _ = ora.search_grid(4.0, 180.0, None, 180.0)
    idx, costs = co.search(circ, circ, (0.0, 0.0), 1, angles, co.offsets_of(tg), "full")
    assert res["best_idx"][0] == idx
    best = costs.reshape(-1)[idx]
    flat = costs.reshape(-1)
    T = 9
    lim = best + 1e-9 * max(1.0, 2.0 + 0.1 * np.sqrt(2))
    cs = np.array([[np.cos(a), np.sin(a)] for a in angles])
    offs = co.offsets_of(tg)
    want = 1 + sum(1 for c in range(len(flat)) if c != idx and flat[c] <= lim and
                   (not np.array_equal(cs[c // T], cs[idx // T]) or not np.array_equal(offs[c % T], offs[idx % T])))
    assert want > 1
    assert res["n_ties"][0] == want
    assert res["trans_idx"][0] == 4                     # the zero translation: every other one is strictly worse


# ---- 6. the public function ------------------------------------------------------------------------------------
@pytest.mark.parametrize("bruteforce", [False, True])
def test_find_best_rigid_transform_against_oracle(bruteforce):
    rng = np.random.default_rng(101)
    tests, refs, _, *_ = make_units(rng, [(80, 90), (64, 64)])
    step, rng_deg = (2.0, 20.0) if bruteforce else (0.5, 20.0)
    out = mm.find_best_rigid_transform(tests, refs, step_rotation_deg=step, range_rotation_deg=rng_deg,
                                       step_translation=0.05, range_translation=0.1, bruteforce=bruteforce)
    offs = co.tgrid_offsets(0.0, 0.0, 0.05, 2)
    for u in range(2):
        cen = (np.cumsum(refs[u][:, 0])[-1] / len(refs[u]), np.cumsum(refs[u][:, 1])[-1] / len(refs[u]))
        a, j, tx, ty, d = co.coarse_to_fine(tests[u], refs[u], cen, 1, step, rng_deg, offs, "full",
                                            bruteforce=bruteforce)
        assert out["angle_rad"][u] == a and out["tx"][u] == tx and out["ty"][u] == ty and out["distance"][u] == d


def test_zero_translation_range_is_find_best_rotation():
    rng = np.random.default_rng(103)
    tests, refs, _, *_ = make_units(rng, [(100, 110)])
    out = mm.find_best_rigid_transform(tests[0], refs[0], step_rotation_deg=0.05, range_rotation_deg=30.0,
                                       step_translation=0.05, range_translation=0.0)
    want = ora.find_best_rotation(tests[0], refs[0], (0.0, 0.0), 1, 0.05, 30.0)
    assert out["angle_rad"][0] == want and out["tx"][0] == 0.0 and out["ty"][0] == 0.0
    cen = (np.cumsum(refs[0][:, 0])[-1] / 110, np.cumsum(refs[0][:, 1])[-1] / 110)
    assert out["distance"][0] == ora.costs(tests[0], refs[0], cen, 1, [want])[0]


# ---- 7. errors -----------------------------------------------------------------------------------------------------
def test_error_cases(ctx):
    rng = np.random.default_rng(107)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(40, 40), (30, 30)])
    g = nat.make_grid(1.0, 10.0)
    ok = nat.make_tgrid(0.05, 1)

    def run(tgrids, tou=None, grids=(g,), **opts):
        return ctx.rigid_sweep_batched(txy, toff, rxy, roff, cents, list(grids), tgrids, tgrid_of_unit=tou, **opts)

    with pytest.raises(nat.MmrsError, match="exceed INT32_MAX"):
        run([nat.make_tgrid(1e-6, 3000)], grids=(nat.make_grid(1.0, 180.0),))
    with pytest.raises(nat.MmrsError, match="tgrid_of_unit out of range"):
        run([ok], tou=np.array([0, 1], np.int32))
    with pytest.raises(nat.MmrsError, match="half_n must be >= 0"):
        run([nat.make_tgrid(0.05, -1)])
    with pytest.raises(nat.MmrsError, match="step must be > 0"):
        run([nat.make_tgrid(0.0, 2)])
    with pytest.raises(nat.MmrsError, match="must be finite"):
        run([nat.make_tgrid(0.05, 1, t0=(np.nan, 0.0))])
    with pytest.raises(nat.MmrsError, match="prune is not supported with a translation grid"):
        run([ok], prune=1)
    for pf in (2, 3):
        with pytest.raises(nat.MmrsError, match="not supported with a translation grid"):
            run([ok], prefilter=pf)
    res = run([ok])                                        # the context still works after the errors
    assert (res["best_idx"] >= 0).all()


def test_shard_transport_is_not_used(ctx):
    rng = np.random.default_rng(109)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(200, 200)] * 4)
    tg = nat.make_tgrid(0.05, 2)
    g = nat.make_grid(1.0, 180.0)
    want = ctx.rigid_sweep_batched(txy, toff, rxy, roff, cents, [g], [tg])
    calls = []
    c2 = nat.Context(0)
    try:
        c2.set_shard(1, 2, lambda buf: calls.append(len(buf)))
        c2.set_prune(True)
        got = c2.rigid_sweep_batched(txy, toff, rxy, roff, cents, [g], [tg])
    finally:
        c2.close()
    assert calls == []
    for f in RIGID_FIELDS:
        assert np.array_equal(want[f], got[f]), f
