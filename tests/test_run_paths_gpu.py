"""Every run path of mmrs_sweep_run, pinned on single-class batches (every unit of one size: C = 1 size class).

For a batch whose C size classes all have work, a run takes C + 3 launches on the dense sweep (K1, K1e, K1e-partial,
K1b), C + 5 with the tensor-core prefilter K1t, 2C + 4 with the expanded-form tier K1x and 2C + 6 with lower-bound
pruning K1p. mmrs_sweep_prefilter_info reports which tier ran, and each tier selects what the dense sweep selects."""
import numpy as np
import pytest

from multimodars import _native as nat
from tests.test_sweep_gpu import contour, make_units

pytestmark = pytest.mark.gpu

SELECTION = ("best_idx", "best_angle", "best_dist", "best_dist_f32")


@pytest.fixture(scope="module")
def ctx():
    c = nat.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def batch():
    """Four 520-point units on a 361-candidate grid: every tier qualifies for it."""
    rng = np.random.default_rng(17)
    tests, refs, cents, txy, toff, rxy, roff = make_units(rng, [(520, 520)] * 4)
    return (txy, toff, rxy, roff, cents), nat.make_grid(0.5, 90.0)


def pinned(ctx, launches):
    assert ctx.timings()["launches"] == launches
    return ctx.prefilter_info()


def test_dense_k1e(ctx, batch):
    arrays, g = batch
    ctx.sweep_batched(*arrays, [g], mode=0)
    info = pinned(ctx, 4)
    assert not info["ran"] and info["kind"] is None
    assert info["eb_candidates"] == 4 * g.n_cand


def test_dense_k1(ctx, batch, monkeypatch):
    arrays, g = batch
    eb = ctx.sweep_batched(*arrays, [g], mode=0)
    monkeypatch.setenv("MMRS_EARLY_BREAK", "0")
    k1 = ctx.sweep_batched(*arrays, [g], mode=0)
    info = pinned(ctx, 4)
    assert not info["ran"] and info["kind"] is None and info["eb_candidates"] == 0
    for f in SELECTION:
        assert np.array_equal(k1[f], eb[f]), f


@pytest.mark.parametrize("opts,launches,kind", [
    (dict(prefilter=2), 6, "tensor-core prefilter"),   # K1t
    (dict(prefilter=3), 6, "expanded-form tier"),      # K1x
    (dict(prune=1), 8, "lower-bound pruning"),         # K1p
])
def test_tier(ctx, batch, opts, launches, kind):
    arrays, g = batch
    dense = ctx.sweep_batched(*arrays, [g], mode=0)
    res = ctx.sweep_batched(*arrays, [g], mode=0, **opts)
    info = pinned(ctx, launches)
    assert info["ran"] and info["kind"] == kind
    for f in SELECTION:
        assert np.array_equal(res[f], dense[f]), f


def test_rigid(ctx, batch):
    arrays, g = batch
    ctx.rigid_sweep_batched(*arrays, [g], [nat.make_tgrid(0.01, 1)], mode=0)
    info = pinned(ctx, 4)
    assert not info["ran"] and info["kind"] is None


def test_partial(ctx, batch):
    arrays, g = batch
    ctx.partial_upload(*arrays, [g], mode=0, inlier_fraction=0.95)
    ctx.sweep_run()
    ctx.sweep_download()
    info = pinned(ctx, 4)
    assert not info["ran"] and info["kind"] is None and info["eb_candidates"] == 4 * g.n_cand


def test_oversize_unit_k1b(ctx):
    big = contour(np.random.default_rng(7), 6000)
    res = ctx.sweep_batched(big, [0, 6000], big, [0, 6000], np.zeros((1, 2)) + 4.5, [nat.make_grid(1.0, 5.0)], mode=0)
    info = pinned(ctx, 4)
    assert not info["ran"] and info["kind"] is None and info["eb_candidates"] == 0
    assert res["best_idx"][0] == 5 and res["best_dist"][0] == 0.0   # the identity rotation of a set on itself
