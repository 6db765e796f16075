"""K1e (k_sweep_eb) against K1 at set sizes on both sides of the edges of K1e's index stepping.

The warp scan of a row moves each lane 16 positions per round after its first round of 32 (a second round exists only
for more than 32 points); a lane's first tries step +1, -2, +3 from the row's hint; the rotation walks the staging
image two points per slot, with a one-point last slot for an odd register tile and a tail block for exact tiling. Every
size here must give every candidate's FP32 distance bit for bit as K1 does."""
import numpy as np
import pytest

from multimodars import _native as nat
from tests.test_early_break_gpu import assert_identical, both, ctx  # noqa: F401  (ctx: the module fixture)
from tests.test_sweep_gpu import make_units

pytestmark = pytest.mark.gpu

EDGES = (2, 3, 4, 15, 16, 17, 31, 32, 33, 47, 48, 49, 63, 64, 65)


@pytest.mark.parametrize("n", EDGES)
def test_scan_and_try_edges(ctx, monkeypatch, n):  # noqa: F811
    """n test points against reference sets on both sides of each edge, and the reverse."""
    rng = np.random.default_rng(100 + n)
    sizes = [(n, n), (n, 33), (33, n), (n, 520), (520, n)]
    tests, refs, cents, *_ = make_units(rng, sizes)
    assert_identical(both(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(0.5, 180.0)]))


def test_staging_slot_edges(ctx, monkeypatch):  # noqa: F811
    """Sizes around the register-tile and exact-tiling boundaries of the staging image (odd and even tiles, a tail
    block of 1 point: 513 and 577, of 31 points: 607, several chunks)."""
    rng = np.random.default_rng(77)
    sizes = [(95, 97), (96, 96), (97, 95), (159, 160), (161, 130), (513, 520), (543, 500), (544, 544), (545, 300),
             (575, 64), (577, 200), (607, 600), (640, 128)]
    tests, refs, cents, *_ = make_units(rng, sizes)
    assert_identical(both(ctx, monkeypatch, tests, refs, cents, [nat.make_grid(0.5, 180.0)]))
