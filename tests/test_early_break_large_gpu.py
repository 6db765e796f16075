"""K1e (k_sweep_eb) against K1 on sets of more than 1 024 points.

A lane of K1e's direction pass tests the hint of each of its rows in one loop, keeping the rows that miss in a 32-bit
mask with one bit per group of 32 rows; a direction of more than 1 024 rows takes that loop in more than one block.
K1e admits such sets with MMRS_EARLY_BREAK=1 wherever its shared memory fits. Every candidate must run K1e and give
its FP32 distance bit for bit as K1 does."""
import numpy as np
import pytest

from multimodars import _native as nat
from tests.test_early_break_gpu import assert_identical, both, ctx  # noqa: F401  (ctx: the module fixture)
from tests.test_sweep_gpu import make_units

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("sizes", [[(1030, 1100), (1500, 700), (700, 1500)], [(1800, 1800)]], ids=["unequal", "1800"])
def test_sets_beyond_one_block(ctx, monkeypatch, sizes):  # noqa: F811
    rng = np.random.default_rng(400 + len(sizes))
    tests, refs, cents, *_ = make_units(rng, sizes)
    g = nat.make_grid(1.0, 180.0)
    info = assert_identical(both(ctx, monkeypatch, tests, refs, cents, [g]))
    assert info["eb_candidates"] == len(sizes) * g.n_cand, info
    # the early break must still skip most pairs (a pass that fell back to full scans would give ~ N M)
    per_cand = info["eb_pairs"] / info["eb_candidates"]
    print(f"{sizes}: {per_cand:.0f} pairs per candidate")
    assert per_cand < 0.1 * np.mean([n * m for n, m in sizes]), per_cand
