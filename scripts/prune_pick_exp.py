"""Experiment: which 32 rows make the tightest lower bound (MMRS_LB_PICK = 0 strided, 1 alternating far/near, 2 far)."""
import sys
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / 'multimoda-rs_b200')]
import numpy as np
import bench
from multimodars import _native as nat
ctx = nat.Context(0)
txy, toff, rxy, roff, cen, U, n = bench.make_units(20261018)
Us = 100
g = nat.make_grid(0.01, 180.0)
ctx.sweep_upload(txy[:Us * n], toff[:Us + 1], rxy[:Us * n], roff[:Us + 1], cen[:Us], [g], mode=0, prune=1)
for _ in range(2):
    ctx.sweep_run(); r = ctx.sweep_download(); t = ctx.timings(); i = ctx.prefilter_info()
print(f"bench units x{Us}: total {t['total_ms']:.2f} ms, bounds {i['tc_ms']:.2f}, survivors {i['rescore_ms']:.2f}, scored {i['rescored'] / (Us * g.n_cand):.4f}", flush=True)
