import sys
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / 'multimoda-rs_b200')]
sys.argv=['x','none','--no-tc']
from scripts import tc_bench as T
from multimodars import _native as nat
ctx=nat.Context(0)
T.run(ctx, 40, 2020, 0.005, 180.0, reps=2)
T.run(ctx, 40, 520, 0.01, 180.0, reps=2)
