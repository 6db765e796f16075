import sys, os
import tempfile
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / 'multimoda-rs_b200')]
os.environ.setdefault("MMRS_TC_TRACE", os.path.join(tempfile.gettempdir(), "mmrs_tc_trace.txt"))   # per-tile clock stamps of CTA 0
import numpy as np
from multimodars import _native as nat
from scripts.quick_bench import contour
ctx=nat.Context(0)
rng=np.random.default_rng(0); U=4; N=520
t=np.concatenate([contour(rng,N,rng.normal(0,.2)) for _ in range(U)]); r=np.concatenate([contour(rng,N) for _ in range(U)])
off=np.arange(U+1)*N; g=nat.make_grid(0.05,180.0)
ctx.sweep_upload(t,off,r,off,np.full((U,2),4.5),[g],mode=0,prefilter=2)
ctx.sweep_run(); ctx.sweep_download(); print(ctx.timings(), ctx.prefilter_info())
