#!/usr/bin/env python
"""bench.py — Hausdorff candidate evaluations / second on B200 (BASELINE.json metric).

Workload (config.workload), the SAME at every --gpus N (strong scaling): 8 pullback pairs of BASELINE.json
configs[1] ("synthetic single-pair: 1 pullback pair, 200 frames x 500 points/contour, 0.01 deg rotation sweep over
360 deg") = 3 184 intrapullback frame-pair units (N = M = 520 points: 500 lumen + 20 catheter), 36 000 candidate
angles each, brute force. One "step" = one pass of the hot path over that batch.

  value  evals/s with the batch resident in HBM (mmrs_sweep_run + mmrs_sweep_download: FP32 sweep + shortlist + f64
         recheck + arg-min, results on the host), CUDA events on the launching stream, max over ranks.
  e2e    the same through the C-ABI call a host binds (mmrs_sweep_batched) with HOST buffers: pinned H2D of the
         points, all kernels, D2H of the per-unit results, every step.
  N > 1  ONE batch partitioned across the ranks by the library itself (mmrs_ctx_comm_init, axis 1: cost-balanced
         blocks of whole units): every rank issues the same calls with the same batch, its GPU sweeps only its
         block, and the 32-byte per-unit results are merged by one NCCL all-reduce on device buffers on the
         context's stream inside the timed region. Every rank ends up with all 3 184 results; the run FAILS unless
         all ranks agree bit for bit and equal the committed 1-GPU result (tests/golden/bench_units.npz). The
         candidate-axis partition (axis 2) is checked in the same run on 72 000-candidate units.
  full_mode  wall time of the public full-mode entry points (the second half of BASELINE.json's metric).

`--impl reference` times the CPU oracle (oracle/, the restatement of the reference's rayon path; the Rust reference
cannot be built in this image) on the host cores, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path[:0] = [str(ROOT), str(ROOT / "multimoda-rs_b200")]

METRIC = "hausdorff_candidate_evals_per_sec"
UNIT = "evals/s"
N_PAIRS = 8
N_FRAMES, N_POINTS, N_CATH = 200, 500, 20
STEP_DEG, RANGE_DEG = 0.01, 180.0
SEED = 20261018
WORKLOAD = (f"{N_PAIRS} x BASELINE configs[1] (synthetic single-pair: 2 pullbacks x 200 frames x 500 pts + 20 catheter pts, "
            "brute-force 0.01 deg sweep over +-180 deg = 36000 candidates): 3184 frame-pair units, the same batch at every "
            "N (strong scaling)")
GOLDEN = ROOT / "tests" / "golden" / "bench_units.npz"


def flops_per_eval(n, m):
    """SURVEY.md §8(d): two directed passes x N*M pairs x 5 FP32 FLOPs + 6 N for the rotation."""
    return 10.0 * n * m + 6.0 * n


# ---- synthetic pullback pair -> sweep units (what align_within_many builds on the host) -------------
def synthetic_pullback(n_frames, n_points, seed):
    """SURVEY.md §8(d) generator: smooth random-walk lumen shape, cumulative rotation N(0, 4 deg),
    centroid jitter 0.3 mm about (4.5, 4.5), 5 um point noise. Returns (frames, n_points, 2)."""
    rng = np.random.default_rng(seed)
    phi = np.linspace(0.0, 2.0 * np.pi, n_points, endpoint=False)
    r0, e, psi = rng.uniform(1.5, 3.0), rng.uniform(0.05, 0.35), rng.uniform(0, np.pi)
    ak, pk = rng.uniform(0, 0.04, 4), rng.uniform(0, 2 * np.pi, 4)
    cum, out = 0.0, []
    for _ in range(n_frames):
        r0 = float(np.clip(r0 + rng.normal(0, 0.02), 1.2, 3.2))
        e = float(np.clip(e + rng.normal(0, 0.01), 0.03, 0.4))
        ak = np.clip(ak + rng.normal(0, 0.002, 4), 0, 0.05)
        cum += np.deg2rad(rng.normal(0, 4.0))
        r = r0 * (1 + e * np.cos(2 * (phi - psi)) + sum(ak[k] * np.cos((k + 3) * phi + pk[k]) for k in range(4)))
        c = 4.5 + rng.normal(0, 0.3, 2)
        out.append(np.stack([r * np.cos(phi + cum) + c[0], r * np.sin(phi + cum) + c[1]], 1)
                   + rng.normal(0, 0.005, (n_points, 2)))
    return np.stack(out)


def make_units(seed=SEED, n_pairs=N_PAIRS):
    """The decoupled frame-pair units of `n_pairs` pullback pairs (398 each), centred like the host does. Pair p uses
    the seeds seed + 1000 p (+0, +1): pair 0 is the round-1 single-pair workload."""
    th = 2.0 * np.pi * np.arange(N_CATH) / N_CATH
    cath = np.stack([4.5 + 0.5 * np.cos(th), 4.5 + 0.5 * np.sin(th)], 1)
    tests, refs = [], []
    for p in range(n_pairs):
        for pb in range(2):
            fr = synthetic_pullback(N_FRAMES, N_POINTS, seed + 1000 * p + pb)
            pts = [np.concatenate([f, cath]) - f.mean(axis=0) for f in fr]   # centred on the frame (lumen) centroid
            for i in range(1, N_FRAMES):
                tests.append(pts[i])
                refs.append(pts[i - 1])
    U = len(tests)
    n = N_POINTS + N_CATH
    off = np.arange(U + 1, dtype=np.int64) * n
    return np.concatenate(tests), off, np.concatenate(refs), off.copy(), np.zeros((U, 2)), U, n


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def dump_outputs(out_dir, fields):
    """One DIR/<name>.npy per result field: float32 fields stay float32, every other field (indices and counts included,
    all exact below 2^53) is written as float64."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in fields.items():
        np.save(d / f"{name}.npy", np.asarray(a, dtype=np.float32 if a.dtype == np.float32 else np.float64))


# ---- clocks ----------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].startswith("Active")})
        # median over the busiest half (the samples taken while kernels were running)
        busy = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    sm_max = 1965.0
    src = "fallback sm_max_mhz 1965 (B200_PROFILING.md)"
    if p.exists():
        try:
            sm_max = float(json.loads(p.read_text())["sm_max_mhz"])
            src = "MEASURED_PEAKS.json sm_max_mhz"
        except Exception:
            pass
    return 148 * 128 * 2 * sm_max * 1e6 / 1e12, src


def base_config(U, ncand, n, world):
    return {"workload": WORKLOAD, "units": U, "candidates_per_unit": ncand, "points": [n, n],
            "parallelism": (f"ONE batch, whole units partitioned x{world} by the library (mmrs_ctx_comm_init, axis 1); "
                            "NCCL all-reduce of the 32-byte per-unit results on device buffers") if world > 1
            else "1 GPU",
            "l2": "256 MB device buffer rewritten between timed iterations", "recheck": "f64 on-device"}


# ---- reference arm: the CPU oracle on the host cores -------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle_py as ora

    ora.build()
    cores = os.cpu_count() or 1
    txy, toff, rxy, roff, cen, U, n = make_units(n_pairs=1)
    sample_units = 1
    sl = slice(0, sample_units * n)
    t_off, r_off = toff[:sample_units + 1], roff[:sample_units + 1]
    ncand = len(ora.search_grid(STEP_DEG, RANGE_DEG, None, RANGE_DEG)[0])

    last = {}

    def step():
        t0 = time.perf_counter()
        last["best_idx"], last["best_dist"] = ora.sweep_batch(txy[sl], t_off, rxy[sl], r_off, cen[:sample_units], 0, STEP_DEG,
                                                              RANGE_DEG, RANGE_DEG, threads=cores)
        return time.perf_counter() - t0

    for _ in range(min(args.warmup, 1)):
        step()
    times = [step() for _ in range(args.steps)]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    evals = sample_units * ncand
    v = evals * len(times) / sum(times)
    sample = (f"per step {sample_units} of the {398 * N_PAIRS} frame-pair units x {ncand} candidates (N=M={n}), {cores} host "
              f"threads over candidates; the units are homogeneous, so the rate carries over to the whole batch")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            # the SAME config object as our arm prints for this N (the workload both arms are quoted on); how the CPU arm
            # runs it — host threads, the bounded sample — is in cpu_baseline
            "config": base_config(398 * N_PAIRS, ncand, n, max(args.gpus, 1)),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "parallelism": f"{cores} host threads (CPU), f64 throughout"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "CPU oracle = C++ f64 restatement of the reference's rayon path (threads over candidate angles, "
                    "serial N x M inside; process_utils.rs:69-118); the Rust reference cannot be built in this image"}
    print(json.dumps(line), flush=True)


# ---- our arm --------------------------------------------------------------------------------------------
_T0 = time.perf_counter()


def progress(rank, msg):
    """Where the run is, on stderr (rank 0): a stuck N-rank run must say which leg it is in."""
    if rank == 0:
        print(f"[bench +{time.perf_counter() - _T0:6.1f} s] {msg}", file=sys.stderr, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-api", action="store_true", help="skip the public-API wall-time legs (e2e_api, full_mode)")
    ap.add_argument("--no-tc", action="store_true", help="skip the opt-in tier legs (tensor-core prefilter, pruning)")
    ap.add_argument("--write-golden", action="store_true", help="N = 1 only: (re)write tests/golden/bench_units.npz")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the per-unit results of the last timed step as DIR/<field>.npy, so that two builds can be "
                         "compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
        return

    # ONE JSON line on stdout: everything any library prints while we run (NCCL's version banner is written to fd 1
    # by the C library) goes to stderr; the saved descriptor is restored just before the line is printed.
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    from multimodars import _dist
    from multimodars import _native as nat

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local)
    stream = torch.cuda.current_stream()
    ctx = nat.Context(local, stream.cuda_stream)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep NCCL's banner off stdout: ONE JSON line there
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        _dist.init_comm(ctx, axis=1)   # the library's own NCCL communicator: sweeps are partitioned from here on
    W = max(args.warmup, 3)
    K = args.steps

    txy, toff, rxy, roff, cen, U, n = make_units()
    grid = nat.make_grid(STEP_DEG, RANGE_DEG)
    ncand = int(grid.n_cand)
    evals = U * ncand
    F = flops_per_eval(n, n)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    progress(rank, f"workload built: {U} units x {ncand} candidates")
    # ---- value: batch resident in HBM ------------------------------------------------------------------
    ctx.sweep_upload(txy, toff, rxy, roff, cen, [grid], mode=0, prefilter=1, prune=-1)   # the dense FP32 sweep
    plan = ctx.plan()
    for _ in range(W):
        ctx.sweep_run()
        ctx.sweep_download()
    clocks = ClockSampler(local)
    barrier()
    clocks.start()
    dev_ms, k1_ms, launches = [], [], 0
    for _ in range(K):
        flush.fill_(1)                      # L2 flush between timed iterations
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ctx.sweep_run()                     # N > 1: ends with the NCCL all-reduce of the per-unit results
        res = ctx.sweep_download()          # D2H of 32 B per unit (stream sync inside)
        e1.record(stream)
        e1.synchronize()
        dev_ms.append(e0.elapsed_time(e1))
        t = ctx.timings()
        k1_ms.append(t["sweep_ms"])
        launches += t["launches"]
    barrier()
    clk = clocks.stop()
    total_ms = max_over_ranks(sum(dev_ms))
    value = evals * K / (total_ms * 1e-3)
    if args.dump_outputs and rank == 0:   # every rank holds the whole merged result
        dump_outputs(args.dump_outputs, {f: res[f] for f in res.dtype.names})

    # ---- every rank holds the whole result: identical across ranks, equal to the committed 1-GPU result -------------
    digest = sha(np.stack([res["best_idx"].astype(np.float64), res["best_angle"], res["best_dist"],
                           res["n_ties"].astype(np.float64)], 1))
    check = {"result_sha256": digest, "all_ranks_identical": True, "equals_1gpu_golden": None}
    if world > 1:
        box = [None] * world
        dist.all_gather_object(box, digest)
        check["all_ranks_identical"] = len(set(box)) == 1
    if args.write_golden and world == 1:
        np.savez_compressed(GOLDEN, best_idx=res["best_idx"], best_dist=res["best_dist"], seed=SEED, n_pairs=N_PAIRS,
                            note="bench.py --write-golden on 1 B200: leftmost f64 arg-min and its f64 Hausdorff distance of "
                                 "every unit of the bench workload (units 0..3 checked against the CPU oracle by "
                                 "tests/test_bench_golden_gpu.py)")
    if GOLDEN.exists():
        g = np.load(GOLDEN)
        check["equals_1gpu_golden"] = bool(np.array_equal(g["best_idx"], res["best_idx"])
                                           and np.array_equal(g["best_dist"], res["best_dist"]))
    ok_partition = check["all_ranks_identical"] and check["equals_1gpu_golden"] is not False

    progress(rank, f"value leg done: {value:.4g} evals/s")
    # ---- e2e: C ABI call with host buffers (pinned), H2D + kernels + D2H every step ------------------------
    pin = [torch.from_numpy(a).pin_memory() for a in (txy, rxy)]
    h_t, h_r = pin[0].numpy(), pin[1].numpy()
    ctx.sweep_batched(h_t, toff, h_r, roff, cen, [grid], mode=0, prefilter=1, prune=-1)
    barrier()
    e2e_ms = []
    for _ in range(K):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        res_e = ctx.sweep_batched(h_t, toff, h_r, roff, cen, [grid], mode=0, prefilter=1, prune=-1)
        e1.record(stream)
        e1.synchronize()
        e2e_ms.append(e0.elapsed_time(e1))
    barrier()
    e2e_value = evals * K / (max_over_ranks(sum(e2e_ms)) * 1e-3)
    ok_partition = ok_partition and bool(np.array_equal(res_e["best_idx"], res["best_idx"]))
    h2d = txy.nbytes + rxy.nbytes + toff.nbytes + roff.nbytes + cen.nbytes + ncand * 17 + U * 96
    d2h = U * 32

    # ---- roofline of the dominant kernel (k_sweep) ------------------------------------------------------------
    peak, peak_src = peaks()
    k1 = float(np.mean(k1_ms))
    units_here = U / world   # cost-balanced blocks of identical units
    achieved = units_here * ncand * F / (k1 * 1e-3) / 1e12
    probe = ctx.fp32_probe(4096)
    traffic, traffic_src = None, None
    tp = ROOT / "profiles" / "sweep_traffic.json"
    if tp.exists():
        try:
            tj = json.loads(tp.read_text())
            per_unit = tj.get("dram_bytes_per_unit")
            traffic = per_unit * units_here if per_unit else None
            traffic_src = {"file": "profiles/sweep_traffic.json", "sha256": hashlib.sha256(tp.read_bytes()).hexdigest()[:16],
                           "ncu_report": tj.get("source"), "kernel": tj.get("kernel"),
                           "note": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this kernel, "
                                   "scaled by units per launch (not measurable inside an unprofiled run)"}
        except Exception:
            traffic = None
    slots = 32 * plan["TA"] * (1 if not plan["multi"] else -(-n // (32 * plan["TA"])))
    exec_flops = 5.0 * n * slots + 6.0 * slots + (5.0 * (n - slots) * 32 * (plan["TA"] + 1) if plan["exact_tiling"] else 0.0)
    kname = f"k_sweep<{plan['TA']},{str(plan['multi']).lower()},false,{str(plan['exact_tiling']).lower()}>"
    roofline = {"bound": "fp32", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "frac_executed": achieved / peak * exec_flops / F,
                "traffic": traffic, "traffic_source": traffic_src, "kernel": kname, "kernel_ms": k1,
                "kernel_share_of_step": k1 / float(np.mean(dev_ms)),
                "peak_source": f"148 SM x 128 FP32 lanes x 2 x {peak_src} (no FP32 figure in MEASURED_PEAKS.json)",
                "ffma_probe_tflops": probe, "frac_of_ffma_probe": achieved / probe,
                # north star: "plus HBM GB/s for the point streams" — DRAM traffic of the launch over its duration (the
                # staging images are read once per CTA and mostly hit L2; dist32 stays in L2): HBM is idle on this path
                "hbm_gbps": (traffic / (k1 * 1e-3) / 1e9) if traffic else None,
                "algorithmic_flops_per_eval": F, "executed_flops_per_eval": exec_flops,
                "note": "frac counts the reference's arithmetic (10 N M + 6 N per evaluation, SURVEY §8d); the kernel computes "
                        "each pair distance once for both directed passes, so it EXECUTES about half of that: frac_executed"}

    def head_line():
        return {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": base_config(U, ncand, n, world),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "call": "mmrs_sweep_batched (host buffers in, host results out); every rank uploads the whole batch"},
                "e2e_api": None,
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": None, "clocks": clk,
                "partition_check": check, "angle_axis_check": None, "full_mode": None,
                "tc_prefilter": None, "pruned": None}

    # ---- the legs reported beside the headline. They run under a watchdog: whatever happens in them (a collective that
    # never completes included), rank 0 still prints the line with the headline numbers measured above, every rank leaves,
    # and the exit code only reflects the partition check of the headline.
    state = {"angle": None, "full_mode": None, "emitted": False, "ok": ok_partition}
    lock = threading.Lock()

    def emit(extra):
        with lock:
            if state["emitted"]:
                return
            state["emitted"] = True
            if rank == 0:
                line = head_line()
                line.update({"angle_axis_check": state["angle"], "full_mode": state["full_mode"]})
                line.update(extra)
                line["e2e_api"] = (state["full_mode"] or {}).get("config2_from_array_singlepair") if isinstance(state["full_mode"], dict) else None
                try:
                    text = json.dumps(line)
                except Exception as e:  # noqa: BLE001  (the watchdog may fire while a leg is still filling its dict)
                    line["full_mode"] = {"error": f"not serialisable when the line was printed: {type(e).__name__}"}
                    line["e2e_api"] = None
                    text = json.dumps(line)
                sys.stdout.flush()
                os.dup2(saved_stdout, 1)
                print(text, flush=True)

    def bail():
        import faulthandler

        print(f"bench.py: rank {rank}: the reported-beside legs exceeded {deadline:.0f} s; printing the headline without them",
              file=sys.stderr, flush=True)
        faulthandler.dump_traceback(file=sys.stderr)
        if state["full_mode"] is None:
            state["full_mode"] = {}
        state["full_mode"]["error"] = f"exceeded the {deadline:.0f} s budget of the reported-beside legs"
        emit({"cpu_baseline": None, "tc_prefilter": None, "pruned": None})
        sys.stderr.flush()
        os._exit(0 if state["ok"] else 3)

    deadline = float(os.environ.get("MMRS_BENCH_LEG_DEADLINE_S", "200"))
    watchdog = threading.Timer(deadline, bail)
    watchdog.daemon = True
    watchdog.start()

    # ---- candidate-axis partition (axis 2), checked in the same run: 72 000-candidate units split `world` ways must
    # equal the unpartitioned (1-GPU) result, ties included ---------------------------------------------------------
    if world > 1:
        progress(rank, "candidate-axis partition check")
        state["angle"] = optional("angle_axis_check", lambda: angle_axis_check(ctx, nat, world, dist))
        state["ok"] = state["ok"] and bool(state["angle"].get("equal_to_unpartitioned")) and bool(state["angle"].get("all_ranks_identical"))

    # ---- full-mode wall times through the public entry points (all ranks take part) --------------------------------
    if not args.no_api:
        progress(rank, "full-mode legs")
        state["full_mode"] = {}   # filled leg by leg: what was measured before a failure or the deadline is kept
        err = optional("full_mode", lambda: full_mode_legs(ctx, nat, world, rank, dist, barrier, state["full_mode"]))
        if isinstance(err, dict) and "error" in err:
            state["full_mode"]["error"] = err["error"]
    progress(rank, "full-mode legs done")

    if rank != 0:
        watchdog.cancel()
        if world > 1:
            dist.destroy_process_group()
        if not state["ok"]:
            raise SystemExit(3)
        return

    cpu = None

    def cpu_leg():
        from oracle import oracle_py as ora

        ora.build()
        cores = os.cpu_count() or 1
        t0 = time.perf_counter()
        bi, _ = ora.sweep_batch(txy[:n], toff[:2], rxy[:n], roff[:2], cen[:1], 0, STEP_DEG, RANGE_DEG, RANGE_DEG, threads=cores)
        dt = time.perf_counter() - t0
        assert int(bi[0]) == int(res["best_idx"][0]), "GPU and CPU oracle disagree on unit 0"
        return {"value": ncand / dt, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"1 of {U} frame pairs x {ncand} candidates (N=M={n}), {cores} threads over candidates, {dt:.1f} s"}

    if world == 1 and not args.no_cpu_baseline:
        cpu = optional("cpu_baseline", cpu_leg)

    # ---- the opt-in tiers on the round-1 slice of the batch (reported, not the headline) ---------------------------------
    tcp = pruned = None
    if world == 1 and not args.no_tc:
        tcp = optional("tc_prefilter", lambda: tc_leg(ctx, txy, toff, rxy, roff, cen, grid, n, ncand))
        pruned = optional("pruned", lambda: pruned_leg(ctx, flush, txy, toff, rxy, roff, cen, grid, n, ncand, res,
                                                       float(np.mean(dev_ms))))

    progress(rank, "opt-in tier legs done")
    watchdog.cancel()
    emit({"cpu_baseline": cpu, "tc_prefilter": tcp, "pruned": pruned})
    if world > 1:
        dist.destroy_process_group()
    if not state["ok"]:
        print("bench.py: partitioned results differ between ranks or from the 1-GPU golden", file=sys.stderr)
        raise SystemExit(3)


def optional(what, leg):
    """The reported-beside legs must never cost the headline line: a failure becomes {"error": ...} in its place."""
    try:
        return leg()
    except Exception as e:  # noqa: BLE001
        print(f"bench.py: {what} leg failed: {type(e).__name__}: {e}", file=sys.stderr)
        return {"error": f"{type(e).__name__}: {e}"[:300]}


# ---- candidate-axis partition check (N > 1) --------------------------------------------------------------------------
def angle_axis_check(ctx, nat, world, dist):
    """Single-frame sweeps split along the candidate axis (mmrs_sweep_opts.partition = 2): three units on a
    72 000-candidate grid (0.005 deg over +-180) — a plain frame pair, a contour against itself (exact zero at angle 0
    plus near-ties at +-180 deg, the winner sits on a shard boundary), and one on a 720-candidate grid where every
    candidate ties (circle on circle). Must equal the unpartitioned sweep of the same batch on this rank's GPU."""
    rng = np.random.default_rng(7)
    fr = synthetic_pullback(3, 500, SEED + 77)
    a, b = fr[1] - fr[1].mean(0), fr[0] - fr[0].mean(0)
    phi = np.linspace(0, 2 * np.pi, 360, endpoint=False)
    ell = np.stack([2.5 * np.cos(phi), 1.7 * np.sin(phi)], 1) + rng.normal(0, 0.003, (360, 2))
    circ = np.stack([2.0 * np.cos(phi), 2.0 * np.sin(phi)], 1)
    tests, refs = [a, ell, circ], [b, ell, circ]
    toff = np.concatenate([[0], np.cumsum([len(t) for t in tests])])
    roff = np.concatenate([[0], np.cumsum([len(r) for r in refs])])
    grids = [nat.make_grid(0.005, 180.0), nat.make_grid(0.5, 180.0)]
    gou = np.array([0, 0, 1], dtype=np.int32)
    kw = dict(grid_of_unit=gou, mode=0, prefilter=1, prune=-1, tie_margin=1e-9)
    args = (np.concatenate(tests), toff, np.concatenate(refs), roff, np.zeros((3, 2)), grids)
    whole = ctx.sweep_batched(*args, partition=-1, **kw)
    t0 = time.perf_counter()
    split = ctx.sweep_batched(*args, partition=2, **kw)
    dt = time.perf_counter() - t0
    fields = ("best_idx", "best_angle", "best_dist", "best_dist_f32", "n_shortlist", "n_ties", "flags")
    equal = all(np.array_equal(whole[f], split[f]) for f in fields)
    box = [None] * world
    dist.all_gather_object(box, sha(np.stack([split["best_idx"].astype(np.float64), split["best_dist"],
                                              split["n_ties"].astype(np.float64)], 1)))
    return {"units": 3, "candidates": [int(grids[0].n_cand), int(grids[0].n_cand), int(grids[1].n_cand)], "ways": world,
            "equal_to_unpartitioned": bool(equal), "all_ranks_identical": len(set(box)) == 1,
            "best_idx": [int(x) for x in split["best_idx"]], "n_ties": [int(x) for x in split["n_ties"]],
            "n_shortlist": [int(x) for x in split["n_shortlist"]], "wall_ms": 1e3 * dt,
            "collectives": "all-reduce(MIN, uint64) of the packed (distance, index) keys; all-gather of the local f64 winners; "
                           "all-reduce(SUM) of shortlist / tie counts"}


# ---- full-mode wall times ---------------------------------------------------------------------------------------------
def pullback_rows(seed, n_frames, n_points):
    fr = synthetic_pullback(n_frames, n_points, seed)
    z = 0.5 * (n_frames - 1 - np.arange(n_frames))
    a = np.concatenate([np.column_stack([np.full(n_points, float(i)), f, np.full(n_points, z[i])]) for i, f in enumerate(fr)])
    last = a[a[:, 0] == n_frames - 1][0]
    return a, np.array([n_frames - 1, last[1] + 0.1, last[2], last[3]])


def full_mode_legs(ctx, nat, world, rank, dist, barrier, out):
    """Wall time (host clock, barrier + device synchronise on both sides, best of the repetitions) of the public entry
    points on BASELINE's other configurations. With N > 1 every rank makes the same call; the library partitions the
    batched sweeps of the call across the ranks (frame pairs of one case / patients of a cohort)."""
    import multimodars as mm
    from multimodars import _processing as P
    from tests import golden_io as gio

    P._ctx = ctx   # the public entry points run on the bench's context (and its communicator)

    def timed(fn, reps=3):
        best = None
        for _ in range(reps):
            barrier()
            t0 = time.perf_counter()
            r = fn()
            barrier()
            dt = time.perf_counter() - t0
            best = dt if best is None or dt < best else best
        return best, r

    def logs_sha(logs):
        return sha(np.concatenate([np.array(l, dtype=np.float64).reshape(-1) for l in logs]))

    # config 1: the reference's headline benchmark, from_file_full on the example pullbacks (files written from the
    # committed arrays of tests/golden/inputs.npz; benchmarks/benchmark_bruteforce_stepsize.py:30-57)
    pack, gold = gio.inputs(), gio.oracle_outputs()
    tmp = Path(tempfile.mkdtemp(prefix=f"mmrs_bench_r{rank}_"))
    rest, stress = str(gio.write_dir(pack, "rest", tmp / "ivus_rest")), str(gio.write_dir(pack, "stress", tmp / "ivus_stress"))
    kw = dict(range_rotation_deg=90.0, write_obj=False, postprocessing=False, interpolation_steps=0)
    mm.from_file_full(rest, stress, step_rotation_deg=0.5, smooth=True, **kw)   # warm-up (page cache, workspaces)
    c1 = {}
    for tag, k2, ref_s in (("defaults_0p5deg_hierarchical", dict(step_rotation_deg=0.5, smooth=True, bruteforce=False), None),
                           ("0p05deg_hierarchical", dict(step_rotation_deg=0.05, smooth=False, bruteforce=False), 6.25),
                           ("0p05deg_bruteforce", dict(step_rotation_deg=0.05, smooth=False, bruteforce=True), 64.4)):
        dt, r = timed(lambda: mm.from_file_full(rest, stress, **k2, **kw), reps=5)
        c1[tag] = {"wall_s": dt, "reference_published_s": ref_s}
        if tag.startswith("defaults"):
            c1[tag]["logs_equal_oracle_golden"] = bool(all(
                np.array_equal(np.array(r[4][i], dtype=np.float64).reshape(-1, 7), gold[f"cfg1_default_logs_{i}"]) for i in range(4)))
    c1["note"] = ("from_file_full(examples ivus_rest, ivus_stress), +-90 deg, write_obj=False, postprocessing=False; published: "
                  "Xeon Gold 6234, 16 threads (docs/benchmark.rst:36-40)")
    out["config1_from_file_full"] = c1
    progress(rank, "full mode: config 1 done")

    # config 2 through the public API: one pullback pair (pair 0 of the bench workload) -> e2e_api
    ins2 = [mm.numpy_to_inputdata(*pullback_rows(SEED + k, N_FRAMES, N_POINTS), k == 0, label="dia" if k == 0 else "sys")
            for k in range(2)]
    dt, r = timed(lambda: mm.from_array_singlepair(*ins2, step_rotation_deg=STEP_DEG, range_rotation_deg=RANGE_DEG,
                                                   sample_size=500, write_obj=False, bruteforce=True, smooth=True,
                                                   postprocessing=False), reps=2)
    st = ctx.process_stats()
    out["config2_from_array_singlepair"] = {
        "call": "from_array_singlepair(bruteforce=True, step 0.01, range 180): ingest, 398 within + 1 between units, chain, post steps",
        "wall_s": dt, "evals": st["evals"], "value": st["evals"] / dt, "unit": UNIT, "units": st["units"],
        "chain_resolved_units": st["chain_resolved"], "logs_sha256": logs_sha(r[1])}

    progress(rank, "full mode: config 2 done")
    # config 4 slice: full mode, OCT-resolution contours, 0.005 deg brute force (72 000 candidates, N = M = 2 020)
    F4 = int(os.environ.get("MMRS_BENCH_CFG4_FRAMES", "26"))
    ins4 = [mm.numpy_to_inputdata(*pullback_rows(SEED + 40 + k, F4, 2000), k % 2 == 0, label=f"phase{k}") for k in range(4)]
    dt, r = timed(lambda: mm.from_array_full(*ins4, step_rotation_deg=0.005, range_rotation_deg=180.0, sample_size=2000,
                                             write_obj=False, bruteforce=True, smooth=True, postprocessing=False), reps=2)
    st = ctx.process_stats()
    out["config4_slice_from_array_full"] = {
        "call": f"from_array_full, 4 phases x {F4} of 1000 frames x 2000 pts, brute 0.005 deg over +-180, sample_size=2000",
        "wall_s": dt, "evals": st["evals"], "value": st["evals"] / dt, "unit": UNIT, "units": st["units"],
        "chain_resolved_units": st["chain_resolved"], "logs_sha256": logs_sha(r[4]),
        "extrapolated_full_config4_s": dt * (4 * 999) / max(4 * (F4 - 1), 1)}

    progress(rank, "full mode: config 4 slice done")
    # config 5 slice: a cohort of full-mode patients (200 frames x 500 pts, brute 0.05 deg over +-90). Patients are
    # independent cases: with N > 1 whole patients are dealt to the ranks (rank r takes patients r, r + N, ...), each rank
    # runs ONE mmrs_process_cases call on its share with the partition of the sweeps switched off, and the per-frame logs
    # are gathered — no host work is replicated (SURVEY.md §8e: "cfg 5: 32 patients/GPU").
    P5 = int(os.environ.get("MMRS_BENCH_CFG5_PATIENTS", "16"))
    mine = list(range(rank, P5, world))
    blobs = []
    for p in mine:
        for k in range(4):
            a, rp = pullback_rows(SEED + 5000 + 10 * p + k, 200, 500)
            blobs.append(nat.geometry_from_arrays(a, rp, diastole=k % 2 == 0, label=f"pt{p}_{k}"))
    ctx.set_partition(0)
    dt, r = timed(lambda: nat.process_cases(ctx, 4, blobs, 0.05, 90.0, 500, False, True, False) if blobs else ([], [], []),
                  reps=2)
    ctx.set_partition(1)
    st = ctx.process_stats() if blobs else {"evals": 0, "units": 0}
    shas = {p: logs_sha(r[1][4 * i:4 * i + 4]) for i, p in enumerate(mine)}
    evals5, units5 = st["evals"], st["units"]
    if world > 1:
        box = [None] * world
        dist.all_gather_object(box, (shas, evals5, units5))
        shas = {k: v for b_ in box for k, v in b_[0].items()}
        evals5, units5 = sum(b_[1] for b_ in box), sum(b_[2] for b_ in box)
    out["config5_slice_process_cases"] = {
        "call": f"mmrs_process_cases, {P5} of 256 patients x full mode (4 x 200 frames x 500 pts), brute 0.05 deg over +-90; "
                f"whole patients dealt to the {world} rank(s), one call per rank",
        "wall_s": dt, "evals": evals5, "value": evals5 / dt, "unit": UNIT, "units": units5,
        "logs_sha256": sha(np.frombuffer("".join(shas[p] for p in sorted(shas)).encode(), dtype=np.uint8)),
        "extrapolated_256_patients_s": dt * 256 / P5}
    if world > 1:   # every rank must have produced the same logs
        mine = [out[k]["logs_sha256"] for k in ("config2_from_array_singlepair", "config4_slice_from_array_full",
                                                  "config5_slice_process_cases")]
        box = [None] * world
        dist.all_gather_object(box, mine)
        out["all_ranks_identical"] = all(b == box[0] for b in box)
    progress(rank, "full mode: config 5 slice done")
    return None


# ---- opt-in tiers --------------------------------------------------------------------------------------------------
def tc_leg(ctx, txy, toff, rxy, roff, cen, grid, n, ncand):
    Us = 40
    sl = slice(0, Us * n)
    out = {}
    for name, pf in (("dense", 1), ("tc", 2)):
        ctx.sweep_upload(txy[sl], toff[:Us + 1], rxy[sl], roff[:Us + 1], cen[:Us], [grid], mode=0, prefilter=pf)
        best = None
        for _ in range(3):
            ctx.sweep_run()
            r = ctx.sweep_download()
            t = ctx.timings()["total_ms"]
            best = t if best is None or t < best else best
        out[name] = (best, r, ctx.prefilter_info())
    info = out["tc"][2]
    return {"kernel": "k_tc_sweep (tcgen05 kind::f16, bf16x3 split operands, FP32 accumulators in TMEM)",
            "units": Us, "evals_per_s": Us * ncand / (out["tc"][0] * 1e-3),
            "dense_evals_per_s": Us * ncand / (out["dense"][0] * 1e-3),
            "speedup_vs_dense": out["dense"][0] / out["tc"][0], "k1t_ms": info["tc_ms"],
            "rescored_fraction": info["rescored"] / (Us * ncand), "max_err_over_rmax2": info["max_err"],
            "window_over_rmax2": info["window"],
            "identical_selection": bool((out["tc"][1]["best_idx"] == out["dense"][1]["best_idx"]).all()
                                        and (out["tc"][1]["best_dist"] == out["dense"][1]["best_dist"]).all()),
            "default": "off (auto resolves to the dense FP32 sweep)"}


def pruned_leg(ctx, flush, txy, toff, rxy, roff, cen, grid, n, ncand, res, dense_ms):
    Us = 398   # pair 0 = the round-1 workload
    sl = slice(0, Us * n)
    dense_idx, dense_dist = res["best_idx"][:Us].copy(), res["best_dist"][:Us].copy()
    ctx.sweep_upload(txy[sl], toff[:Us + 1], rxy[sl], roff[:Us + 1], cen[:Us], [grid], mode=0, prefilter=1, prune=1)
    ms = []
    for _ in range(4):
        flush.fill_(1)
        ctx.sweep_run()
        r = ctx.sweep_download()
        ms.append(ctx.timings()["total_ms"])
    info = ctx.prefilter_info()
    pm = float(np.mean(ms[1:]))
    return {"kernels": "k_lb<1,8> (rows-only bounds over 32 sampled points of each set, 8 candidates per warp) + k_sweep<..,LIST> on the survivors",
            "units": Us, "ms_per_step": pm, "candidates_decided_per_s": Us * ncand / (pm * 1e-3),
            "speedup_vs_dense": dense_ms * Us / (len(res) * pm), "scored_fraction": info["rescored"] / (Us * ncand),
            "bounds_ms": info["tc_ms"], "survivors_ms": info["rescore_ms"],
            "identical_selection": bool((r["best_idx"] == dense_idx).all() and (r["best_dist"] == dense_dist).all()),
            "default": "off (mmrs_sweep_opts.prune / mmrs_ctx_set_prune / MMRS_PRUNE=1)"}


if __name__ == "__main__":
    main()
