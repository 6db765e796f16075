"""ctypes binding of libmmrs_b200.so (the C ABI of include/mmrs_b200.h).

This is what a maintainer's FFI stub binds (INTEGRATION.md shows the Rust
`extern "C"` block for the same symbols). There is no CPU fallback: importing
works without a GPU (so symbol checks can run), every compute call raises
MmrsError when no B200 is present or the library is not built."""
from __future__ import annotations

import ctypes as C
import os
import weakref
from pathlib import Path

import numpy as np

_PKG_ROOT = Path(__file__).resolve().parent.parent  # multimoda-rs_b200/
LIB_PATH = Path(os.environ.get("MMRS_B200_LIB", _PKG_ROOT / "libmmrs_b200.so"))

c_dp = C.POINTER(C.c_double)
c_i64p = C.POINTER(C.c_int64)
c_i32p = C.POINTER(C.c_int32)


class MmrsError(RuntimeError):
    """Mirrors the reference's PyRuntimeError(format!("{e:#}")) (binding/functions.rs:228)."""


class Grid(C.Structure):
    _fields_ = [("start_rad", C.c_double), ("step_rad", C.c_double), ("n_cand", C.c_int64),
                ("degenerate", C.c_int32), ("fallback", C.c_double)]


class SweepBatch(C.Structure):
    _fields_ = [("n_units", C.c_int64), ("test_xy", c_dp), ("test_off", c_i64p), ("ref_xy", c_dp),
                ("ref_off", c_i64p), ("centre_xy", c_dp), ("grids", C.POINTER(Grid)), ("n_grids", C.c_int64),
                ("grid_of_unit", c_i32p), ("mode", C.c_int32)]


class SweepOpts(C.Structure):
    _fields_ = [("shortlist_rel", C.c_double), ("shortlist_abs", C.c_double), ("shortlist_cap", C.c_int32),
                ("tie_margin", C.c_double), ("keep_dist32", C.c_int32), ("prefilter", C.c_int32),
                ("prefilter_abs", C.c_double), ("prune", C.c_int32), ("partition", C.c_int32)]


class UnitResult(C.Structure):
    _fields_ = [("best_idx", C.c_int64), ("best_angle", C.c_double), ("best_dist", C.c_double),
                ("best_dist_f32", C.c_float), ("n_shortlist", C.c_int32), ("n_ties", C.c_int32),
                ("flags", C.c_int32)]


class TGrid(C.Structure):
    """mmrs_tgrid: (2 half_n + 1)^2 translations t0 + (jx - half_n, jy - half_n) * step."""
    _fields_ = [("t0x", C.c_double), ("t0y", C.c_double), ("step", C.c_double), ("half_n", C.c_int32)]


class RigidResult(C.Structure):
    _fields_ = [("r", UnitResult), ("angle_idx", C.c_int64), ("trans_idx", C.c_int32), ("pad", C.c_int32),
                ("best_tx", C.c_double), ("best_ty", C.c_double)]


class AlignParams(C.Structure):
    _fields_ = [("step_deg", C.c_double), ("range_deg", C.c_double), ("sample_size", C.c_int64),
                ("smooth", C.c_int32), ("bruteforce", C.c_int32), ("postprocessing", C.c_int32)]


class CenterlineParams(C.Structure):
    _fields_ = [("main_ref_pt", C.c_double * 3), ("ccw_ref_pt", C.c_double * 3), ("cw_ref_pt", C.c_double * 3),
                ("angle_step_rad", C.c_double), ("manual_rotation_deg", C.c_double), ("points", c_dp),
                ("n_points", C.c_int64), ("angle_range_rad", C.c_double), ("index_range", C.c_int64),
                ("align_wall_anomalous", C.c_int32)]


RESULT_DTYPE = np.dtype([("best_idx", "<i8"), ("best_angle", "<f8"), ("best_dist", "<f8"), ("best_dist_f32", "<f4"),
                         ("n_shortlist", "<i4"), ("n_ties", "<i4"), ("flags", "<i4")], align=True)
assert RESULT_DTYPE.itemsize == C.sizeof(UnitResult)
# mmrs_rigid_result: the unit result (best_idx = flattened candidate i T + j) plus the angle / translation indices
RIGID_RESULT_DTYPE = np.dtype([("best_idx", "<i8"), ("best_angle", "<f8"), ("best_dist", "<f8"), ("best_dist_f32", "<f4"),
                               ("n_shortlist", "<i4"), ("n_ties", "<i4"), ("flags", "<i4"), ("angle_idx", "<i8"),
                               ("trans_idx", "<i4"), ("pad", "<i4"), ("best_tx", "<f8"), ("best_ty", "<f8")], align=True)
assert RIGID_RESULT_DTYPE.itemsize == C.sizeof(RigidResult)

FLAG_DEGENERATE, FLAG_FULL_F64, FLAG_EMPTY = 1, 2, 4

EXCHANGE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, c_i64p, C.c_int64)

# every symbol include/mmrs_b200.h declares
EXPORTS = [
    "mmrs_ctx_create", "mmrs_ctx_destroy", "mmrs_last_error", "mmrs_version", "mmrs_grid_from_reference_params",
    "mmrs_grid_angle", "mmrs_stage_plan", "mmrs_sweep_batched", "mmrs_sweep_upload", "mmrs_sweep_regrid", "mmrs_sweep_run",
    "mmrs_sweep_download", "mmrs_sweep_plan", "mmrs_sweep_get_dist32", "mmrs_sweep_get_shortlist", "mmrs_last_timings",
    "mmrs_eval_exact", "mmrs_fp32_probe", "mmrs_free", "mmrs_geometry_from_dir", "mmrs_geometry_from_arrays",
    "mmrs_process_cases", "mmrs_process_stats", "mmrs_ctx_set_shard", "mmrs_export_pair", "mmrs_export_single",
    "mmrs_align_centerline", "mmrs_sweep_prefilter_info", "mmrs_ctx_set_prune", "mmrs_contour_metrics",
    "mmrs_comm_unique_id", "mmrs_ctx_comm_init", "mmrs_ctx_set_partition", "mmrs_ctx_comm_info",
    "mmrs_rigid_sweep_batched", "mmrs_rigid_sweep_upload", "mmrs_rigid_sweep_regrid", "mmrs_rigid_sweep_download",
    "mmrs_eval_exact_rigid", "mmrs_partial_sweep_upload", "mmrs_eval_exact_partial", "mmrs_mean_sweep_upload",
    "mmrs_eval_exact_mean",
]

_lib = None


def lib():
    """Loads the shared library; fails loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise MmrsError(f"{LIB_PATH} is missing: build it with __graft_entry__.build() "
                            f"(multimoda-rs_b200/csrc/build.sh). There is no CPU fallback.")
        L = C.CDLL(str(LIB_PATH))
        L.mmrs_last_error.restype = C.c_char_p
        L.mmrs_last_error.argtypes = [C.c_void_p]
        L.mmrs_version.restype = C.c_char_p
        L.mmrs_grid_angle.restype = C.c_double
        L.mmrs_grid_angle.argtypes = [C.POINTER(Grid), C.c_int64]
        L.mmrs_ctx_create.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
        L.mmrs_ctx_destroy.argtypes = [C.c_void_p]
        L.mmrs_free.argtypes = [C.c_void_p]
        L.mmrs_grid_from_reference_params.argtypes = [C.c_double, C.c_double, C.c_int, C.c_double, C.c_double,
                                                      C.POINTER(Grid)]
        L.mmrs_stage_plan.argtypes = [C.c_double, C.c_double, c_dp, c_dp]
        L.mmrs_sweep_batched.argtypes = [C.c_void_p, C.POINTER(SweepBatch), C.POINTER(SweepOpts), C.c_void_p]
        L.mmrs_sweep_upload.argtypes = [C.c_void_p, C.POINTER(SweepBatch), C.POINTER(SweepOpts)]
        L.mmrs_sweep_regrid.argtypes = [C.c_void_p, C.POINTER(Grid), C.c_int64, c_i32p, C.c_double]
        L.mmrs_sweep_run.argtypes = [C.c_void_p]
        L.mmrs_sweep_download.argtypes = [C.c_void_p, C.c_void_p]
        L.mmrs_sweep_plan.argtypes = [C.c_void_p, c_i64p]
        L.mmrs_sweep_get_dist32.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_float), C.c_int64]
        L.mmrs_sweep_get_shortlist.argtypes = [C.c_void_p, C.c_int64, c_i64p, c_dp, C.c_int32, c_i32p]
        L.mmrs_last_timings.argtypes = [C.c_void_p, C.POINTER(C.c_float), c_i32p]
        L.mmrs_eval_exact.argtypes = [C.c_void_p, c_dp, C.c_int64, c_dp, C.c_int64, C.c_double, C.c_double,
                                      C.c_int32, c_dp, C.c_int64, c_dp]
        L.mmrs_fp32_probe.argtypes = [C.c_void_p, C.c_int32, c_dp]
        L.mmrs_process_stats.argtypes = [C.c_void_p, c_i64p]
        L.mmrs_ctx_set_shard.argtypes = [C.c_void_p, C.c_int32, C.c_int32, EXCHANGE_FN, C.c_void_p]
        L.mmrs_rigid_sweep_batched.argtypes = [C.c_void_p, C.POINTER(SweepBatch), C.POINTER(TGrid), C.c_int64, c_i32p,
                                               C.POINTER(SweepOpts), C.c_void_p]
        L.mmrs_rigid_sweep_upload.argtypes = [C.c_void_p, C.POINTER(SweepBatch), C.POINTER(TGrid), C.c_int64, c_i32p,
                                              C.POINTER(SweepOpts)]
        L.mmrs_rigid_sweep_regrid.argtypes = [C.c_void_p, C.POINTER(Grid), C.c_int64, c_i32p, C.POINTER(TGrid), C.c_int64,
                                              c_i32p, C.c_double]
        L.mmrs_rigid_sweep_download.argtypes = [C.c_void_p, C.c_void_p]
        L.mmrs_eval_exact_rigid.argtypes = [C.c_void_p, c_dp, C.c_int64, c_dp, C.c_int64, C.c_double, C.c_double,
                                            C.c_int32, c_dp, c_dp, C.c_int64, c_dp]
        L.mmrs_partial_sweep_upload.argtypes = [C.c_void_p, C.POINTER(SweepBatch), C.POINTER(TGrid), C.c_int64, c_i32p,
                                                C.c_double, C.POINTER(SweepOpts)]
        L.mmrs_eval_exact_partial.argtypes = [C.c_void_p, c_dp, C.c_int64, c_dp, C.c_int64, C.c_double, C.c_double,
                                              C.c_int32, c_dp, c_dp, C.c_int64, C.c_double, c_dp]
        L.mmrs_mean_sweep_upload.argtypes = [C.c_void_p, C.POINTER(SweepBatch), C.POINTER(TGrid), C.c_int64, c_i32p,
                                             C.POINTER(SweepOpts)]
        L.mmrs_eval_exact_mean.argtypes = [C.c_void_p, c_dp, C.c_int64, c_dp, C.c_int64, C.c_double, C.c_double,
                                           C.c_int32, c_dp, c_dp, C.c_int64, c_dp]
        _lib = L
    return _lib


def _err(ctx_ptr):
    return lib().mmrs_last_error(ctx_ptr).decode(errors="replace")


def make_grid(step_deg, range_deg, center=None, limes_deg=None) -> Grid:
    """mmrs_grid_from_reference_params: the grid of process_utils.rs:43-67."""
    g = Grid()
    limes_deg = range_deg if limes_deg is None else limes_deg
    rc = lib().mmrs_grid_from_reference_params(step_deg, range_deg, int(center is not None),
                                               0.0 if center is None else float(center), limes_deg, C.byref(g))
    if rc:
        raise MmrsError(_err(None))
    return g


def grid_angle(g: Grid, i: int) -> float:
    return lib().mmrs_grid_angle(C.byref(g), int(i))


def make_tgrid(step, half_n, t0=(0.0, 0.0)) -> TGrid:
    """Translation grid of (2 half_n + 1)^2 offsets t0 + ((jx - half_n) step, (jy - half_n) step), j = jy (2 half_n + 1) + jx."""
    return TGrid(float(t0[0]), float(t0[1]), float(step), int(half_n))


def stage_plan(step_deg, range_deg):
    s = (C.c_double * 4)()
    w = (C.c_double * 4)()
    n = lib().mmrs_stage_plan(step_deg, range_deg, s, w)
    return [(s[i], w[i]) for i in range(n)]


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class Context:
    """Owns one mmrs_ctx (one device, one stream, grow-only device workspaces)."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self._p = C.c_void_p()
        rc = lib().mmrs_ctx_create(int(device), C.c_void_p(stream) if stream else None, C.byref(self._p))
        if rc:
            raise MmrsError(_err(None))
        self.device = device
        self._keep = None

    def close(self):
        if self._p:
            lib().mmrs_ctx_destroy(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc:
            raise MmrsError(_err(self._p))

    # -- sweep --------------------------------------------------------------------
    def _batch(self, test_xy, test_off, ref_xy, ref_off, centre_xy, grids, grid_of_unit, mode):
        test_xy, ref_xy, centre_xy = _f64(test_xy).reshape(-1), _f64(ref_xy).reshape(-1), _f64(centre_xy).reshape(-1)
        test_off = np.ascontiguousarray(test_off, dtype=np.int64)
        ref_off = np.ascontiguousarray(ref_off, dtype=np.int64)
        U = len(test_off) - 1
        assert len(ref_off) == U + 1 and len(centre_xy) == 2 * U
        garr = (Grid * max(len(grids), 1))(*grids)
        gou = None if grid_of_unit is None else np.ascontiguousarray(grid_of_unit, dtype=np.int32)
        b = SweepBatch(U, test_xy.ctypes.data_as(c_dp), test_off.ctypes.data_as(c_i64p), ref_xy.ctypes.data_as(c_dp),
                       ref_off.ctypes.data_as(c_i64p), centre_xy.ctypes.data_as(c_dp), garr, len(grids),
                       None if gou is None else gou.ctypes.data_as(c_i32p), int(mode))
        self._keep = (test_xy, test_off, ref_xy, ref_off, centre_xy, garr, gou)
        return b, U

    @staticmethod
    def _opts(shortlist_rel=0.0, shortlist_abs=0.0, shortlist_cap=0, tie_margin=0.0, keep_dist32=False, prefilter=0,
              prefilter_abs=0.0, prune=0, partition=0):
        """prefilter: 0 auto, 1 off (dense FP32 sweep), 2 required (tensor-core tier, mmrs_b200.h).
        prune: > 0 exact lower-bound pruning on, < 0 off, 0 the context default (set_prune).
        partition: 0 the context's axis, -1 not partitioned, 1 whole units, 2 candidate angles (comm_init)."""
        return SweepOpts(shortlist_rel, shortlist_abs, shortlist_cap, tie_margin, int(keep_dist32), int(prefilter),
                         float(prefilter_abs), int(prune), int(partition))

    def set_prune(self, on: bool):
        """mmrs_ctx_set_prune: context-wide default for exact lower-bound pruning (mmrs_process_cases uses it)."""
        lib().mmrs_ctx_set_prune.argtypes = [C.c_void_p, C.c_int32]
        self._check(lib().mmrs_ctx_set_prune(self._p, int(bool(on))))

    def sweep_batched(self, test_xy, test_off, ref_xy, ref_off, centre_xy, grids, grid_of_unit=None, mode=0, **opts):
        """Host arrays in, structured result array (RESULT_DTYPE) out."""
        b, U = self._batch(test_xy, test_off, ref_xy, ref_off, centre_xy, grids, grid_of_unit, mode)
        o = self._opts(**opts)
        out = np.zeros(U, dtype=RESULT_DTYPE)
        self._check(lib().mmrs_sweep_batched(self._p, C.byref(b), C.byref(o), out.ctypes.data_as(C.c_void_p)))
        self._n_units = U
        return out

    def sweep_upload(self, test_xy, test_off, ref_xy, ref_off, centre_xy, grids, grid_of_unit=None, mode=0, **opts):
        b, U = self._batch(test_xy, test_off, ref_xy, ref_off, centre_xy, grids, grid_of_unit, mode)
        o = self._opts(**opts)
        self._check(lib().mmrs_sweep_upload(self._p, C.byref(b), C.byref(o)))
        self._n_units = U

    def sweep_regrid(self, grids, grid_of_unit=None, tie_margin=0.0):
        garr = (Grid * max(len(grids), 1))(*grids)
        gou = None if grid_of_unit is None else np.ascontiguousarray(grid_of_unit, dtype=np.int32)
        self._check(lib().mmrs_sweep_regrid(self._p, garr, len(grids), None if gou is None else gou.ctypes.data_as(c_i32p),
                                            float(tie_margin)))

    def sweep_run(self):
        self._check(lib().mmrs_sweep_run(self._p))

    def sweep_download(self):
        out = np.zeros(self._n_units, dtype=RESULT_DTYPE)
        self._check(lib().mmrs_sweep_download(self._p, out.ctypes.data_as(C.c_void_p)))
        return out

    # -- rigid candidates (angle grid x translation grid, mmrs_b200.h "rigid candidates") -------------------------
    @staticmethod
    def _tgrids(tgrids, tgrid_of_unit):
        """(array, count, tgrid_of_unit pointer) of the C calls; tgrids=None (rotation only): (None, 0, None)."""
        if tgrids is None:
            return None, 0, None
        tarr = (TGrid * max(len(tgrids), 1))(*tgrids)
        tou = None if tgrid_of_unit is None else np.ascontiguousarray(tgrid_of_unit, dtype=np.int32)
        return tarr, len(tgrids), None if tou is None else tou.ctypes.data_as(c_i32p)   # the pointer keeps tou alive

    def rigid_sweep_batched(self, test_xy, test_off, ref_xy, ref_off, centre_xy, grids, tgrids, grid_of_unit=None,
                            tgrid_of_unit=None, mode=0, **opts):
        """mmrs_rigid_sweep_batched: host arrays in, structured result array (RIGID_RESULT_DTYPE) out."""
        b, U = self._batch(test_xy, test_off, ref_xy, ref_off, centre_xy, grids, grid_of_unit, mode)
        tarr, n_t, ptou = self._tgrids(tgrids, tgrid_of_unit)
        o = self._opts(**opts)
        out = np.zeros(U, dtype=RIGID_RESULT_DTYPE)
        self._check(lib().mmrs_rigid_sweep_batched(self._p, C.byref(b), tarr, n_t, ptou, C.byref(o),
                                                   out.ctypes.data_as(C.c_void_p)))
        self._n_units = U
        return out

    def rigid_upload(self, test_xy, test_off, ref_xy, ref_off, centre_xy, grids, tgrids, grid_of_unit=None,
                     tgrid_of_unit=None, mode=0, **opts):
        b, U = self._batch(test_xy, test_off, ref_xy, ref_off, centre_xy, grids, grid_of_unit, mode)
        tarr, n_t, ptou = self._tgrids(tgrids, tgrid_of_unit)
        o = self._opts(**opts)
        self._check(lib().mmrs_rigid_sweep_upload(self._p, C.byref(b), tarr, n_t, ptou, C.byref(o)))
        self._n_units = U

    def rigid_regrid(self, grids, tgrids, grid_of_unit=None, tgrid_of_unit=None, tie_margin=0.0):
        garr = (Grid * max(len(grids), 1))(*grids)
        gou = None if grid_of_unit is None else np.ascontiguousarray(grid_of_unit, dtype=np.int32)
        tarr, n_t, ptou = self._tgrids(tgrids, tgrid_of_unit)
        self._check(lib().mmrs_rigid_sweep_regrid(self._p, garr, len(grids), None if gou is None else gou.ctypes.data_as(c_i32p),
                                                  tarr, n_t, ptou, float(tie_margin)))

    def rigid_download(self):
        out = np.zeros(self._n_units, dtype=RIGID_RESULT_DTYPE)
        self._check(lib().mmrs_rigid_sweep_download(self._p, out.ctypes.data_as(C.c_void_p)))
        return out

    def _eval(self, fn, name, test_xy, ref_xy, centre, mode, angles, txy, *cost_args):
        """mmrs_eval_exact_<cost>: f64 cost of the candidates (angles[k], txy[k]); txy=None passes NULL."""
        t, r, a = _f64(test_xy).reshape(-1, 2), _f64(ref_xy).reshape(-1, 2), _f64(angles).reshape(-1)
        tt = None
        if txy is not None:
            tt = _f64(txy).reshape(-1, 2)
            if len(tt) != len(a):
                raise ValueError(f"{name}: angles and txy differ in length")
        out = np.empty(len(a), dtype=np.float64)
        self._check(fn(self._p, t.ctypes.data_as(c_dp), len(t), r.ctypes.data_as(c_dp), len(r), float(centre[0]),
                       float(centre[1]), int(mode), a.ctypes.data_as(c_dp),
                       None if tt is None else tt.ctypes.data_as(c_dp), len(a), *cost_args, out.ctypes.data_as(c_dp)))
        return out

    def eval_exact_rigid(self, test_xy, ref_xy, centre, mode, angles, txy):
        """f64 cost of the rigid candidates (angles[k], txy[k]) (mmrs_eval_exact_rigid)."""
        return self._eval(lib().mmrs_eval_exact_rigid, "eval_exact_rigid", test_xy, ref_xy, centre, mode, angles, txy)

    # -- partial cost (rank-K Hausdorff distance, mmrs_b200.h "partial cost") -------------------------------------
    def partial_upload(self, test_xy, test_off, ref_xy, ref_off, centre_xy, grids, tgrids=None, grid_of_unit=None,
                       tgrid_of_unit=None, mode=0, inlier_fraction=1.0, **opts):
        """mmrs_partial_sweep_upload: rigid_upload (tgrids given) or sweep_upload (tgrids=None) with the partial cost.
        Run with sweep_run; download with sweep_download, or rigid_download after a rigid upload."""
        b, U = self._batch(test_xy, test_off, ref_xy, ref_off, centre_xy, grids, grid_of_unit, mode)
        o = self._opts(**opts)
        tarr, n_t, ptou = self._tgrids(tgrids, tgrid_of_unit)
        self._check(lib().mmrs_partial_sweep_upload(self._p, C.byref(b), tarr, n_t, ptou, float(inlier_fraction),
                                                    C.byref(o)))
        self._n_units = U

    def eval_exact_partial(self, test_xy, ref_xy, centre, mode, angles, txy=None, inlier_fraction=1.0):
        """f64 partial cost of the candidates (angles[k], txy[k]) (txy=None: rotation only; mmrs_eval_exact_partial)."""
        return self._eval(lib().mmrs_eval_exact_partial, "eval_exact_partial", test_xy, ref_xy, centre, mode, angles,
                          txy, float(inlier_fraction))

    # -- mean cost (modified Hausdorff distance, mmrs_b200.h "mean cost") -------------------------------------------
    def mean_upload(self, test_xy, test_off, ref_xy, ref_off, centre_xy, grids, tgrids=None, grid_of_unit=None,
                    tgrid_of_unit=None, mode=0, **opts):
        """mmrs_mean_sweep_upload: rigid_upload (tgrids given) or sweep_upload (tgrids=None) with the mean cost.
        Run with sweep_run; download with sweep_download, or rigid_download after a rigid upload."""
        b, U = self._batch(test_xy, test_off, ref_xy, ref_off, centre_xy, grids, grid_of_unit, mode)
        o = self._opts(**opts)
        tarr, n_t, ptou = self._tgrids(tgrids, tgrid_of_unit)
        self._check(lib().mmrs_mean_sweep_upload(self._p, C.byref(b), tarr, n_t, ptou, C.byref(o)))
        self._n_units = U

    def eval_exact_mean(self, test_xy, ref_xy, centre, mode, angles, txy=None):
        """f64 mean cost of the candidates (angles[k], txy[k]) (txy=None: rotation only; mmrs_eval_exact_mean)."""
        return self._eval(lib().mmrs_eval_exact_mean, "eval_exact_mean", test_xy, ref_xy, centre, mode, angles, txy)

    def plan(self):
        p = (C.c_int64 * 5)()
        self._check(lib().mmrs_sweep_plan(self._p, p))
        return dict(TA=p[0], multi=bool(p[1] & 1), exact_tiling=bool(p[1] & 2), blocked=bool(p[1] & 4), ctas=p[2], smem_bytes=p[3],
                    size_classes=p[4])

    def dist32(self, unit, n_cand):
        out = np.empty(n_cand, dtype=np.float32)
        self._check(lib().mmrs_sweep_get_dist32(self._p, unit, out.ctypes.data_as(C.POINTER(C.c_float)), n_cand))
        return out

    def shortlist(self, unit, cap=1 << 17):
        idx = np.empty(cap, dtype=np.int64)
        d = np.empty(cap, dtype=np.float64)
        n = C.c_int32()
        self._check(lib().mmrs_sweep_get_shortlist(self._p, unit, idx.ctypes.data_as(c_i64p), d.ctypes.data_as(c_dp),
                                                   cap, C.byref(n)))
        k = min(n.value, cap)
        return idx[:k].copy(), d[:k].copy()

    def timings(self):
        ms = (C.c_float * 4)()
        n = C.c_int32()
        self._check(lib().mmrs_last_timings(self._p, ms, C.byref(n)))
        return dict(sweep_ms=ms[0], shortlist_ms=ms[1], recheck_ms=ms[2], total_ms=ms[3], launches=n.value)

    def prefilter_info(self):
        """mmrs_sweep_prefilter_info of the last run."""
        o = (C.c_double * 6)()
        lib().mmrs_sweep_prefilter_info.argtypes = [C.c_void_p, c_dp]
        self._check(lib().mmrs_sweep_prefilter_info(self._p, o))
        ran = bool(o[0])
        # when no tier ran, [3] / [4] count the early-break dense sweep (K1e): pair distances evaluated, candidates scored
        return dict(ran=ran, kind={0: None, 1: "tensor-core prefilter", 2: "lower-bound pruning", 3: "expanded-form tier"}[int(o[0])],
                    tc_ms=o[1], rescore_ms=o[2], rescored=int(o[3]) if ran else 0, max_err=o[4] if ran else 0.0, window=o[5],
                    eb_pairs=0 if ran else int(o[3]), eb_candidates=0 if ran else int(o[4]))

    def eval_exact(self, test_xy, ref_xy, centre, mode, angles):
        t, r, a = _f64(test_xy).reshape(-1, 2), _f64(ref_xy).reshape(-1, 2), _f64(angles).reshape(-1)
        out = np.empty(len(a), dtype=np.float64)
        self._check(lib().mmrs_eval_exact(self._p, t.ctypes.data_as(c_dp), len(t), r.ctypes.data_as(c_dp), len(r),
                                          float(centre[0]), float(centre[1]), int(mode), a.ctypes.data_as(c_dp),
                                          len(a), out.ctypes.data_as(c_dp)))
        return out

    def fp32_probe(self, iters=4096):
        t = C.c_double()
        self._check(lib().mmrs_fp32_probe(self._p, iters, C.byref(t)))
        return t.value

    def set_shard(self, rank: int, world: int, allreduce_sum_int64):
        """mmrs_ctx_set_shard. `allreduce_sum_int64(np.ndarray[int64]) -> None` sums the array in place across
        ranks (see multimodars._dist.make_exchange). world <= 1 switches sharding off."""
        if world <= 1 or allreduce_sum_int64 is None:
            self._exchange_cb = None
            self._check(lib().mmrs_ctx_set_shard(self._p, 0, 1, C.cast(None, EXCHANGE_FN), None))
            return

        def _cb(_user, buf, n):
            try:
                allreduce_sum_int64(np.ctypeslib.as_array(buf, shape=(n,)))
                return 0
            except Exception:  # surfaced as an MmrsError by the C side
                import traceback

                traceback.print_exc()
                return 1

        self._exchange_cb = EXCHANGE_FN(_cb)   # keep the trampoline alive
        self._check(lib().mmrs_ctx_set_shard(self._p, int(rank), int(world), self._exchange_cb, None))

    def comm_init(self, uid: bytes, rank: int, world: int):
        """mmrs_ctx_comm_init: binds an NCCL communicator (collective over all `world` ranks). `uid` is the 128-byte
        token rank 0 obtained from comm_unique_id() and handed to the others (multimodars._dist.init_comm)."""
        if len(uid) != COMM_ID_BYTES:
            raise ValueError("uid must be 128 bytes")
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(uid)
        lib().mmrs_ctx_comm_init.argtypes = [C.c_void_p, C.POINTER(C.c_uint8), C.c_int32, C.c_int32]
        self._check(lib().mmrs_ctx_comm_init(self._p, buf, int(rank), int(world)))

    def set_partition(self, axis: int):
        """mmrs_ctx_set_partition: 1 whole units (default), 2 candidate angles, 0 none."""
        lib().mmrs_ctx_set_partition.argtypes = [C.c_void_p, C.c_int32]
        self._check(lib().mmrs_ctx_set_partition(self._p, int(axis)))

    def comm_info(self):
        out = (C.c_int32 * 4)()
        lib().mmrs_ctx_comm_info.argtypes = [C.c_void_p, C.POINTER(C.c_int32)]
        lib().mmrs_ctx_comm_info(self._p, out)
        return dict(rank=out[0], world=out[1], axis=out[2], nccl=bool(out[3]))

    def process_stats(self):
        s = (C.c_int64 * 5)()
        self._check(lib().mmrs_process_stats(self._p, s))
        return dict(units=s[0], evals=s[1], rechecks=s[2], chain_resolved=s[3], launches=s[4])


COMM_ID_BYTES = 128


def comm_unique_id() -> bytes:
    """mmrs_comm_unique_id (ncclGetUniqueId): called on rank 0, the token goes to every rank's comm_init."""
    buf = (C.c_uint8 * COMM_ID_BYTES)()
    lib().mmrs_comm_unique_id.argtypes = [C.POINTER(C.c_uint8)]
    if lib().mmrs_comm_unique_id(buf):
        raise MmrsError(_err(None))
    return bytes(buf)


def contour_metrics(xyz, centroid=None):
    """mmrs_contour_metrics: (area, (far_i, far_j, far_dist), (opp_i, opp_j, opp_dist_2d), opp_dist_3d) of n packed
    (x, y, z) points by the reference's own loops (types/native/contour.rs:227-363); host only, no context."""
    a = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
    out = (C.c_double * 8)()
    c = None if centroid is None else (C.c_double * 3)(float(centroid[0]), float(centroid[1]), float(centroid[2]))
    L = lib()
    L.mmrs_contour_metrics.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_double * 8]
    rc = L.mmrs_contour_metrics(a.ctypes.data_as(C.c_void_p), len(a), 0 if c is None else 1, c, out)
    if rc:
        raise MmrsError(_err(None))
    return out[0], (int(out[1]) if out[1] == out[1] else -1, int(out[2]) if out[2] == out[2] else -1, out[3]), \
        (int(out[4]) if out[4] == out[4] else -1, int(out[5]) if out[5] == out[5] else -1, out[6]), out[7]


# ---- geometry-level entry points ---------------------------------------------------
def _take_blob(ptr, n):
    """Wraps a malloc'ed f64 buffer handed out by the library as a numpy array WITHOUT copying; the buffer is
    released with mmrs_free when the last view of it dies."""
    if n <= 0:
        lib().mmrs_free(ptr)
        return np.zeros(0, dtype=np.float64)
    buf = (C.c_double * n).from_address(C.addressof(ptr.contents))
    weakref.finalize(buf, lib().mmrs_free, C.cast(ptr, C.c_void_p))
    return np.frombuffer(buf, dtype=np.float64)


def geometry_from_dir(path, label, diastole, image_center=(4.5, 4.5), radius=0.5, n_points=20, ctx: Context | None = None):
    """mmrs_geometry_from_dir -> geometry blob (host-only; replaces io/build.rs:9-205 + io/input.rs:62-147)."""
    L = lib()
    L.mmrs_geometry_from_dir.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_int, C.c_double, C.c_double,
                                         C.c_double, C.c_uint32, C.POINTER(c_dp), c_i64p]
    blob, n = c_dp(), C.c_int64()
    p = ctx._p if ctx is not None else None
    rc = L.mmrs_geometry_from_dir(p, os.fsencode(str(path)), label.encode(), int(diastole), image_center[0],
                                  image_center[1], radius, int(n_points), C.byref(blob), C.byref(n))
    if rc:
        raise MmrsError(_err(p))
    return _take_blob(blob, n.value)


def geometry_from_arrays(lumen, ref_point, eem=None, calc=None, side=None, records=None, diastole=True, label="geom",
                         image_center=(4.5, 4.5), radius=0.5, n_points=20, ctx: Context | None = None):
    """mmrs_geometry_from_arrays -> geometry blob. Arrays are (N,4) [frame, x, y, z]."""
    L = lib()
    L.mmrs_geometry_from_arrays.argtypes = [C.c_void_p, c_dp, C.c_int64, c_dp, C.c_int64, c_dp, C.c_int64, c_dp,
                                            C.c_int64, c_dp, C.c_int64, c_dp, C.c_int, C.c_char_p, C.c_double,
                                            C.c_double, C.c_double, C.c_uint32, C.POINTER(c_dp), c_i64p]

    def arr(a):
        if a is None:
            return None, None, 0
        a = np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(-1, 4))
        return a, a.ctypes.data_as(c_dp), a.shape[0]

    keep = [arr(lumen), arr(eem), arr(calc), arr(side), arr(records)]
    rp = np.ascontiguousarray(np.asarray(ref_point, dtype=np.float64).reshape(4))
    blob, n = c_dp(), C.c_int64()
    p = ctx._p if ctx is not None else None
    args = []
    for k in keep:
        args += [k[1], k[2]]
    rc = L.mmrs_geometry_from_arrays(p, *args, rp.ctypes.data_as(c_dp), int(diastole), label.encode(),
                                     image_center[0], image_center[1], radius, int(n_points), C.byref(blob),
                                     C.byref(n))
    if rc:
        raise MmrsError(_err(p))
    return _take_blob(blob, n.value)


N_IN = {4: 4, 3: 4, 2: 2, 1: 1}
N_OUT = {4: 8, 3: 4, 2: 2, 1: 1}


def process_cases(ctx: Context, mode, blobs, step_deg, range_deg, sample_size, smooth, bruteforce, postprocessing=False):
    """mmrs_process_cases for len(blobs)/N_IN[mode] cases. Returns (out_blobs, logs, anomalous)."""
    L = lib()
    n_in, n_out = N_IN[mode], N_OUT[mode]
    assert len(blobs) % n_in == 0
    n_cases = len(blobs) // n_in
    arrs = [np.ascontiguousarray(b, dtype=np.float64) for b in blobs]
    ptrs = (c_dp * max(len(arrs), 1))(*[a.ctypes.data_as(c_dp) for a in arrs])
    lens = (C.c_int64 * max(len(arrs), 1))(*[len(a) for a in arrs])
    ob = (c_dp * max(n_cases * n_out, 1))()
    ol = (C.c_int64 * max(n_cases * n_out, 1))()
    lg = (c_dp * max(len(arrs), 1))()
    nl = (C.c_int64 * max(len(arrs), 1))()
    an = (C.c_int32 * max(len(arrs), 1))()
    prm = AlignParams(step_deg, range_deg, int(sample_size), int(smooth), int(bruteforce), int(postprocessing))
    L.mmrs_process_cases.argtypes = [C.c_void_p, C.c_int32, C.c_int64, C.POINTER(c_dp), c_i64p,
                                     C.POINTER(AlignParams), C.POINTER(c_dp), c_i64p, C.POINTER(c_dp), c_i64p, c_i32p]
    rc = L.mmrs_process_cases(ctx._p, int(mode), n_cases, ptrs, lens, C.byref(prm), ob, ol, lg, nl, an)
    if rc:
        raise MmrsError(_err(ctx._p))
    outs = [_take_blob(ob[i], ol[i]) for i in range(n_cases * n_out)]
    logs = [_take_blob(lg[i], nl[i] * 7).reshape(-1, 7) for i in range(len(arrs))]
    return outs, logs, [bool(an[i]) for i in range(len(arrs))]


# ---- export + centerline alignment --------------------------------------------------
def _kinds(kinds):
    k = np.ascontiguousarray([int(x) for x in kinds], dtype=np.int32)
    return k, k.ctypes.data_as(c_i32p), len(k)


def export_pair(blob_a, blob_b, label_a, case_name, output_dir, interpolation_steps, watertight, kinds,
                ctx: Context | None = None):
    """mmrs_export_pair (to_object::process_case, to_object/process.rs:9-61)."""
    L = lib()
    L.mmrs_export_pair.argtypes = [C.c_void_p, c_dp, C.c_int64, c_dp, C.c_int64, C.c_char_p, C.c_char_p, C.c_char_p,
                                   C.c_int64, C.c_int32, c_i32p, C.c_int32]
    a, b = _f64(blob_a), _f64(blob_b)
    keep, kp, kn = _kinds(kinds)
    p = ctx._p if ctx is not None else None
    rc = L.mmrs_export_pair(p, a.ctypes.data_as(c_dp), len(a), b.ctypes.data_as(c_dp), len(b), str(label_a).encode(),
                            str(case_name).encode(), os.fsencode(str(output_dir)), int(interpolation_steps),
                            int(bool(watertight)), kp, kn)
    if rc:
        raise MmrsError(_err(p))


def export_single(blob, name, output_dir, watertight, kinds, naming, ctx: Context | None = None):
    """mmrs_export_single (entry.rs:741-818 for naming 0, to_object/process.rs:63-121 for naming 1)."""
    L = lib()
    L.mmrs_export_single.argtypes = [C.c_void_p, c_dp, C.c_int64, C.c_char_p, C.c_char_p, C.c_int32, c_i32p,
                                     C.c_int32, C.c_int32]
    a = _f64(blob)
    keep, kp, kn = _kinds(kinds)
    p = ctx._p if ctx is not None else None
    rc = L.mmrs_export_single(p, a.ctypes.data_as(c_dp), len(a), str(name).encode(), os.fsencode(str(output_dir)),
                              int(bool(watertight)), kp, kn, int(naming))
    if rc:
        raise MmrsError(_err(p))


def align_centerline(ctx: Context | None, method, centerline_rows, blobs, main_ref_pt=(0, 0, 0), ccw_ref_pt=(0, 0, 0),
                     cw_ref_pt=(0, 0, 0), angle_step_rad=0.0, manual_rotation_deg=0.0, points=None,
                     angle_range_rad=0.0, index_range=0, align_wall_anomalous=False):
    """mmrs_align_centerline. centerline_rows: (n, 8) [x, y, z, tx, ty, tz, branch_id, radius].
    Returns (out_blobs, spacing_mm, rotation_rad, (refine_hausdorff, refine_candidates))."""
    L = lib()
    L.mmrs_align_centerline.argtypes = [C.c_void_p, C.c_int32, c_dp, C.c_int64, C.c_int32, C.POINTER(c_dp), c_i64p,
                                        C.POINTER(CenterlineParams), C.POINTER(c_dp), c_i64p, c_dp, c_dp, c_dp]
    cl = np.ascontiguousarray(np.asarray(centerline_rows, dtype=np.float64).reshape(-1, 8))
    arrs = [_f64(b) for b in blobs]
    ptrs = (c_dp * len(arrs))(*[a.ctypes.data_as(c_dp) for a in arrs])
    lens = (C.c_int64 * len(arrs))(*[len(a) for a in arrs])
    prm = CenterlineParams()
    prm.main_ref_pt[:] = [float(v) for v in main_ref_pt]
    prm.ccw_ref_pt[:] = [float(v) for v in ccw_ref_pt]
    prm.cw_ref_pt[:] = [float(v) for v in cw_ref_pt]
    prm.angle_step_rad = float(angle_step_rad)
    prm.manual_rotation_deg = float(manual_rotation_deg)
    pts = None
    if points is not None and len(points):
        pts = np.ascontiguousarray(np.asarray(points, dtype=np.float64).reshape(-1, 3))
        prm.points = pts.ctypes.data_as(c_dp)
        prm.n_points = len(pts)
    prm.angle_range_rad = float(angle_range_rad)
    prm.index_range = int(index_range)
    prm.align_wall_anomalous = int(bool(align_wall_anomalous))
    ob = (c_dp * len(arrs))()
    ol = (C.c_int64 * len(arrs))()
    spacing, rot = C.c_double(), C.c_double()
    refine = (C.c_double * 2)()
    p = ctx._p if ctx is not None else None
    rc = L.mmrs_align_centerline(p, int(method), cl.ctypes.data_as(c_dp), len(cl), len(arrs), ptrs, lens,
                                 C.byref(prm), ob, ol, C.byref(spacing), C.byref(rot), refine)
    if rc:
        raise MmrsError(_err(p))
    outs = [_take_blob(ob[i], ol[i]) for i in range(len(arrs))]
    return outs, spacing.value, rot.value, (refine[0], int(refine[1]))
