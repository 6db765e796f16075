/* ============================================================================
 * mmrs_b200.h — C ABI of the B200-native Hausdorff rotation-sweep library
 * (libmmrs_b200.so, built from multimoda-rs_b200/csrc/).
 *
 * This is the drop-in boundary for ONE path of yungselm/multimoda-rs v0.7.0:
 * the brute-force / coarse-to-fine rotation sweep scored by symmetric 2-D
 * Hausdorff distance. Every entry point cites the reference interface it
 * replaces (paths relative to the reference checkout root). Plain pointers and
 * sizes only; no C++ / torch types. All host arrays are caller-owned; the
 * opaque context owns device workspaces. Functions return 0 on success and a
 * non-zero status otherwise; mmrs_last_error() gives the message (the
 * reference surfaces anyhow::Error chains as PyRuntimeError,
 * src/intravascular/binding/functions.rs:228).
 *
 * There is NO CPU fallback: every compute entry point fails with
 * MMRS_ERR_CUDA when no CUDA device / sm_100a image is available.
 * ========================================================================== */
#ifndef MMRS_B200_H
#define MMRS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMRS_OK 0
#define MMRS_ERR_ARG 1    /* invalid argument                                  */
#define MMRS_ERR_CUDA 2   /* CUDA runtime / no device / wrong architecture     */
#define MMRS_ERR_INPUT 3  /* reference-style input error (anyhow! in the ref)  */
#define MMRS_ERR_STATE 4  /* call order (e.g. run before upload)               */

typedef struct mmrs_ctx mmrs_ctx;

/* ---- context ------------------------------------------------------------- */
/* `stream` is a cudaStream_t the library launches on (so the caller's CUDA
 * events see the kernels); NULL = the library creates its own stream.        */
int mmrs_ctx_create(int device, void* stream, mmrs_ctx** out);
void mmrs_ctx_destroy(mmrs_ctx* ctx);
/* Message of the last failing call on `ctx` (or of the last failing call that
 * had no context when ctx == NULL). Never NULL.                               */
const char* mmrs_last_error(const mmrs_ctx* ctx);
const char* mmrs_version(void);

/* ---- candidate grid ----------------------------------------------------------
 * Replaces the grid construction inside `search_range`
 * (src/intravascular/processing/process_utils.rs:43-67): start/stop clipped to
 * +-limes, steps = max(ceil((stop-start)/step) as usize, 1), candidates
 * start + i*step while <= stop, each wrapped to [-pi, pi).
 * degenerate != 0  <=>  search_range returns `fallback` without evaluating.   */
typedef struct mmrs_grid {
    double start_rad;
    double step_rad;
    int64_t n_cand;
    int32_t degenerate;
    double fallback;
} mmrs_grid;

int mmrs_grid_from_reference_params(double step_deg, double range_deg, int has_center, double center_rad,
                                    double limes_deg, mmrs_grid* out);
/* Wrapped candidate angle i: ((start + i*step + pi).rem_euclid(2pi)) - pi.    */
double mmrs_grid_angle(const mmrs_grid* g, int64_t i);

/* The stage plan of the coarse-to-fine driver `find_best_rotation`
 * (src/intravascular/processing/align_within.rs:208-246, identical copy in
 * align_between.rs:219-257). Writes up to 4 (step_deg, half_window_deg) pairs;
 * stage 0 is centred on 0 (None), stage k>0 on the result of stage k-1; every
 * stage is clipped to +-range_deg. Returns the number of stages.              */
int mmrs_stage_plan(double step_deg, double range_deg, double step_out[4], double window_out[4]);

/* ---- batched sweep -------------------------------------------------------------
 * One "unit" = one `search_range` call with the Hausdorff cost closure:
 *   mode 0: intrapullback closure, align_within.rs:99-105 / :200-206
 *           (ContourPoint::rotate about `centre`, identity iff angle == 0.0,
 *            src/types/native/contour_point.rs:38-52)
 *   mode 1: inter-pullback closure, align_between.rs:189-216 (no shortcut;
 *           `centre` = the reference cloud's mean, align_between.rs:260-271)
 * followed by `hausdorff_distance(reference, rotated)`
 * (process_utils.rs:78-121) and the leftmost arg-min of process_utils.rs:69-74.
 *
 * Points are packed (x, y) doubles, units concatenated; unit u owns
 * test_xy[2*test_off[u] .. 2*test_off[u+1]) and likewise for ref.
 * `grid_of_unit` == NULL: every unit uses grids[0] (the brute-force case).    */
typedef struct mmrs_sweep_batch {
    int64_t n_units;
    const double* test_xy;
    const int64_t* test_off; /* [n_units + 1] */
    const double* ref_xy;
    const int64_t* ref_off;  /* [n_units + 1] */
    const double* centre_xy; /* [n_units][2]  */
    const mmrs_grid* grids;
    int64_t n_grids;
    const int32_t* grid_of_unit; /* [n_units] or NULL */
    int32_t mode;
} mmrs_sweep_batch;

typedef struct mmrs_sweep_opts {
    /* FP32 filter -> f64 exact recheck. A candidate is rechecked in the
     * reference's f64 arithmetic when its FP32 distance is <=
     * d32_min * (1 + shortlist_rel) + shortlist_abs * Rmax, Rmax being the
     * unit's largest centred coordinate magnitude. <= 0 selects the defaults
     * (2e-6 and 2e-6, twice the analysed FP32 error bound, DESIGN.md §4).    */
    double shortlist_rel;
    double shortlist_abs;
    int32_t shortlist_cap; /* AVERAGE recheck budget per unit (<= 0 selects 64): the units
                              share one pool of max(n_units * shortlist_cap, 65536)
                              items, a single unit may take any share of it. A unit
                              that does not fit is rechecked over ALL its candidates
                              in f64 (MMRS_FLAG_FULL_F64).                        */
    /* n_ties = 1 + number of OTHER rechecked candidates whose f64 distance is
     * <= best + tie_margin * max(1, Rmax) and whose wrapped angle differs from
     * the winner's (same-angle duplicates, e.g. -pi / +pi, are not ambiguous).
     * 0 = exact ties only.                                                    */
    double tie_margin;
    int32_t keep_dist32; /* != 0: the caller wants the exact FP32 distance of EVERY candidate from
                            mmrs_sweep_get_dist32 (tests, diagnostics): with prefilter == 0
                            (auto) this selects the dense FP32 sweep.                     */
    /* Tensor-core prefilter tier (tcgen05, bf16x3 split operands, FP32 accumulation in TMEM): every
     * candidate is first scored on the tensor cores with FP32-level (not bf16-level) error; only the
     * candidates with d_tc^2 <= d_tc_min^2 + prefilter_abs * Rmax^2 are re-scored by the exact FP32
     * kernel, and from there the FP32 window / f64 recheck / arg-min are unchanged, so the selected
     * candidate and its f64 distance are identical to the dense path. With the prefilter,
     * mmrs_sweep_get_dist32 returns prefilter-quality values (|error| <~ 1e-6 * Rmax^2 / d on d) for
     * candidates outside that window and exact FP32 values inside it.
     * 0 = auto, 1 = off (dense FP32 sweep of every candidate), 2 = required (every unit must have
     * 64..2048 points per set). Auto currently resolves to OFF: measured on B200 the prefilter kernel
     * is slower than the dense FP32 sweep (DESIGN.md §4), so it is an opt-in experimental tier.   */
    int32_t prefilter;
    double prefilter_abs; /* <= 0 selects 4e-6 (about 7x the largest error measured, DESIGN.md §4) */
    /* Exact lower-bound pruning (opt-in): before the FP32 sweep every candidate gets the lower bound
     *   LB = max( max_{a in A'} min_{b in B} |a-b| , max_{b in B'} min_{a in A} |a-b| ) <= Hausdorff(A, B)
     * over 32 (128 for sets of >= 1024 points) sampled points A', B' of the two sets; the candidate with the smallest
     * bound is scored exactly, and only candidates whose bound does not exceed that distance (plus twice the
     * FP32 window) are scored by the FP32 kernel — the others cannot be the arg-min. Selection, angle and f64
     * distance are identical to the dense path; mmrs_sweep_get_dist32 then returns the BOUND for pruned
     * candidates. > 0 on, < 0 off, 0 = the context default (mmrs_ctx_set_prune; off unless set). Applies when
     * every unit has >= 128 points per set and the batch averages >= 256 candidates per unit.        */
    int32_t prune;
    /* Partition of this batch across the ranks of the context (mmrs_ctx_comm_init / mmrs_ctx_set_shard):
     * 0 = the context's axis (mmrs_ctx_set_partition; whole units unless set), -1 = not partitioned (every rank
     * sweeps the whole batch by itself: no collective is issued for it), 1 = whole units, 2 = candidate angles. */
    int32_t partition;
} mmrs_sweep_opts;

#define MMRS_FLAG_DEGENERATE 1 /* grid degenerate: best_angle = fallback, nothing evaluated */
#define MMRS_FLAG_FULL_F64 2   /* recheck pool exhausted: all candidates rechecked in f64   */
#define MMRS_FLAG_EMPTY 4      /* empty point set: every candidate costs 0.0 (ref :86-88)   */

typedef struct mmrs_unit_result {
    int64_t best_idx;     /* leftmost arg-min in f64 (reference semantics); -1 if degenerate */
    double best_angle;    /* wrapped angle of best_idx (what search_range returns)           */
    double best_dist;     /* f64 Hausdorff distance at best_idx, reference arithmetic        */
    float best_dist_f32;  /* FP32 sweep minimum (before the recheck)                         */
    int32_t n_shortlist;  /* candidates rechecked in f64                                     */
    int32_t n_ties;       /* 1 + distinct-angle candidates within tie_margin of best         */
    int32_t flags;
} mmrs_unit_result;

/* Host buffers in, host results out: H2D, sweep, recheck, arg-min, D2H.      */
int mmrs_sweep_batched(mmrs_ctx* ctx, const mmrs_sweep_batch* batch, const mmrs_sweep_opts* opts,
                       mmrs_unit_result* out /* [n_units] */);

/* The same in three steps, so a caller can keep inputs resident in HBM:
 * upload (H2D + layout), run (all kernels; results stay on the device),
 * download (D2H of the n_units results).                                     */
int mmrs_sweep_upload(mmrs_ctx* ctx, const mmrs_sweep_batch* batch, const mmrs_sweep_opts* opts);
/* Keeps the uploaded points (and their device layout) and replaces only the candidate grids —
 * what the 2nd..4th window of find_best_rotation needs (align_within.rs:208-246): same point
 * sets, a new grid per unit centred on the previous window's result. A unit whose grid is
 * degenerate is skipped. */
int mmrs_sweep_regrid(mmrs_ctx* ctx, const mmrs_grid* grids, int64_t n_grids, const int32_t* grid_of_unit,
                      double tie_margin);
int mmrs_sweep_run(mmrs_ctx* ctx);
int mmrs_sweep_download(mmrs_ctx* ctx, mmrs_unit_result* out);

/* Launch plan of the uploaded batch. The units are grouped into size classes (register tile, chunked or not, exact
 * tiling or not) and the sweep kernel is launched once per class. For the class that carries most of the work:
 * [0] register tile TA (test points per lane of the sweep kernel), [1] bit 0: the test set is walked in several
 * register chunks, bit 1: exact tiling (32 TA points in register slots + a tail pass over the remaining n mod 32),
 * bit 2: the blocked kernel for units beyond the shared-memory staging (more than ~4 000 points per set),
 * [3] dynamic shared memory per CTA in bytes; [2] CTAs of all sweep launches, [4] number of size classes.   */
int mmrs_sweep_plan(mmrs_ctx* ctx, int64_t plan_out[5]);

/* Diagnostics on the last run (valid until the next upload).                 */
/* FP32 distance of every candidate of `unit` (needs opts.keep_dist32). After a
 * rigid run, in flattened candidate order c = i*T + j (see mmrs_tgrid).      */
int mmrs_sweep_get_dist32(mmrs_ctx* ctx, int64_t unit, float* out, int64_t cap);
/* Rechecked candidates of `unit`: indices and their f64 distances (flattened
 * candidate indices c = i*T + j after a rigid run).                          */
int mmrs_sweep_get_shortlist(mmrs_ctx* ctx, int64_t unit, int64_t* idx_out, double* dist_out, int32_t cap,
                             int32_t* n_out);
/* Device time of the last run in ms: [0] FP32 sweep kernel, [1] shortlist,
 * [2] f64 recheck + select, [3] whole run. Kernel launches of the last run.   */
int mmrs_last_timings(mmrs_ctx* ctx, float ms_out[4], int32_t* launches_out);

/* Context-wide default of mmrs_sweep_opts.prune (used by mmrs_process_cases and every sweep whose opts leave it 0). */
int mmrs_ctx_set_prune(mmrs_ctx* ctx, int32_t on);

/* For a pruned run (out[0] == 2): [1] bound passes + first exact score in ms, [2] survivor selection + exact FP32
 * scoring in ms, [3] candidates scored exactly (survivors, all units).
 * Tensor-core prefilter of the last run: [0] 1 if it ran, [1] K1t device time in ms, [2] tier-1 window +
 * tier-2 exact FP32 re-scoring time in ms, [3] candidates re-scored in FP32 (all units), [4] largest observed
 * |d_tc^2 - d_fp32^2| / Rmax^2 over them, [5] the window prefilter_abs in force.
 * When no tier ran ([0] == 0) and the dense sweep ran the early-break kernel K1e: [3] pair distances it evaluated,
 * [4] candidates it scored (divide for pairs per candidate; K1 evaluates N M).                                */
int mmrs_sweep_prefilter_info(mmrs_ctx* ctx, double out[6]);

/* Reference-arithmetic f64 cost of an explicit list of angles for one unit
 * (the cost closure itself; used by the host to resolve tie sets on the
 * sequential frame chain).                                                   */
int mmrs_eval_exact(mmrs_ctx* ctx, const double* test_xy, int64_t n_test, const double* ref_xy, int64_t n_ref,
                    double cx, double cy, int32_t mode, const double* angles, int64_t n_angles, double* dist_out);

/* Pure-FFMA FP32 throughput probe (denominator check for the roofline): runs
 * `iters` dependent FFMA chains on every SM, returns achieved TFLOP/s.        */
int mmrs_fp32_probe(mmrs_ctx* ctx, int32_t iters, double* tflops_out);

/* ---- rigid candidates: rotation grid x translation grid (opt-in) -------------------------------------------
 * Searches the best rigid transform (theta, tx, ty) instead of the best theta about a fixed offset. The reference
 * has no counterpart (it always aligns centroids, align_within.rs:84-90, align_between.rs:33-40); the semantics
 * below are this library's own and are restated by the test oracle.
 *
 * Translation grid: T = (2 half_n + 1)^2 offsets; translation j = jy (2 half_n + 1) + jx, jx, jy in [0, 2 half_n],
 *   tx = t0x + (double)(jx - half_n) * step,   ty = t0y + (double)(jy - half_n) * step   (host f64, as written).
 * Candidate c = i T + j: angle i of the unit's mmrs_grid, translation j of its mmrs_tgrid. With half_n = 0 and
 * t0 = (0, 0), c == i.
 * Cost (f64): the rotation of the batch's mode (0 / 1, same operation order, same angle == 0.0 identity in mode 0,
 *   same host cos / sin), then x' = rx + tx, y' = ry + ty (one rounding each; + 0.0 is exact, so a zero translation
 *   gives the rotation-only cost bit for bit), then hausdorff_distance(reference, transformed).
 * Selection: leftmost arg-min over c (strict <): ties go to the lowest angle index, then the lowest jy, then jx.
 * n_ties: 1 + rechecked candidates within tie_margin * max(1, R_eff) whose TRANSFORM differs from the winner's
 *   (a different (cos, sin) or a different (tx, ty)); R_eff = Rmax + max_j |t_j| replaces Rmax in the FP32
 *   shortlist window as well.
 * Execution: the dense FP32 sweep on this context's device alone (no lower-bound pruning, no prefilter tier, no
 * partition across ranks: a bound communicator or shard transport is not used). opts.prune > 0 or
 * opts.prefilter 2 / 3 is an error; the context's prune default is ignored.
 * Edge cases: degenerate angle grid -> best_idx = -1, best_angle = fallback, angle_idx = trans_idx = -1,
 *   (best_tx, best_ty) = (t0x, t0y); an empty set -> every candidate costs 0, candidate 0 wins; non-finite points
 *   are dropped as in the rotation-only sweep. half_n < 0, a non-finite t0 / step, step <= 0 with half_n > 0, or
 *   more than INT32_MAX candidates (angles x translations) in one unit is MMRS_ERR_ARG.                     */
typedef struct mmrs_tgrid {
    double t0x, t0y; /* centre of the grid                 */
    double step;     /* spacing (same unit as the points)  */
    int32_t half_n;  /* 2 half_n + 1 offsets per axis      */
} mmrs_tgrid;

typedef struct mmrs_rigid_result {
    mmrs_unit_result r;  /* r.best_idx = flattened candidate index, r.best_angle = its (wrapped) angle */
    int64_t angle_idx;   /* best_idx / T (-1 if degenerate)                                          */
    int32_t trans_idx;   /* best_idx % T (-1 if degenerate)                                          */
    int32_t pad;
    double best_tx, best_ty;
} mmrs_rigid_result;

/* mmrs_sweep_batched with a translation grid per unit: `tgrid_of_unit` == NULL -> every unit uses tgrids[0]. */
int mmrs_rigid_sweep_batched(mmrs_ctx* ctx, const mmrs_sweep_batch* batch, const mmrs_tgrid* tgrids, int64_t n_tgrids,
                             const int32_t* tgrid_of_unit, const mmrs_sweep_opts* opts, mmrs_rigid_result* out);
/* The same in steps: upload, regrid (new angle and translation grids on the uploaded points), mmrs_sweep_run,
 * download. mmrs_sweep_download after a rigid run returns the mmrs_unit_result part.                          */
int mmrs_rigid_sweep_upload(mmrs_ctx* ctx, const mmrs_sweep_batch* batch, const mmrs_tgrid* tgrids, int64_t n_tgrids,
                            const int32_t* tgrid_of_unit, const mmrs_sweep_opts* opts);
int mmrs_rigid_sweep_regrid(mmrs_ctx* ctx, const mmrs_grid* grids, int64_t n_grids, const int32_t* grid_of_unit,
                            const mmrs_tgrid* tgrids, int64_t n_tgrids, const int32_t* tgrid_of_unit, double tie_margin);
int mmrs_rigid_sweep_download(mmrs_ctx* ctx, mmrs_rigid_result* out);
/* f64 cost of explicit rigid candidates k = (angles[k], txy[2k], txy[2k+1]) for one unit (mmrs_eval_exact plus the
 * translation).                                                                                                */
int mmrs_eval_exact_rigid(mmrs_ctx* ctx, const double* test_xy, int64_t n_test, const double* ref_xy, int64_t n_ref,
                          double cx, double cy, int32_t mode, const double* angles, const double* txy, int64_t n_cand,
                          double* dist_out);

/* ---- partial cost: rank-K Hausdorff distance, a set fraction of outlier points ignored (opt-in) ---------------
 * The symmetric Hausdorff distance is a maximum, so one artefact (a side-branch bulge, a calcification, a catheter
 * shadow) decides every candidate's cost. The partial distance (Huttenlocher, Klanderman and Rucklidge, IEEE TPAMI
 * 1993) takes, in each direction, the K-th smallest point minimum instead of the largest, so the worst n - K points
 * of each set do not count. Like the rigid candidates, this is this library's own extension, restated by the tests.
 *
 * One inlier_fraction f, finite, 0 < f <= 1, for both directions. For a set of n finite points (non-finite points
 *   are dropped, as everywhere): K(n) = max(1, ceil(f * n)) (host f64, as written); q(n) = n - K(n) points do not count.
 * Row value of a point p against a set Q: v(p) = min_{x in Q} d^2(p, x); a non-finite minimum counts as 0.
 * Directed partial value: the (q + 1)-th largest v(p) over the set, duplicates counted. Cost (f64):
 *   fmax(sqrt(fwd), sqrt(bwd)), fwd: the reference points against the transformed test set, q = q(m);
 *   bwd: the transformed test points against the reference set, q = q(n).
 * The transform (mode 0 / 1 rotation, plus the optional translation grid) and the selection (leftmost arg-min, tie
 *   margin, R_eff for rigid runs) are those of the rotation-only and rigid sweeps. f = 1 gives q = 0: today's cost.
 *   An empty set still costs 0.
 * Limits (MMRS_ERR_ARG, checked before any device work): q <= 255 per direction and unit; no unit beyond the
 *   shared-memory staging (more than ~4 000 points per set); opts.prune > 0 or opts.prefilter 2 / 3. The context's
 *   prune default and any partition across ranks are not used, as for rigid runs.
 * Exactness: the FP32 sweep computes each candidate's partial FP32 distance exactly (an early-break kernel whose
 *   threshold only holds exact minima of the current candidate); MMRS_EARLY_BREAK=0 at upload switches the early
 *   break off in the same kernel. The FP32 -> f64 window is that of the full cost.                               */

/* mmrs_sweep_upload (tgrids == NULL) or mmrs_rigid_sweep_upload with the partial cost. inlier_fraction == 1.0 is
 * exactly the plain upload with the same opts. The fraction stays with the uploaded points: mmrs_sweep_regrid /
 * mmrs_rigid_sweep_regrid, mmrs_sweep_run and the download calls work on it unchanged; a later plain upload clears it. */
int mmrs_partial_sweep_upload(mmrs_ctx* ctx, const mmrs_sweep_batch* batch, const mmrs_tgrid* tgrids /* NULL: rotation only */,
                              int64_t n_tgrids, const int32_t* tgrid_of_unit, double inlier_fraction,
                              const mmrs_sweep_opts* opts);
/* f64 partial cost of explicit candidates k = (angles[k], txy[2k], txy[2k+1]) for one unit (txy == NULL: no
 * translation), on the finite points of each set.                                                              */
int mmrs_eval_exact_partial(mmrs_ctx* ctx, const double* test_xy, int64_t n_test, const double* ref_xy, int64_t n_ref,
                            double cx, double cy, int32_t mode, const double* angles, const double* txy /* NULL: none */,
                            int64_t n_cand, double inlier_fraction, double* dist_out);

/* ---- mean cost: modified Hausdorff distance, every point's closest-point distance averaged (opt-in) ------------
 * Both costs above are decided by one or a few extreme points. The modified Hausdorff distance (Dubuisson and Jain,
 * ICPR 1994) averages each point's closest-point distance in each direction and takes the larger direction, so every
 * point counts and there is no parameter. Like the rigid and partial costs, this is this library's own extension,
 * restated by the tests.
 *
 * For a candidate: A, the n finite transformed test points; B, the m finite reference points (non-finite points are
 *   dropped, as everywhere).
 * Row value of a point p against a set Q: v(p) = sqrt(min_{x in Q} (dx*dx + dy*dy)), reference arithmetic (unfused,
 *   IEEE sqrt); a non-finite minimum counts as 0.
 * fwd = (v(b_0) + v(b_1) + ... + v(b_{m-1})) / m: a sequential left-to-right f64 sum in point order, then one
 *   division. bwd: the same over A against B, divided by n. Cost (f64): fmax(fwd, bwd). The summation order is part of
 *   the definition.
 * The transform (mode 0 / 1 rotation, plus the optional translation grid) and the selection (leftmost arg-min, tie
 *   margin, R_eff for rigid runs) are those of the rotation-only and rigid sweeps. An empty set costs 0
 *   (MMRS_FLAG_EMPTY).
 * Limits (MMRS_ERR_ARG, checked before any device work): no unit beyond the shared-memory staging (more than ~4 000
 *   points per set); opts.prune > 0 or opts.prefilter 2 / 3. The context's prune default and any partition across
 *   ranks are not used, as for rigid runs; MMRS_EARLY_BREAK does not apply (every pair is evaluated).
 * FP32 -> f64: the sweep's FP32 value of a candidate is within 5e-7 R + 3.6e-7 d of its f64 cost (R: Rmax, or R_eff
 *   for rigid runs), inside the FP32 window of the full cost, which is used unchanged.                             */

/* mmrs_sweep_upload (tgrids == NULL) or mmrs_rigid_sweep_upload with the mean cost. The cost stays with the uploaded
 * points: mmrs_sweep_regrid / mmrs_rigid_sweep_regrid, mmrs_sweep_run and the download calls work on it unchanged; a
 * later plain or partial upload clears it.                                                                        */
int mmrs_mean_sweep_upload(mmrs_ctx* ctx, const mmrs_sweep_batch* batch, const mmrs_tgrid* tgrids /* NULL: rotation only */,
                           int64_t n_tgrids, const int32_t* tgrid_of_unit, const mmrs_sweep_opts* opts);
/* f64 mean cost of explicit candidates k = (angles[k], txy[2k], txy[2k+1]) for one unit (txy == NULL: no
 * translation), on the finite points of each set.                                                              */
int mmrs_eval_exact_mean(mmrs_ctx* ctx, const double* test_xy, int64_t n_test, const double* ref_xy, int64_t n_ref,
                         double cx, double cy, int32_t mode, const double* angles, const double* txy /* NULL: none */,
                         int64_t n_cand, double* dist_out);

/* ---- geometry blob -------------------------------------------------------------
 * Geometries cross the boundary as one f64 stream (u32 ids are exact in f64):
 *   n_frames,
 *   per frame : id, cx, cy, cz, has_ref, ref{frame_index, point_index, x, y, z, aortic}, n_contours,
 *     per contour (lumen first, then extras by kind):
 *       kind, id, original_frame, has_centroid, cx, cy, cz,
 *       has_aortic_thickness, aortic_thickness, has_pulmonary_thickness, pulmonary_thickness, n_points,
 *       per point: frame_index, point_index, x, y, z, aortic
 * kind: 0 Lumen, 1 Eem, 2 Calcification, 3 Sidebranch, 4 Catheter, 5 Wall
 * (src/types/native/contour.rs:8-16). Mirrors Geometry/Frame/Contour/
 * ContourPoint of src/types/native/{geometry,frame,contour,contour_point}.rs.
 * Blobs returned by the library are malloc'ed; release with mmrs_free.        */
void mmrs_free(void* p);

/* AlignLog rows (align_within.rs:14-22 as emitted by logs_to_tuples,
 * binding/functions.rs:26-40): n x 7 doubles
 * (contour_id, matched_to, rot_deg, tx, ty, centroid_x, centroid_y).          */

/* Replaces `build_geometry_from_inputdata` (src/intravascular/io/build.rs:9-205)
 * for a directory (io/input.rs:62-147) ...                                    */
int mmrs_geometry_from_dir(mmrs_ctx* ctx, const char* path, const char* label, int diastole, double image_cx,
                           double image_cy, double radius, uint32_t n_points, double** blob_out, int64_t* len_out);
/* ... and for in-memory (N,4) [frame, x, y, z] arrays (PyInputData,
 * src/types/binding/py_input_data.rs:103-172). records: (R,4)
 * [frame, is_diastole, measurement_1, measurement_2], NaN = missing; any array
 * pointer may be NULL except lumen and ref_point[4].                          */
int mmrs_geometry_from_arrays(mmrs_ctx* ctx, const double* lumen, int64_t n_lumen, const double* eem, int64_t n_eem,
                              const double* calc, int64_t n_calc, const double* side, int64_t n_side,
                              const double* records, int64_t n_rec, const double* ref_point, int diastole,
                              const char* label, double image_cx, double image_cy, double radius, uint32_t n_points,
                              double** blob_out, int64_t* len_out);

typedef struct mmrs_align_params {
    double step_deg;      /* step_rotation_deg  */
    double range_deg;     /* range_rotation_deg */
    int64_t sample_size;
    int32_t smooth;
    int32_t bruteforce;
    int32_t postprocessing; /* != 0: postprocess_geom_pair on every pair (modes 2-4),
                               src/intravascular/processing/postprocessing.rs:12-87, tolerance 0.03 mm
                               (binding/entry.rs:21) */
} mmrs_align_params;

/* Replaces the *_processing_rs orchestration of
 * src/intravascular/binding/entry.rs for a batch of `n_cases` independent
 * cases (patients): mode 4 = full_processing_rs (:71-361), 3 =
 * double_pair_processing_rs (:363-570), 2 = pair_processing_rs (:572-689),
 * 1 = single_processing_rs (:691-780); each with write_obj = false (the OBJ / MTL / PNG
 * export is a separate call: mmrs_export_pair / mmrs_export_single below). Input: n_cases *
 * n_in(mode) geometry blobs (n_in = 4,4,2,1). Output: n_cases * n_out(mode)
 * blobs (8,4,2,1: pair ab = (a,b), cd, ac, bd) and n_cases * n_in log arrays.
 * All intrapullback sweeps of all cases run as ONE batch per search stage, all
 * inter-pullback sweeps of a dependency level likewise.
 * Ownership: every output slot is set to NULL / 0 on entry; on success the caller owns the malloc'ed blobs and
 * log arrays (mmrs_free); on a non-zero return everything written so far has been released and the slots are NULL. */
int mmrs_process_cases(mmrs_ctx* ctx, int32_t mode, int64_t n_cases, const double* const* blobs,
                       const int64_t* blob_lens, const mmrs_align_params* params, double** out_blobs,
                       int64_t* out_lens, double** out_logs, int64_t* out_nlogs, int32_t* out_anomalous);

/* ---- OBJ / MTL / texture export ---------------------------------------------------------------
 * Replaces to_object::process_case (src/intravascular/to_object/process.rs:9-61: interpolation
 * between the two geometries, to_object/interpolation.rs:9-157; one texture PNG + MTL per mesh,
 * to_object/write_mtl.rs:15-273 and to_object/texture.rs:6-95; one OBJ per mesh,
 * io/output.rs:10-181, :245-307) for one geometry pair. File names, OBJ/MTL text and texture
 * pixels follow the reference; the PNG files use stored (uncompressed) deflate blocks.
 * kinds: contour kinds to write, in order (0 Lumen ... 5 Wall). label_a names the interpolated
 * geometries ("{label_a}_inter_{k}"). ctx may be NULL (no GPU work).                          */
int mmrs_export_pair(mmrs_ctx* ctx, const double* blob_a, int64_t len_a, const double* blob_b, int64_t len_b,
                     const char* label_a, const char* case_name, const char* output_dir, int64_t interpolation_steps,
                     int32_t watertight, const int32_t* kinds, int32_t n_kinds);
/* One geometry, no UV coordinates. naming 0: the export of single_processing_rs
 * (binding/entry.rs:741-818, files "{type}_{name}.obj/.mtl"); naming 1:
 * to_object::write_single_geometry (process.rs:63-121, files "{name}_{type}.obj/.mtl"); naming 2: the to_obj
 * entry point (binding/functions.rs:1435-1501, files "{name}_{type}" or, for an empty name, "{type}").        */
int mmrs_export_single(mmrs_ctx* ctx, const double* blob, int64_t len, const char* name, const char* output_dir,
                       int32_t watertight, const int32_t* kinds, int32_t n_kinds, int32_t naming);

/* ---- value-type helpers (host only, no context) --------------------------------------------------
 * Contour::area, find_farthest_points, find_closest_opposite, find_closest_opposite_3d
 * (src/types/native/contour.rs:227-363; behind PyContour.get_area / find_farthest_points / find_closest_opposite /
 * get_elliptic_ratio, src/types/binding/py_contour.rs:144-213) on n packed (x, y, z) points. `centroid` = the
 * contour's stored centroid (has_centroid != 0) — otherwise the mean of the points, like the reference.
 * out[8] = { area, farthest_i, farthest_j, farthest_dist, opposite_i, opposite_j, opposite_dist_2d,
 * opposite_dist_3d }; entries that the reference refuses for this n (n <= 2 for the opposite searches, n == 0 for
 * the farthest pair) are NaN.                                                                        */
int mmrs_contour_metrics(const double* xyz, int64_t n, int32_t has_centroid, const double* centroid, double out[8]);

/* ---- centerline alignment ----------------------------------------------------------------------
 * Replaces align_three_point_rs / align_manual_rs / align_combined_rs
 * (src/intravascular/centerline_align/align.rs:61-121, :123-164, :166-283; PyO3 wrappers in
 * src/intravascular/binding/align.rs:65-155, :199-284, :334-463) without the `write` step (call
 * mmrs_export_pair / mmrs_export_single with naming 1 afterwards).
 *   method 0: three-point search (align_algorithms.rs:264-337) — 3-point squared error, not
 *             Hausdorff-scored, host f64;
 *   method 1: manual rotation (`manual_rotation_deg`, reference point in main_ref_pt);
 *   method 2: three-point search + refine_alignment_hausdorff (align_algorithms.rs:339-451):
 *             every (centerline index, angle) candidate is scored by the symmetric Hausdorff
 *             distance on the GPU as one batch of sweep units (needs ctx; no CPU fallback).
 * centerline: n_cl rows of 8 doubles (x, y, z, tangent_x, tangent_y, tangent_z, branch_id, radius)
 * (CenterlinePoint, src/types/native/centerline_point.rs:4-11). n_geoms: 1 (Geometry) or 2
 * (GeometryPair: the first blob is the primary geometry). Outputs: n_geoms malloc'ed blobs,
 * the resampling spacing in mm, the total rotation in radians, and refine_out[2] =
 * (best Hausdorff distance, candidates scored) for method 2 (-1, 0 otherwise).                */
typedef struct mmrs_centerline_params {
    double main_ref_pt[3];
    double ccw_ref_pt[3];
    double cw_ref_pt[3];
    double angle_step_rad;
    double manual_rotation_deg;
    const double* points; /* method 2: CCTA point cloud, n_points x (x, y, z) */
    int64_t n_points;
    double angle_range_rad;
    int64_t index_range;
    int32_t align_wall_anomalous;
} mmrs_centerline_params;
int mmrs_align_centerline(mmrs_ctx* ctx, int32_t method, const double* centerline, int64_t n_cl, int32_t n_geoms,
                          const double* const* blobs, const int64_t* blob_lens, const mmrs_centerline_params* params,
                          double** out_blobs, int64_t* out_lens, double* spacing_out, double* rotation_rad_out,
                          double* refine_out);

/* ---- multi-GPU: one process per GPU, every batched sweep partitioned across the ranks ------------------------
 * The path shards on independent work (the reference runs candidates, and whole pullbacks, concurrently:
 * process_utils.rs:69-74, binding/entry.rs:140-277). Every rank issues the same sweep calls with the same batch;
 * each rank's GPU evaluates only its part and the per-unit results are merged so that every rank downloads the
 * complete, identical result array:
 *   axis 1 (default) whole UNITS: cost-balanced contiguous blocks of the units; merged with ONE all-reduce(SUM) over the
 *          32-byte device results per run (entries of other ranks are zero, so the sum is an exact merge);
 *   axis 2 CANDIDATE ANGLES: every unit's grid is cut into `world` contiguous sub-ranges (global candidate indices
 *          kept). After the FP32 sweep the packed (distance, index) keys are merged with all-reduce(MIN, uint64) —
 *          the reduction of process_utils.rs:69-74: lowest distance, ties -> lowest index — so every rank shortlists
 *          its sub-range against the GLOBAL FP32 minimum; the local f64 winners are all-gathered (32 B per unit and
 *          rank), the global leftmost f64 arg-min is taken and the tie counts are summed. For single-frame sweeps.
 * With a communicator bound (mmrs_ctx_comm_init) the collectives are NCCL calls on device buffers on the context's
 * stream, between the kernels of a run. mmrs_ctx_set_shard binds a host callback instead (axis 1 only).
 * The context's default (axis 1 with `partition` left 0 in the opts) is a policy decided from the batch shape alone,
 * identically on every rank: whole units where they balance; candidate sub-ranges (axis 2, communicator bound, every
 * unit >= 64 candidates per rank) where a few large units cannot be dealt evenly (block cost > 1.25 x the mean: the
 * inter-pullback stages); NO partition (no collective, every rank sweeps the batch) below 2e9 pair evaluations.
 * An explicit `partition` of 1, 2 or -1 in the opts overrides the policy.
 *
 * mmrs_comm_unique_id: rank 0 creates the rendezvous token (ncclGetUniqueId) and hands it to the other ranks by any
 * means (MPI, torch.distributed, a file); mmrs_ctx_comm_init is collective (ncclCommInitRank on the context's device).
 * NCCL is bound at run time (dlopen); both calls fail with MMRS_ERR_STATE where libnccl.so.2 is absent.          */
#define MMRS_COMM_ID_BYTES 128
int mmrs_comm_unique_id(uint8_t id_out[MMRS_COMM_ID_BYTES]);
int mmrs_ctx_comm_init(mmrs_ctx* ctx, const uint8_t id[MMRS_COMM_ID_BYTES], int32_t rank, int32_t world);
/* Axis used by batches whose opts leave `partition` 0: 1 whole units (default), 2 candidate angles, 0 none. */
int mmrs_ctx_set_partition(mmrs_ctx* ctx, int32_t axis);
/* rank / world / axis of the context: out[0..2]; out[3] = 1 when an NCCL communicator is bound. */
int mmrs_ctx_comm_info(const mmrs_ctx* ctx, int32_t out[4]);

/* ---- the same with a host callback as the transport (e.g. gloo, MPI) ---------------------------------------------
 * Axis 1 only. The per-unit results (32 B each, 4 int64 words) are combined at download with `exchange`, an in-place
 * all-reduce(SUM) over int64 words across ranks (non-owned entries are zero, so the sum is an exact merge; the host
 * binds it to MPI_Allreduce / torch.distributed.all_reduce over gloo, ...). world <= 1 or fn == NULL switches it off.
 * A communicator bound with mmrs_ctx_comm_init takes precedence.                                            */
typedef int (*mmrs_exchange_fn)(void* user, int64_t* buf, int64_t n_words);
int mmrs_ctx_set_shard(mmrs_ctx* ctx, int32_t rank, int32_t world, mmrs_exchange_fn fn, void* user);

/* Counters of the last mmrs_process_cases call: [0] units swept, [1] candidate
 * evaluations (FP32), [2] f64 rechecks, [3] units resolved on the sequential
 * chain (tie sets), [4] kernel launches.                                      */
int mmrs_process_stats(mmrs_ctx* ctx, int64_t stats_out[5]);

#ifdef __cplusplus
}
#endif
#endif /* MMRS_B200_H */
