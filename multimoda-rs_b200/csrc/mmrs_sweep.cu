// =============================================================================
// mmrs_sweep.cu — context, device workspaces and the sweep entry points of the
// C ABI declared in include/mmrs_b200.h. No CPU fallback: every compute entry
// point needs a CUDA device that can run the sm_100a image.
// =============================================================================
#include "mmrs_internal.hpp"
#include "mmrs_comm.hpp"
#include "mmrs_pool.hpp"
#include "sweep_kernels.cuh"
#include "tc_kernels.cuh"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

using namespace mmrs;

static thread_local std::string g_err_noctx = "";

#define CUDA_TRY(ctx, expr)                                                                       \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            return set_err(ctx, MMRS_ERR_CUDA,                                                    \
                           std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" __FILE__ ":" + \
                               std::to_string(__LINE__) + ")");                                   \
        }                                                                                         \
    } while (0)

// Every entry point runs on the context's device and leaves the caller's current device as it found it (a host that
// manages several GPUs itself, e.g. a PyTorch process, must not have its later launches redirected).
struct DeviceGuard {
    int prev = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int device) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != device) err = cudaSetDevice(device);
        else prev = -1;   // nothing to restore
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};
#define ENTER_DEVICE(ctx)                  \
    DeviceGuard _device_guard((ctx)->device); \
    CUDA_TRY(ctx, _device_guard.err)

int mmrs::set_err(mmrs_ctx* ctx, int code, const std::string& msg) {
    if (ctx)
        ctx->err = msg;
    else
        g_err_noctx = msg;
    return code;
}

// ---- reference grid arithmetic (process_utils.rs:43-67) -------------------------
static const double kPi = 3.14159265358979323846264338327950288;
static inline double to_radians(double d) { return d * (kPi / 180.0); }
static inline double rem_euclid(double a, double b) {
    double r = std::fmod(a, b);
    return (r < 0.0) ? r + std::fabs(b) : r;
}
static inline uint64_t f64_as_usize(double v) {
    if (!(v == v) || v <= 0.0) return 0;
    if (v >= 18446744073709551615.0) return ~0ull;
    return (uint64_t)v;
}

extern "C" int mmrs_grid_from_reference_params(double step_deg, double range_deg, int has_center, double center_rad,
                                               double limes_deg, mmrs_grid* out) {
    if (!out) return set_err(nullptr, MMRS_ERR_ARG, "mmrs_grid_from_reference_params: out is NULL");
    mmrs_grid g{};
    const double range_rad = to_radians(range_deg), step_rad = to_radians(step_deg);
    const double center = has_center ? center_rad : 0.0;
    g.step_rad = step_rad;
    g.fallback = center;
    if (step_rad <= 0.0) {
        g.degenerate = 1;
        *out = g;
        return MMRS_OK;
    }
    const double limes = to_radians(limes_deg);
    const double start = std::fmax(center - range_rad, -limes);
    const double stop = std::fmin(center + range_rad, limes);
    g.start_rad = start;
    if (stop <= start) {
        g.degenerate = 1;
        *out = g;
        return MMRS_OK;
    }
    uint64_t steps = std::max<uint64_t>(f64_as_usize(std::ceil((stop - start) / step_rad)), 1);
    if (steps > (1ull << 31) - 2) return set_err(nullptr, MMRS_ERR_ARG, "grid has more than 2^31 candidates");
    // take_while(a <= stop): candidates are increasing in i, so the count is the first failing i.
    int64_t n = 0;
    for (uint64_t i = 0; i <= steps; ++i) {
        const double a = start + (double)i * step_rad;
        if (!(a <= stop)) break;
        ++n;
    }
    g.n_cand = n;
    if (n == 0) g.degenerate = 1;  // .unwrap_or(center)
    *out = g;
    return MMRS_OK;
}

extern "C" double mmrs_grid_angle(const mmrs_grid* g, int64_t i) {
    const double a = g->start_rad + (double)i * g->step_rad;
    return rem_euclid(a + kPi, 2.0 * kPi) - kPi;
}

extern "C" int mmrs_stage_plan(double step_deg, double range_deg, double step_out[4], double window_out[4]) {
    // align_within.rs:208-246 match arms: 1.0..=INF | 0.1..1.0 | 0.01..0.1 | _
    const double r5 = (range_deg > 5.0) ? 5.0 : range_deg;
    const double r10s = (range_deg > 10.0 * step_deg) ? 10.0 * step_deg : range_deg;
    if (step_deg >= 1.0) {
        step_out[0] = step_deg, window_out[0] = range_deg;
        return 1;
    }
    step_out[0] = 1.0, window_out[0] = range_deg;
    if (step_deg >= 0.1 && step_deg < 1.0) {
        step_out[1] = step_deg, window_out[1] = r5;
        return 2;
    }
    step_out[1] = 0.1, window_out[1] = r5;
    if (step_deg >= 0.01 && step_deg < 0.1) {
        step_out[2] = step_deg, window_out[2] = r10s;
        return 3;
    }
    step_out[2] = 0.01, window_out[2] = (range_deg > 0.1) ? 0.1 : range_deg;
    step_out[3] = step_deg, window_out[3] = r10s;
    return 4;
}

// ---- context -----------------------------------------------------------------------
extern "C" const char* mmrs_version(void) { return "mmrs_b200 0.1.0 (sm_100a)"; }

extern "C" const char* mmrs_last_error(const mmrs_ctx* ctx) { return ctx ? ctx->err.c_str() : g_err_noctx.c_str(); }

extern "C" int mmrs_ctx_create(int device, void* stream, mmrs_ctx** out) {
    if (!out) return set_err(nullptr, MMRS_ERR_ARG, "mmrs_ctx_create: out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return set_err(nullptr, MMRS_ERR_CUDA,
                       std::string("no CUDA device available (") + cudaGetErrorString(e) +
                           "); this library has no CPU fallback");
    if (device < 0 || device >= n) return set_err(nullptr, MMRS_ERR_ARG, "mmrs_ctx_create: bad device index");
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return set_err(nullptr, MMRS_ERR_CUDA, cudaGetErrorString(e));
    if (prop.major != 10)
        return set_err(nullptr, MMRS_ERR_CUDA,
                       "device compute capability " + std::to_string(prop.major) + "." + std::to_string(prop.minor) +
                           " cannot run the sm_100a image (B200 required); no fallback path exists");
    mmrs_ctx* ctx = new mmrs_ctx();
    ctx->device = device;
    ctx->n_sm = prop.multiProcessorCount;
    ctx->sm_clock_khz = prop.clockRate;
    DeviceGuard guard(device);
    if (stream) {
        ctx->stream = (cudaStream_t)stream;
        ctx->own_stream = false;
    } else {
        e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            delete ctx;
            return set_err(nullptr, MMRS_ERR_CUDA, cudaGetErrorString(e));
        }
        ctx->own_stream = true;
    }
    bool ev_ok = true;
    for (auto& ev : ctx->ev) ev_ok = ev_ok && cudaEventCreate(&ev) == cudaSuccess;
    for (auto& ev : ctx->ev_tc) ev_ok = ev_ok && cudaEventCreate(&ev) == cudaSuccess;
    if (!ev_ok) {
        const std::string msg = std::string("cudaEventCreate: ") + cudaGetErrorString(cudaGetLastError());
        mmrs_ctx_destroy(ctx);
        return set_err(nullptr, MMRS_ERR_CUDA, msg);
    }
    *out = ctx;
    return MMRS_OK;
}

extern "C" void mmrs_ctx_destroy(mmrs_ctx* ctx) {
    if (!ctx) return;
    DeviceGuard guard(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->comm && nccl_api().ok()) nccl_api().CommDestroy(ctx->comm);
    ctx->comm = nullptr;
    ctx->free_all();
    for (auto& ev : ctx->ev)
        if (ev) cudaEventDestroy(ev);
    for (auto& ev : ctx->ev_tc)
        if (ev) cudaEventDestroy(ev);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

void mmrs_ctx::free_all() {
    for (DevBuf* b : {&d_test, &d_ref, &d_units, &d_work, &d_lay, &d_cs64, &d_cs32, &d_zero, &d_dist32, &d_key,
                      &d_rmax, &d_sl_base, &d_sl_dist, &d_sl_count, &d_items, &d_nitems, &d_res, &d_tmp, &d_work_tc,
                      &d_key_tc, &d_l1_items, &d_l1_count, &d_l1_base, &d_l1_n, &d_units_lb, &d_lay_lb,
                      &d_work_lb, &d_res_all, &d_cnt, &d_bcast, &d_big_rows, &d_exact_scratch, &d_eb_pairs}) {
        if (b->p) cudaFree(b->p);
        b->p = nullptr;
        b->cap = 0;
    }
    if (h_res) cudaFreeHost(h_res);
    h_res = nullptr;
    h_res_cap = 0;
}

static int ensure(mmrs_ctx* ctx, DevBuf& b, size_t bytes) {
    if (bytes <= b.cap) return MMRS_OK;
    if (b.p) {
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        CUDA_TRY(ctx, cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    size_t want = bytes + bytes / 4 + 256;
    CUDA_TRY(ctx, cudaMalloc(&b.p, want));
    b.cap = want;
    return MMRS_OK;
}
#define ENSURE(buf, bytes)                                 \
    do {                                                   \
        int _r = ensure(ctx, buf, (size_t)(bytes));        \
        if (_r != MMRS_OK) return _r;                      \
    } while (0)

constexpr bool kXfDefault = false;   // what mmrs_sweep_opts.prefilter = 0 (auto) resolves to for large batches

// Early-break dense sweep K1e (k_sweep_eb). A warp walks a contiguous run of candidates and carries its hints from one
// candidate to the next. Measured on B200 (profiles/r03_early_break_bench.json) it beats K1 on every grid tried, from
// 0.01 deg (7.3x) to 1 deg steps (1.05x) and 41-candidate sweeps (1.9x), so the rule is only that a CTA fits 3 per SM.
constexpr size_t kEbAutoSmem = 72 * 1024;
constexpr long long kEbMinRun = 32, kEbMaxRun = 256;   // candidates per warp run

// ---- kernel dispatch over TA ----------------------------------------------------------
struct ListArgs {  // LIST arguments of k_sweep; all null for the dense sweep
    const int2* items = nullptr;
    const unsigned* n_items = nullptr;  // device counter: items in the global list
    unsigned cap = 0;                   // capacity of the list (upper bound of *n_items)
    int chunk = 64;                     // list positions per CTA
    const unsigned* rmax = nullptr;
    unsigned* diag = nullptr;
};
// The dynamic shared-memory limit is per-FUNCTION state shared by every host thread and context on the device, so it is
// raised ONCE per instantiation to the 227 KB opt-in maximum and never lowered (several contexts may launch the same
// instantiation with different sizes from different threads: process_cases_pipelined).
constexpr int kMaxDynSmem = 227 * 1024;
template <class K>
static cudaError_t raise_smem_once(K kernel, std::once_flag& once, cudaError_t& result) {
    std::call_once(once, [&] { result = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynSmem); });
    return result;
}
#define RAISE_SMEM(kernel)                                       \
    ([&]() -> cudaError_t {                                      \
        static std::once_flag once;                              \
        static cudaError_t result = cudaSuccess;                 \
        return raise_smem_once(kernel, once, result);            \
    }())

template <int TA, bool MULTI, bool LIST, bool TAILP, bool XF, bool RIGID = false, bool MEAN = false>
static void launch_sweep_k(int grid, size_t smem, cudaStream_t s, const UnitDesc* units, const WorkItem* work,
                           const float4* lay, const float2* cs32, float* dist32, unsigned long long* key,
                           const ListArgs& l, const float2* t32 = nullptr) {
    RAISE_SMEM((k_sweep<TA, MULTI, LIST, TAILP, XF, RIGID, MEAN>));
    k_sweep<TA, MULTI, LIST, TAILP, XF, RIGID, MEAN><<<grid, kThreads, smem, s>>>(
        units, work, lay, cs32, dist32, key, l.items, l.n_items, l.cap, l.chunk, l.rmax, l.diag, t32);
}
// xf: the expanded-form tier K1x (dense launches only; a list is always re-scored in direct form)
// t32 != NULL: rigid candidates (dense direct-form launches only)
// mean: the mean cost (dense direct-form launches only, rotation only or rigid)
template <int TA>
static void launch_sweep_ta(bool multi, bool tailp, bool xf, int grid, size_t smem, cudaStream_t s, const UnitDesc* units,
                            const WorkItem* work, const float4* lay, const float2* cs32, float* dist32,
                            unsigned long long* key, const ListArgs* l, const float2* t32, bool mean) {
    const ListArgs none{};
    const ListArgs& la = l ? *l : none;
#define GO(M, L, T, X) launch_sweep_k<TA, M, L, T, X>(grid, smem, s, units, work, lay, cs32, dist32, key, la)
#define GO_RIGID(M, T) launch_sweep_k<TA, M, false, T, false, true>(grid, smem, s, units, work, lay, cs32, dist32, key, la, t32)
#define GO_MEAN(M, T, R) launch_sweep_k<TA, M, false, T, false, R, true>(grid, smem, s, units, work, lay, cs32, dist32, key, la, t32)
    if (mean) {
        if constexpr (TA % 2 == 0 && TA >= 4) {
            if (tailp) {
                if (t32) GO_MEAN(false, true, true);
                else GO_MEAN(false, true, false);
                return;
            }
        }
        if (multi) {
            if (t32) GO_MEAN(true, false, true);
            else GO_MEAN(true, false, false);
        } else {
            if (t32) GO_MEAN(false, false, true);
            else GO_MEAN(false, false, false);
        }
        return;
    }
    if (t32) {
        if constexpr (TA % 2 == 0 && TA >= 4) {
            if (tailp) {
                GO_RIGID(false, true);
                return;
            }
        }
        if (multi) GO_RIGID(true, false);
        else GO_RIGID(false, false);
        return;
    }
    if constexpr (TA % 2 == 0 && TA >= 4) {   // exact tiling is instantiated for even register tiles
        if (tailp) {
            if (l) GO(false, true, true, false);
            else if (xf) GO(false, false, true, true);
            else GO(false, false, true, false);
            return;
        }
    }
    if (l) {
        if (multi) GO(true, true, false, false);
        else GO(false, true, false, false);
    } else if (xf) {
        if (multi) GO(true, false, false, true);
        else GO(false, false, false, true);
    } else {
        if (multi) GO(true, false, false, false);
        else GO(false, false, false, false);
    }
#undef GO
#undef GO_RIGID
#undef GO_MEAN
}
static bool launch_sweep(int TA, bool multi, bool tailp, int grid, size_t smem, cudaStream_t s, const UnitDesc* units,
                         const WorkItem* work, const float4* lay, const float2* cs32, float* dist32,
                         unsigned long long* key, const ListArgs* l = nullptr, bool xf = false, const float2* t32 = nullptr,
                         bool mean = false) {
    switch (TA) {
#define CASE(T)                                                                                              \
    case T:                                                                                                  \
        launch_sweep_ta<T>(multi, tailp, xf, grid, smem, s, units, work, lay, cs32, dist32, key, l, t32, mean); \
        return true;
        CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8) CASE(9) CASE(10) CASE(11) CASE(12) CASE(13) CASE(14)
            CASE(15) CASE(16) CASE(17) CASE(18)
#undef CASE
    }
    return false;
}

// Size class of one unit: the register tile TA in [2,18] (test points per lane) minimising the padded work
// ceil(n / (32 TA)) * 32 TA (a chunk loop adds ~5 % per extra chunk: column minima go through shared memory;
// ties -> larger TA), against exact tiling: TA = floor(n / 32) full slots plus a tail pass over the remaining
// R = n mod 32 points, which costs R * ceil(m / 32) pair evaluations per lane at about 1.5x the main loop's price.
struct ClassChoice {
    int ta;
    bool tailp;
    int n_chunks;
};
static ClassChoice choose_class(int n, int m) {
    ClassChoice best{2, false, 1};
    double best_cost = 1e300;
    if (n <= 0) return best;
    for (int ta = 2; ta <= 18; ++ta) {
        const int per = 32 * ta;
        const int chunks = (n + per - 1) / per;
        const double cost = (double)chunks * per * (chunks > 1 ? 1.05 : 1.0);
        if (cost <= best_cost) best_cost = cost, best = ClassChoice{ta, false, chunks};
    }
    const int tf = n / 32, R = n - 32 * tf;
    const bool allow = !(std::getenv("MMRS_NO_TAILPASS") && std::getenv("MMRS_NO_TAILPASS")[0] == '1');
    if (allow && tf >= 4 && tf <= 18 && tf % 2 == 0 && R > 0 && 2 * ((m + 1) / 2) <= 32 * (tf + 1)) {
        const double cost = 32.0 * tf + 1.5 * ((R + 1) / 2 * 2) * (double)(tf + 1) * 32.0 / std::max(m, 1);
        if (cost < best_cost) best = ClassChoice{tf, true, 1};
    }
    return best;
}

// Partial cost: points of an n-point set that do not count, q(n) = n - K(n), K(n) = max(1, ceil(f n)) in f64.
static int partial_q(double f, int n) {
    if (n <= 0) return 0;
    return n - (int)std::max(1.0, std::ceil(f * (double)n));
}

static const char* cost_name(Cost c) { return c == kCostMean ? "mean cost" : c == kCostPartial ? "partial cost" : "cost"; }

// ---- upload ----------------------------------------------------------------------------
// Points part of an upload: validates the offsets, chooses the register tile, lays every unit out in the
// staging image (k_prep) and keeps the f64 points on the device. Grid-independent.
// Non-finite points. directed_hausdorff (process_utils.rs:84-121) keeps a row minimum only if it is finite (:112) and a
// NaN distance never passes `d2 < min_sq` (:108): a point with a NaN or infinite coordinate therefore takes part in
// neither directed pass, in either role, at any angle (rotating it keeps it non-finite) — exactly as if it were not in
// its set; only the emptiness test (:86-88) sees it, and a set whose points are all non-finite yields 0.0 like an empty
// one. The sweep kernels order distances by the bit patterns of non-negative finite floats, so such points are dropped
// HERE (rare: the batch is copied only when one is found). Returns true when a filtered copy was made.
static bool drop_non_finite(mmrs_ctx* ctx, const mmrs_sweep_batch* b, mmrs_sweep_batch* fb) {
    const int64_t U = b->n_units;
    const size_t n_test = (size_t)b->test_off[U], n_ref = (size_t)b->ref_off[U];
    bool finite = true;
    for (size_t i = 0; i < 2 * n_test && finite; ++i) finite = std::isfinite(b->test_xy[i]);
    for (size_t i = 0; i < 2 * n_ref && finite; ++i) finite = std::isfinite(b->ref_xy[i]);
    if (finite) return false;
    auto filter = [U](const double* xy, const int64_t* off, std::vector<double>& oxy, std::vector<int64_t>& ooff) {
        oxy.clear();
        ooff.assign(1, 0);
        for (int64_t u = 0; u < U; ++u) {
            for (int64_t i = off[u]; i < off[u + 1]; ++i)
                if (std::isfinite(xy[2 * i]) && std::isfinite(xy[2 * i + 1])) oxy.push_back(xy[2 * i]), oxy.push_back(xy[2 * i + 1]);
            ooff.push_back((int64_t)oxy.size() / 2);
        }
    };
    filter(b->test_xy, b->test_off, ctx->f_test, ctx->f_toff);
    filter(b->ref_xy, b->ref_off, ctx->f_ref, ctx->f_roff);
    *fb = *b;
    fb->test_xy = ctx->f_test.data(), fb->test_off = ctx->f_toff.data();
    fb->ref_xy = ctx->f_ref.data(), fb->ref_off = ctx->f_roff.data();
    return true;
}

static int upload_points(mmrs_ctx* ctx, const mmrs_sweep_batch* b_in) {
    const mmrs_sweep_batch* b = b_in;
    mmrs_sweep_batch filtered;
    {
        const int64_t U0 = b->n_units;
        for (int64_t u = 0; u < U0; ++u)
            if (b->test_off[u + 1] < b->test_off[u] || b->ref_off[u + 1] < b->ref_off[u] || b->test_off[0] < 0 || b->ref_off[0] < 0)
                return set_err(ctx, MMRS_ERR_ARG, "bad point offsets");
        if ((b->test_off[U0] && !b->test_xy) || (b->ref_off[U0] && !b->ref_xy))
            return set_err(ctx, MMRS_ERR_ARG, "point arrays are NULL");
        if (drop_non_finite(ctx, b, &filtered)) b = &filtered;
    }
    const int64_t U = b->n_units;
    int max_n = 1, max_m = 1;
    for (int64_t u = 0; u < U; ++u) {
        const int64_t n = b->test_off[u + 1] - b->test_off[u], m = b->ref_off[u + 1] - b->ref_off[u];
        if (n < 0 || m < 0 || n > (1 << 24) || m > (1 << 24)) return set_err(ctx, MMRS_ERR_ARG, "bad point offsets");
        max_n = std::max(max_n, (int)n);
        max_m = std::max(max_m, (int)m);
    }
    ctx->max_pts = std::max(max_n, max_m);
    std::vector<UnitDesc>& units = ctx->h_units;
    units.assign(U, UnitDesc{});
    ctx->classes.clear();
    ctx->class_of_unit.assign(U, -1);
    ctx->big_scratch_per_warp = 0;
    std::vector<size_t> ebp_stage, ebp_warp;   // partial cost, per class: the largest staging and per-warp block
    long long lay_off = 0;
    for (int64_t u = 0; u < U; ++u) {
        UnitDesc& d = units[u];
        d.test_off = b->test_off[u];
        d.ref_off = b->ref_off[u];
        d.n = (int)(b->test_off[u + 1] - b->test_off[u]);
        d.m = (int)(b->ref_off[u + 1] - b->ref_off[u]);
        d.cx = b->centre_xy[2 * u];
        d.cy = b->centre_xy[2 * u + 1];
        d.lay_off = lay_off;
        if (ctx->cost == kCostPartial) {
            const int q_f = partial_q(ctx->inlier_fraction, d.m), q_b = partial_q(ctx->inlier_fraction, d.n);
            if (q_f > kPartialMaxQ || q_b > kPartialMaxQ)
                return set_err(ctx, MMRS_ERR_ARG, "partial cost: unit " + std::to_string(u) + " leaves out " +
                                                      std::to_string(std::max(q_f, q_b)) +
                                                      " points in one direction; at most q = 255 per direction and unit");
            d.q_fwd = (short)q_f, d.q_bwd = (short)q_b;
        }
        d.ta = 2;
        if (d.n > 0 && d.m > 0) {
            const ClassChoice cc = choose_class(d.n, d.m);
            d.ta = cc.ta;
            d.n_chunks = cc.n_chunks;
            d.n_tail = cc.tailp ? d.n - 32 * cc.ta : 0;
            d.m_pairs = (d.m + 1) / 2;
            const StageLayout sl = stage_layout(cc.ta, d.n_chunks, d.n_tail, d.m_pairs);
            const size_t stage = 16 + (size_t)sl.total() * 16;   // mbarrier + key, then the staging image
            // shared memory of a K1 CTA of this unit: the staging, then per warp either the chunked column minima (MULTI;
            // the mean cost: every class but exact tiling) or the tail pass's column seeds (exact tiling)
            size_t smem = stage;
            if (d.n_chunks > 1 || (ctx->cost == kCostMean && !cc.tailp)) smem += (size_t)kWarpsPerCta * ((2 * d.m_pairs + 3) & ~3) * 4;
            if (cc.tailp) smem += (size_t)kWarpsPerCta * 32 * (cc.ta + 1) * 4;
            static const bool force_big = std::getenv("MMRS_FORCE_BIG") && std::getenv("MMRS_FORCE_BIG")[0] == '1';
            const bool big = smem > (size_t)kMaxDynSmem || (force_big && d.n >= 64);
            if (big) {
                // does not fit K1's shared-memory staging: K1b streams the reference set through shared memory in blocks
                // (k_sweep_big; register tile 16, the whole staging image stays in global memory / L2)
                d.ta = kBigTA;
                d.n_chunks = (d.n + 32 * kBigTA - 1) / (32 * kBigTA);
                d.n_tail = 0;
                smem = 0;
                ctx->big_scratch_per_warp = std::max<long long>(ctx->big_scratch_per_warp, (long long)d.n_chunks * 32 * kBigTA);
            }
            lay_off += stage_layout(d.ta, d.n_chunks, d.n_tail, d.m_pairs).total();
            int k = 0;
            for (; k < (int)ctx->classes.size(); ++k) {
                const auto& c = ctx->classes[k];
                if (c.big == big && (big || (c.ta == cc.ta && c.multi == (d.n_chunks > 1) && c.tailp == cc.tailp))) break;
            }
            if (k == (int)ctx->classes.size()) {
                mmrs_ctx::SweepClass c;
                c.ta = big ? kBigTA : cc.ta, c.multi = d.n_chunks > 1, c.tailp = !big && cc.tailp, c.big = big;
                c.eb_warps = kWarpsPerCta;
                ctx->classes.push_back(c);
                ebp_stage.push_back(0), ebp_warp.push_back(0);
            }
            auto& cl = ctx->classes[k];
            cl.smem = std::max(cl.smem, smem);
            cl.cost += (long long)d.n_chunks * 32 * d.ta * d.m;
            ctx->class_of_unit[u] = k;
            if (ctx->cost != kCostFull && big)
                return set_err(ctx, MMRS_ERR_ARG, std::string(cost_name(ctx->cost)) + ": unit " + std::to_string(u) +
                                                      " is beyond the shared-memory staging (more than ~4 000 points per set)");
            if (ctx->cost == kCostPartial) {
                ebp_stage[k] = std::max(ebp_stage[k], stage);
                ebp_warp[k] = std::max(ebp_warp[k], (size_t)ebp_warp_bytes(d.n, d.m, d.q_bwd, d.q_fwd));
            } else if (!big) {   // K1e: the same staging image plus, per warp, A' and the row / column hints
                cl.smem_eb = std::max(cl.smem_eb, stage + (size_t)kWarpsPerCta * eb_warp_bytes(d.n, d.m));
            }
        }
    }
    if (ctx->cost == kCostPartial) {
        // K1e-partial: 8 warps per CTA where the largest staging image and 8 of the largest per-warp blocks fit the
        // 227 KB a CTA may have, else 4, 2 or 1 (the chunked 2 020-point units take 4)
        for (size_t k = 0; k < ctx->classes.size(); ++k) {
            auto& cl = ctx->classes[k];
            cl.eb_warps = 0;
            for (int wp = kWarpsPerCta; wp >= 1 && !cl.eb_warps; wp /= 2)
                if (ebp_stage[k] + wp * ebp_warp[k] <= (size_t)kMaxDynSmem) cl.eb_warps = wp;
            if (!cl.eb_warps)
                return set_err(ctx, MMRS_ERR_ARG, "partial cost: a unit does not fit the shared memory of one warp");
            cl.smem_eb = ebp_stage[k] + cl.eb_warps * ebp_warp[k];
        }
    }
    {   // tensor-core prefilter: every non-empty unit must fit its operand layout
        bool ok = true;
        size_t smem_tc = 0;
        for (auto& d : units) {
            if (d.n <= 0 || d.m <= 0) continue;
            if (d.n < kTcMinPts || d.m < kTcMinPts || d.n > kTcMaxPts || d.m > kTcMaxPts) {
                ok = false;
                break;
            }
            const int ra = (d.n + 127) / 128 * 128;
            smem_tc = std::max(smem_tc, tc_smem_bytes(d.n, d.m, ra <= 1024 ? 2 : 1));
        }
        for (const auto& cl : ctx->classes) ok = ok && !cl.big;
        ctx->tc_shape_ok = ok && smem_tc > 0 && smem_tc <= 227 * 1024;
        ctx->smem_tc = smem_tc;
    }
    {   // lower-bound pruning tier: R strided rows of one set against all points of the other, both ways
        bool ok = U > 0;
        int biggest = 0;
        for (auto& d : units) {
            if (d.n <= 0 || d.m <= 0) continue;
            if (d.n < 128 || d.m < 128) ok = false;
            biggest = std::max(biggest, std::max(d.n, d.m));
        }
        for (const auto& cl : ctx->classes) ok = ok && !cl.big;   // the list re-scoring kernel does not take K1b's units
        ctx->lb_R = biggest >= 1024 ? 128 : 32;  // rows per lower-bound pass: k_lb<1,8> or k_lb<4,2>
        // the bound tier's staging images are only built for a batch that may use it (opts / context default / MMRS_PRUNE)
        const char* prune_env = std::getenv("MMRS_PRUNE");
        const bool may_prune = !ctx->rigid && ctx->cost == kCostFull && ((prune_env && *prune_env) ? (*prune_env != '0') : ctx->opt_prune == 1);
        ctx->lb_shape_ok = ok && biggest > 0 && may_prune;
        ctx->h_units_lb.assign(2 * (size_t)U, UnitDesc{});
        long long off = 0;
        size_t smem_lb = 0;
        if (ctx->lb_shape_ok)
            for (int pass = 0; pass < 2; ++pass)
                for (int64_t u = 0; u < U; ++u) {
                    const UnitDesc& d = units[u];
                    UnitDesc& l = ctx->h_units_lb[u + pass * U];
                    l = d;
                    l.n = ctx->lb_R;
                    l.m = pass == 0 ? d.m : d.n;
                    l.n_chunks = 1;
                    l.m_pairs = (l.m + 1) / 2;
                    l.lay_off = off;
                    if (d.n > 0 && d.m > 0) {
                        off += ctx->lb_R / 2 + l.m_pairs;
                        smem_lb = std::max(smem_lb, (size_t)(ctx->lb_R / 2 + l.m_pairs) * 16);
                    }
                }
        ctx->smem_lb = 16 + smem_lb;
        if (ctx->lb_shape_ok) {
            ENSURE(ctx->d_units_lb, 2 * U * sizeof(UnitDesc));
            ENSURE(ctx->d_lay_lb, (size_t)off * 16);
        }
    }
    const size_t n_test = (size_t)b->test_off[U], n_ref = (size_t)b->ref_off[U];
    if ((n_test && !b->test_xy) || (n_ref && !b->ref_xy)) return set_err(ctx, MMRS_ERR_ARG, "point arrays are NULL");
    ENSURE(ctx->d_test, n_test * 16);
    ENSURE(ctx->d_ref, n_ref * 16);
    ENSURE(ctx->d_units, U * sizeof(UnitDesc));
    ENSURE(ctx->d_lay, (size_t)lay_off * 16);
    ENSURE(ctx->d_key, U * 8);
    ENSURE(ctx->d_rmax, U * 4);
    ENSURE(ctx->d_sl_base, U * 4);
    ENSURE(ctx->d_sl_count, U * 4);
    ENSURE(ctx->d_nitems, 16);
    ENSURE(ctx->d_res, U * sizeof(UnitResultDev));
    if ((size_t)U > ctx->h_res_cap) {
        if (ctx->h_res) cudaFreeHost(ctx->h_res);
        ctx->h_res = nullptr;
        CUDA_TRY(ctx, cudaMallocHost(&ctx->h_res, (size_t)U * sizeof(UnitResultDev)));
        ctx->h_res_cap = (size_t)U;
    }
    cudaStream_t s = ctx->stream;
    if (n_test) CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_test.p, b->test_xy, n_test * 16, cudaMemcpyHostToDevice, s));
    if (n_ref) CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_ref.p, b->ref_xy, n_ref * 16, cudaMemcpyHostToDevice, s));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_units.p, units.data(), U * sizeof(UnitDesc), cudaMemcpyHostToDevice, s));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_rmax.p, 0, U * 4, s));
    k_prep<<<(unsigned)U, 256, 0, s>>>((const UnitDesc*)ctx->d_units.p, (const double*)ctx->d_test.p,
                                       (const double*)ctx->d_ref.p, (float4*)ctx->d_lay.p, (unsigned*)ctx->d_rmax.p);
    CUDA_TRY(ctx, cudaGetLastError());
    ctx->upload_launches = 1;
    if (ctx->lb_shape_ok) {
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_units_lb.p, ctx->h_units_lb.data(), 2 * U * sizeof(UnitDesc),
                                      cudaMemcpyHostToDevice, s));
        k_prep_lb<<<(unsigned)U, 256, 0, s>>>((const UnitDesc*)ctx->d_units.p, (const UnitDesc*)ctx->d_units_lb.p, (int)U,
                                              (const double*)ctx->d_test.p, (const double*)ctx->d_ref.p,
                                              (float4*)ctx->d_lay_lb.p, ctx->lb_R,
                                              std::getenv("MMRS_LB_ROWS") ? std::max(8, std::min(ctx->lb_R, std::atoi(std::getenv("MMRS_LB_ROWS")))) : ctx->lb_R,
                                              std::getenv("MMRS_LB_PICK") ? std::atoi(std::getenv("MMRS_LB_PICK")) : 2);
        CUDA_TRY(ctx, cudaGetLastError());
        ctx->upload_launches += 1;
    }
    return MMRS_OK;
}

// Translation grid checks of mmrs_tgrid (include/mmrs_b200.h).
static int check_tgrid(mmrs_ctx* ctx, const mmrs_tgrid& t) {
    if (t.half_n < 0) return set_err(ctx, MMRS_ERR_ARG, "translation grid: half_n must be >= 0");
    if (!std::isfinite(t.t0x) || !std::isfinite(t.t0y) || !std::isfinite(t.step))
        return set_err(ctx, MMRS_ERR_ARG, "translation grid: t0 and step must be finite");
    if (t.half_n > 0 && !(t.step > 0.0)) return set_err(ctx, MMRS_ERR_ARG, "translation grid: step must be > 0 when half_n > 0");
    if (t.half_n > 23169) return set_err(ctx, MMRS_ERR_ARG, "translation grid: more than INT32_MAX translations");
    return MMRS_OK;
}
// Translation j = jy (2 half_n + 1) + jx of a translation grid, evaluated in f64 exactly as the header states.
static inline void tgrid_offset(const mmrs_tgrid& t, int64_t j, double* tx, double* ty) {
    const int64_t w = 2 * (int64_t)t.half_n + 1, jy = j / w, jx = j - jy * w;
    *tx = t.t0x + (double)(jx - t.half_n) * t.step;
    *ty = t.t0y + (double)(jy - t.half_n) * t.step;
}

// The tier of the uploaded grids, in order of precedence: the tensor-core prefilter K1t, the expanded form K1x, then
// lower-bound pruning K1p. solo (rigid candidates, the partial or the mean cost) and the candidate-axis partition take the dense sweep.
// Sizes the tier's candidate list and builds its work list.
static int plan_tier(mmrs_ctx* ctx, bool solo, long long live) {
    const int64_t U = ctx->n_units;
    const std::vector<UnitDesc>& units = ctx->h_units;
    long long live_units = 0;
    for (auto& d : units)
        if (!d.flags) ++live_units;
    bool any_big = false;
    for (const auto& cl : ctx->classes) any_big = any_big || cl.big;
    ctx->tier = kTierDense;
    ctx->h_work_tc.clear();
    ctx->h_work_lb.clear();
    if (solo) return MMRS_OK;
    const bool part2 = ctx->part_active == 2;
    // Tensor-core prefilter: worth it when the units carry enough candidates to amortise the per-CTA operand set-up.
    const char* env = std::getenv("MMRS_PREFILTER");  // experiments: 0 = off, 1 = on where the shapes allow
    int tc_mode = ctx->opt_prefilter;
    if (env && *env) tc_mode = (*env == '0') ? 1 : 2;
    // auto (0) currently resolves to the dense FP32 sweep: on B200 the prefilter's per-tile TMEM hand-shakes and
    // the FMNMX-bound epilogue make K1t slower than K1 (17 vs 24 M evaluations/s, DESIGN.md §4).
    const bool tc = tc_mode == 2 && ctx->tc_shape_ok && live_units > 0 && !part2;
    if (tc_mode == 2 && !tc && ctx->opt_prefilter == 2)
        return set_err(ctx, MMRS_ERR_ARG,
                       "prefilter required but the batch does not fit the tensor-core operand layout (64 <= points "
                       "per set <= 2048)");
    // Expanded-form tier K1x (k_sweep<.., XF>): the same work list and size classes as the dense sweep, 6 instead of 8
    // packed FP32 instructions per 2 x 2 block; candidates inside its error window are re-scored in direct form.
    env = std::getenv("MMRS_XF");   // experiments: 1 = on for every batch that qualifies, 0 = off
    int xf_mode = ctx->opt_prefilter;
    if (env && *env && xf_mode == 0) xf_mode = (*env == '0') ? 1 : 3;
    if (xf_mode == 0) xf_mode = kXfDefault ? 3 : 1;
    // worth it when the sweep is long enough to pay for two extra launches (window + re-scoring)
    const bool xf = xf_mode == 3 && !any_big && !part2 && live >= (ctx->opt_prefilter == 3 ? 1 : (1 << 20));
    // Lower-bound pruning: worth it when a unit carries enough candidates for the two extra passes to pay off.
    env = std::getenv("MMRS_PRUNE");
    int prune_mode = ctx->opt_prune;
    if (env && *env) prune_mode = (*env == '0') ? 0 : 1;
    const bool prune = prune_mode == 1 && ctx->lb_shape_ok && live_units > 0 && live >= 256 * live_units && !part2;
    ctx->tier = tc ? kTierTc : xf ? kTierXf : prune ? kTierPrune : kTierDense;
    if (ctx->tier == kTierTc) {
        long long tile = (live + (long long)ctx->n_sm * 6 - 1) / ((long long)ctx->n_sm * 6);
        tile = std::max<long long>(64, std::min<long long>(tile, 512));
        for (int64_t u = 0; u < U; ++u) {
            const UnitDesc& d = units[u];
            if (d.flags) continue;
            const int parts = (int)((d.n_cand + tile - 1) / tile);
            const int per = (d.n_cand + parts - 1) / parts;
            for (int c0 = 0; c0 < d.n_cand; c0 += per)
                ctx->h_work_tc.push_back(WorkItem{(int)u, c0, std::min(per, d.n_cand - c0), 0});
        }
        ctx->l1_cap = (unsigned)std::min<unsigned long long>(
            std::max<unsigned long long>((unsigned long long)U * 256, 1ull << 20), 0x7fffffffull);
        ENSURE(ctx->d_work_tc, ctx->h_work_tc.size() * sizeof(WorkItem));
        ENSURE(ctx->d_key_tc, U * 8);
    } else if (ctx->tier == kTierXf) {
        ctx->l1_cap = (unsigned)std::min<long long>(std::max<long long>({(long long)U * 64, 65536LL, live / 32}),
                                                    std::max<long long>(live, 1));
        ENSURE(ctx->d_key_tc, U * 8);
    } else if (ctx->tier == kTierPrune) {
        for (int pass = 0; pass < 2; ++pass)
            for (int64_t u = 0; u < U; ++u) {
                UnitDesc& l = ctx->h_units_lb[u + pass * U];
                const UnitDesc& d = units[u];
                l.cand_off = d.cand_off, l.n_cand = d.n_cand, l.dist_off = d.dist_off;
                l.flags = d.flags | (pass == 1 ? kLbNegSin : 0);
            }
        const long long slots = (long long)ctx->n_sm * 2 * 4;
        long long per_warp = (2 * live + slots * kWarpsPerCta - 1) / (slots * kWarpsPerCta);
        per_warp = std::max<long long>(8, std::min<long long>((per_warp + 7) / 8 * 8, 64));  // k_lb: 8 candidates per warp pass
        const int tile = (int)per_warp * kWarpsPerCta;
        for (int pass = 0; pass < 2; ++pass)
            for (int64_t u = 0; u < U; ++u) {
                const UnitDesc& d = units[u];
                if (d.flags) continue;
                for (int c0 = 0; c0 < d.n_cand; c0 += tile)
                    ctx->h_work_lb.push_back(WorkItem{(int)(u + pass * U), c0, std::min(tile, d.n_cand - c0), 0});
            }
        ctx->l1_cap = (unsigned)std::min<long long>(std::max<long long>(ctx->total_cands, 1), 0x7fffffffLL);
        ENSURE(ctx->d_work_lb, ctx->h_work_lb.size() * sizeof(WorkItem));
    } else {
        return MMRS_OK;
    }
    ENSURE(ctx->d_l1_items, (size_t)ctx->l1_cap * 8);
    ENSURE(ctx->d_l1_count, U * 4);
    ENSURE(ctx->d_l1_base, U * 4);
    ENSURE(ctx->d_l1_n, 16);
    return MMRS_OK;
}

// Grid part: candidate tables (host glibc cos/sin), per-unit candidate ranges, the CTA work list.
// tgrids == NULL: rotation-only candidates (every unit has one translation, none applied). Otherwise rigid candidates:
// unit u sweeps grid x tgrids[tgrid_of_unit[u]], candidate c = i T + j (angle i, translation j), densely and on this
// rank alone (no pruning / prefilter tier, no partition).
static int apply_grids(mmrs_ctx* ctx, const mmrs_grid* grids, int64_t n_grids, const int32_t* grid_of_unit,
                       const mmrs_tgrid* tgrids = nullptr, int64_t n_tgrids = 0, const int32_t* tgrid_of_unit = nullptr) {
    const int64_t U = ctx->n_units;
    ctx->grids.assign(grids, grids + n_grids);
    ctx->grid_of_unit.resize(U);
    for (int64_t u = 0; u < U; ++u) {
        const int g = grid_of_unit ? grid_of_unit[u] : 0;
        if (g < 0 || g >= n_grids) return set_err(ctx, MMRS_ERR_ARG, "grid_of_unit out of range");
        ctx->grid_of_unit[u] = g;
    }
    ctx->rigid = tgrids != nullptr;
    const bool solo = ctx->rigid || ctx->cost != kCostFull;   // the dense sweep on this device alone: no tier, no partition
    std::vector<long long> tgrid_off(1, 0);
    if (ctx->rigid) {
        if (n_tgrids < 1) return set_err(ctx, MMRS_ERR_ARG, "rigid sweep: n_tgrids must be >= 1");
        ctx->tgrids.assign(tgrids, tgrids + n_tgrids);
        ctx->tgrid_of_unit.resize(U);
        for (int64_t u = 0; u < U; ++u) {
            const int g = tgrid_of_unit ? tgrid_of_unit[u] : 0;
            if (g < 0 || g >= n_tgrids) return set_err(ctx, MMRS_ERR_ARG, "tgrid_of_unit out of range");
            ctx->tgrid_of_unit[u] = g;
        }
        tgrid_off.assign(n_tgrids + 1, 0);
        for (int64_t g = 0; g < n_tgrids; ++g) {
            if (int rc = check_tgrid(ctx, tgrids[g])) return rc;
            const long long w = 2LL * tgrids[g].half_n + 1;
            tgrid_off[g + 1] = tgrid_off[g] + w * w;
        }
        for (int64_t u = 0; u < U; ++u) {
            const mmrs_grid& gr = grids[ctx->grid_of_unit[u]];
            const long long T = tgrid_off[ctx->tgrid_of_unit[u] + 1] - tgrid_off[ctx->tgrid_of_unit[u]];
            if (!gr.degenerate && (double)gr.n_cand * (double)T > 2147483646.0)
                return set_err(ctx, MMRS_ERR_ARG,
                               "rigid sweep: angles x translations of unit " + std::to_string(u) + " exceed INT32_MAX candidates");
        }
        ctx->h_t.resize(2 * (size_t)tgrid_off[n_tgrids]);
        std::vector<double> tmax_of_grid(n_tgrids, 0.0);
        for (int64_t g = 0; g < n_tgrids; ++g)
            for (long long j = 0; j < tgrid_off[g + 1] - tgrid_off[g]; ++j) {
                double* t = &ctx->h_t[2 * (tgrid_off[g] + j)];
                tgrid_offset(tgrids[g], j, &t[0], &t[1]);
                tmax_of_grid[g] = std::max(tmax_of_grid[g], std::hypot(t[0], t[1]));
            }
        ctx->h_tmax.resize(U);
        for (int64_t u = 0; u < U; ++u) ctx->h_tmax[u] = tmax_of_grid[ctx->tgrid_of_unit[u]];
    } else {
        ctx->tgrids.clear();
        ctx->tgrid_of_unit.clear();
    }
    // cos/sin tables: HOST glibc (bit-identical to Rust's f64::sin/cos), one per grid.
    std::vector<long long> grid_off(n_grids + 1, 0);
    for (int64_t g = 0; g < n_grids; ++g) {
        const mmrs_grid& gr = grids[g];
        if (gr.n_cand < 0 || gr.n_cand > (1ll << 31) - 2) return set_err(ctx, MMRS_ERR_ARG, "grid: bad n_cand");
        grid_off[g + 1] = grid_off[g] + (gr.degenerate ? 0 : gr.n_cand);
    }
    const long long n_cs = grid_off[n_grids];
    ctx->h_cs.resize(2 * (size_t)n_cs);
    ctx->h_zero.resize((size_t)n_cs);
    {   // spans of <= 2048 candidates, filled on the host pool when the tables are large (config 3: 1 596 grids x 361
        // candidates = 23 ms of glibc sin/cos on one thread)
        struct Span {
            int64_t g, i0, i1;
        };
        std::vector<Span> spans;
        for (int64_t g = 0; g < n_grids; ++g) {
            if (grids[g].degenerate) continue;
            for (int64_t i0 = 0; i0 < grids[g].n_cand; i0 += 2048) spans.push_back(Span{g, i0, std::min<int64_t>(i0 + 2048, grids[g].n_cand)});
        }
        auto fill = [&](size_t k) {
            const Span sp = spans[k];
            const mmrs_grid& gr = grids[sp.g];
            for (int64_t i = sp.i0; i < sp.i1; ++i) {
                const double a = mmrs_grid_angle(&gr, i);
                ctx->h_cs[2 * (grid_off[sp.g] + i)] = std::cos(a);
                ctx->h_cs[2 * (grid_off[sp.g] + i) + 1] = std::sin(a);
                ctx->h_zero[grid_off[sp.g] + i] = (ctx->mode == 0 && a == 0.0) ? 1 : 0;
            }
        };
        if (n_cs >= 16384) parallel_for(spans.size(), fill);
        else for (size_t k = 0; k < spans.size(); ++k) fill(k);
    }
    std::vector<UnitDesc>& units = ctx->h_units;
    long long dist_off = 0, live = 0;
    for (int64_t u = 0; u < U; ++u) {
        UnitDesc& d = units[u];
        const mmrs_grid& gr = grids[ctx->grid_of_unit[u]];
        d.cand_off = grid_off[ctx->grid_of_unit[u]];
        d.t_off = ctx->rigid ? tgrid_off[ctx->tgrid_of_unit[u]] : 0;
        d.n_trans = ctx->rigid ? (int)(tgrid_off[ctx->tgrid_of_unit[u] + 1] - d.t_off) : 1;
        d.n_cand = gr.degenerate ? 0 : (int)(gr.n_cand * d.n_trans);
        d.flags = 0;
        if (gr.degenerate) d.flags |= MMRS_FLAG_DEGENERATE;
        if (d.n == 0 || d.m == 0) d.flags |= MMRS_FLAG_EMPTY;
        d.dist_off = dist_off;
        dist_off += d.n_cand;
        d.c_lo = 0;
        d.c_hi = d.n_cand;
    }
    ctx->total_cands = dist_off;
    // Partition across ranks (mmrs_ctx_comm_init / mmrs_ctx_set_shard): which candidates of which units THIS rank sweeps.
    {
        const int world = ctx->shard_world, rank = ctx->shard_rank;
        int axis = ctx->opt_partition == 0 ? ctx->part_axis : ctx->opt_partition;
        if (world <= 1 || (!ctx->comm && !ctx->exchange) || axis < 1 || axis > 2 || solo) axis = 0;
        if (axis == 1 && ctx->opt_partition == 0) {
            // The context's default axis is a POLICY, decided from the shape of the batch alone (so every rank decides
            // alike): whole units where they balance; candidate sub-ranges where a handful of large units cannot be
            // dealt evenly (the inter-pullback stages: 2 units, 72 000 candidates each, would keep 2 of 8 GPUs busy);
            // no partition at all where the whole batch is cheaper than the collective that would merge it.
            double total = 0.0, biggest = 0.0;
            long long min_cand = (1ll << 62);
            for (int64_t u = 0; u < U; ++u) {
                const UnitDesc& d = units[u];
                if (d.flags) continue;
                const double c = (double)d.n * d.m * d.n_cand;
                total += c;
                biggest = std::max(biggest, c);
                min_cand = std::min<long long>(min_cand, d.n_cand);
            }
            constexpr double kTinyBatch = 2.0e9;   // pair evaluations: ~0.3 ms of one B200, a few NCCL latencies
            if (total < kTinyBatch) {
                axis = 0;
            } else if (ctx->comm && min_cand >= 64ll * world) {
                // best unit partition possible: no block can be smaller than the largest unit
                const double block = std::max(total / world, biggest);
                if (block > 1.25 * total / world) axis = 2;
            }
        }
        if (axis == 2 && !ctx->comm)
            return set_err(ctx, MMRS_ERR_STATE, "the candidate-axis partition needs a communicator (mmrs_ctx_comm_init)");
        ctx->part_active = axis;
        if (axis == 1) {
            // whole units in contiguous blocks balanced by cost (pair evaluations), identical on every rank
            std::vector<double> pre(U + 1, 0.0);
            for (int64_t u = 0; u < U; ++u) {
                const UnitDesc& d = units[u];
                pre[u + 1] = pre[u] + 1.0 + (d.flags ? 0.0 : (double)d.n * d.m * d.n_cand);
            }
            const double total = pre[U];
            for (int64_t u = 0; u < U; ++u) {
                // owner = the block the unit's cost midpoint falls into
                const double mid = 0.5 * (pre[u] + pre[u + 1]);
                int owner = (int)(mid * world / total);
                owner = std::min(std::max(owner, 0), world - 1);
                if (owner != rank) units[u].flags |= kFlagRemote, units[u].c_hi = 0;
            }
        } else if (axis == 2) {
            for (int64_t u = 0; u < U; ++u) {
                UnitDesc& d = units[u];
                const long long base = d.n_cand / world, extra = d.n_cand % world;
                d.c_lo = (int)(rank * base + std::min<long long>(rank, extra));
                d.c_hi = d.c_lo + (int)(base + (rank < extra ? 1 : 0));
            }
        }
    }
    for (auto& cl : ctx->classes) cl.live = 0;
    for (int64_t u = 0; u < U; ++u)
        if (!units[u].flags) {
            live += units[u].c_hi - units[u].c_lo;
            ctx->classes[ctx->class_of_unit[u]].live += units[u].c_hi - units[u].c_lo;
        }
    // K1e per size class (MMRS_EARLY_BREAK: 0 = K1 everywhere, 1 = K1e wherever its shared memory fits). A class beyond
    // the per-warp A' and hints (sets above ~1 000 points, the chunked 2 020-point units among them) keeps K1.
    // A partial run takes K1e-partial in every class (MMRS_EARLY_BREAK=0 only switches its early break off), a mean run
    // the mean K1 in every class.
    for (auto& cl : ctx->classes)
        cl.eb = ctx->cost == kCostFull && ctx->eb_env != 0 && !cl.big && cl.smem_eb <= (ctx->eb_env == 1 ? (size_t)kMaxDynSmem : kEbAutoSmem);
    // work list: one CTA = one unit x one tile of candidates (8 warps, one candidate per warp per pass; K1e: one
    // contiguous run per warp, as long as the batch still gives ~4 waves of 3 CTAs per SM)
    {
        const long long slots = (long long)ctx->n_sm * 2 * 4;  // CTAs for ~4 waves at 2 CTAs/SM
        long long per_warp = (live + slots * kWarpsPerCta - 1) / (slots * kWarpsPerCta);
        // a CTA stages its unit once (one TMA bulk copy) and every warp walks `per_warp` candidates; measured on B200
        // (profiles/r02_tile_per_warp.txt): 8, 32 and 64 per warp are within 0.5 % of each other, 8 keeps the tail short
        static const long long cap = std::getenv("MMRS_TILE_PER_WARP") ? std::atoll(std::getenv("MMRS_TILE_PER_WARP")) : 8;
        per_warp = std::max<long long>(1, std::min<long long>(per_warp, std::max<long long>(cap, 1)));
        const int tile = (int)per_warp * kWarpsPerCta;
        ctx->h_work.clear();
        for (size_t k = 0; k < ctx->classes.size(); ++k) {   // one contiguous range of the work list per size class
            auto& cl = ctx->classes[k];
            cl.work_begin = ctx->h_work.size();
            const long long eb_slots = (long long)ctx->n_sm * 3 * 4 * kWarpsPerCta;
            const long long run = std::max(kEbMinRun, std::min(kEbMaxRun, (cl.live + eb_slots - 1) / eb_slots));
            const int tile_k = ctx->cost == kCostPartial || cl.eb ? (int)(cl.eb_warps * run) : tile;
            for (int64_t u = 0; u < U; ++u) {
                const UnitDesc& d = units[u];
                if (d.flags || ctx->class_of_unit[u] != (int)k) continue;
                for (int c0 = d.c_lo; c0 < d.c_hi; c0 += tile_k)
                    ctx->h_work.push_back(WorkItem{(int)u, c0, std::min(tile_k, d.c_hi - c0), 0});
            }
            cl.work_count = ctx->h_work.size() - cl.work_begin;
        }
    }
    if (int rc = plan_tier(ctx, solo, live)) return rc;
    ENSURE(ctx->d_work, ctx->h_work.size() * sizeof(WorkItem));
    ENSURE(ctx->d_cs64, (size_t)n_cs * 16);
    ENSURE(ctx->d_cs32, (size_t)n_cs * 8);
    ENSURE(ctx->d_zero, (size_t)n_cs);
    ENSURE(ctx->d_dist32, (size_t)dist_off * 4);
    // item pool shared by all units: `cap` per unit on average, never less than 64 Ki items
    ctx->pool_cap = (unsigned)std::min<unsigned long long>(
        std::max<unsigned long long>((unsigned long long)U * ctx->cap, 1ull << 16), 0x7fffffffull);
    ENSURE(ctx->d_sl_dist, (size_t)ctx->pool_cap * 8);
    ENSURE(ctx->d_items, (size_t)ctx->pool_cap * 8);
    cudaStream_t s = ctx->stream;
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_units.p, units.data(), U * sizeof(UnitDesc), cudaMemcpyHostToDevice, s));
    if (!ctx->h_work.empty())
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_work.p, ctx->h_work.data(), ctx->h_work.size() * sizeof(WorkItem),
                                      cudaMemcpyHostToDevice, s));
    if (ctx->tier == kTierPrune && !ctx->h_work_lb.empty()) {
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_units_lb.p, ctx->h_units_lb.data(), 2 * U * sizeof(UnitDesc),
                                      cudaMemcpyHostToDevice, s));
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_work_lb.p, ctx->h_work_lb.data(), ctx->h_work_lb.size() * sizeof(WorkItem),
                                      cudaMemcpyHostToDevice, s));
    }
    if (ctx->tier == kTierTc && !ctx->h_work_tc.empty()) {
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_work_tc.p, ctx->h_work_tc.data(), ctx->h_work_tc.size() * sizeof(WorkItem),
                                      cudaMemcpyHostToDevice, s));
    }
    if (n_cs) {
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_cs64.p, ctx->h_cs.data(), (size_t)n_cs * 16, cudaMemcpyHostToDevice, s));
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_zero.p, ctx->h_zero.data(), (size_t)n_cs, cudaMemcpyHostToDevice, s));
        k_cs32<<<(unsigned)((n_cs + 255) / 256), 256, 0, s>>>((const double2*)ctx->d_cs64.p, (float2*)ctx->d_cs32.p,
                                                              n_cs);
        CUDA_TRY(ctx, cudaGetLastError());
        ctx->upload_launches += 1;
    }
    if (ctx->rigid) {   // translation tables (f64 for K3 / K4, rounded once to FP32 for the sweep) and R_eff per unit
        const long long n_t = (long long)ctx->h_t.size() / 2;
        ENSURE(ctx->d_t64, (size_t)n_t * 16);
        ENSURE(ctx->d_t32, (size_t)n_t * 8);
        ENSURE(ctx->d_tmax, (size_t)U * 8);
        ENSURE(ctx->d_reff, (size_t)U * 4);
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_t64.p, ctx->h_t.data(), (size_t)n_t * 16, cudaMemcpyHostToDevice, s));
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_tmax.p, ctx->h_tmax.data(), (size_t)U * 8, cudaMemcpyHostToDevice, s));
        k_cs32<<<(unsigned)((n_t + 255) / 256), 256, 0, s>>>((const double2*)ctx->d_t64.p, (float2*)ctx->d_t32.p, n_t);
        CUDA_TRY(ctx, cudaGetLastError());
        k_reff<<<(unsigned)((U + 255) / 256), 256, 0, s>>>((const unsigned*)ctx->d_rmax.p, (const double*)ctx->d_tmax.p,
                                                           (unsigned*)ctx->d_reff.p, (int)U);
        CUDA_TRY(ctx, cudaGetLastError());
        ctx->upload_launches += 2;
    }
    return MMRS_OK;
}

// Translation grids of a rigid upload / regrid, checked before any device work.
static int check_tgrids(mmrs_ctx* ctx, const char* fn, int64_t n_units, const mmrs_tgrid* tgrids, int64_t n_tgrids,
                        const int32_t* tgrid_of_unit) {
    if (!tgrids || n_tgrids < 1) return set_err(ctx, MMRS_ERR_ARG, std::string(fn) + ": bad translation grids");
    for (int64_t g = 0; g < n_tgrids; ++g)
        if (int rc = check_tgrid(ctx, tgrids[g])) return rc;
    for (int64_t u = 0; tgrid_of_unit && u < n_units; ++u)
        if (tgrid_of_unit[u] < 0 || tgrid_of_unit[u] >= n_tgrids) return set_err(ctx, MMRS_ERR_ARG, "tgrid_of_unit out of range");
    return MMRS_OK;
}

// Upload of a rotation-only batch (tgrids == NULL) or of a rigid one, with its cost (the partial cost: inlier_fraction).
static int upload_impl(mmrs_ctx* ctx, const mmrs_sweep_batch* b, const mmrs_sweep_opts* o, const mmrs_tgrid* tgrids,
                       int64_t n_tgrids, const int32_t* tgrid_of_unit, const char* fn, Cost cost = kCostFull,
                       double inlier_fraction = 1.0) {
    if (!ctx) return set_err(nullptr, MMRS_ERR_ARG, std::string(fn) + ": ctx is NULL");
    if (!b || b->n_units < 0 || (b->n_units > 0 && (!b->test_off || !b->ref_off || !b->centre_xy || !b->grids)) ||
        (b->n_grids < 1 && b->n_units > 0))
        return set_err(ctx, MMRS_ERR_ARG, std::string(fn) + ": bad batch");
    if (b->mode != 0 && b->mode != 1) return set_err(ctx, MMRS_ERR_ARG, std::string(fn) + ": mode must be 0 or 1");
    if (tgrids || n_tgrids) {
        if (int rc = check_tgrids(ctx, fn, b->n_units, tgrids, n_tgrids, tgrid_of_unit)) return rc;
        if (o && o->prune > 0) return set_err(ctx, MMRS_ERR_ARG, std::string(fn) + ": prune is not supported with a translation grid");
        if (o && (o->prefilter == 2 || o->prefilter == 3))
            return set_err(ctx, MMRS_ERR_ARG, std::string(fn) + ": prefilter 2 / 3 is not supported with a translation grid");
    }
    if (cost != kCostFull) {
        const std::string with = std::string(" is not supported with the ") + cost_name(cost);
        if (o && o->prune > 0) return set_err(ctx, MMRS_ERR_ARG, std::string(fn) + ": prune" + with);
        if (o && (o->prefilter == 2 || o->prefilter == 3))
            return set_err(ctx, MMRS_ERR_ARG, std::string(fn) + ": prefilter 2 / 3" + with);
    }
    ENTER_DEVICE(ctx);
    ctx->ready = false;
    ctx->ran = false;
    ctx->rigid = tgrids != nullptr;
    ctx->cost = cost;
    ctx->inlier_fraction = inlier_fraction;
    ctx->n_units = b->n_units;
    ctx->mode = b->mode;
    {
        const char* env = std::getenv("MMRS_EARLY_BREAK");   // A/B runs and tests: 0 = K1 everywhere, 1 = K1e wherever it fits
        ctx->eb_env = (env && *env) ? (*env == '0' ? 0 : 1) : -1;
    }
    ctx->opt_rel = (o && o->shortlist_rel > 0) ? o->shortlist_rel : 2e-6;
    ctx->opt_abs = (o && o->shortlist_abs > 0) ? o->shortlist_abs : 2e-6;
    ctx->cap = (o && o->shortlist_cap > 0) ? o->shortlist_cap : 64;
    ctx->tie_margin = (o && o->tie_margin > 0) ? o->tie_margin : 0.0;
    ctx->opt_prune = (o && o->prune != 0) ? (o->prune > 0 ? 1 : 0) : ctx->ctx_prune;
    ctx->opt_partition = o ? o->partition : 0;
    if (ctx->opt_partition < -1 || ctx->opt_partition > 2)
        return set_err(ctx, MMRS_ERR_ARG, "mmrs_sweep_upload: partition must be -1 (off), 0 (context default), 1 (units) or 2 (angles)");
    ctx->opt_prefilter = o ? o->prefilter : 0;
    if (o && o->keep_dist32 && ctx->opt_prefilter == 0) ctx->opt_prefilter = 1;  // exact FP32 for EVERY candidate
    if (o && o->keep_dist32) ctx->opt_prune = 0;
    ctx->tc_abs = (o && o->prefilter_abs > 0) ? o->prefilter_abs : 4e-6;
    ctx->xf_abs = (o && o->prefilter_abs > 0) ? o->prefilter_abs : 8e-6;
    if (ctx->opt_prefilter < 0 || ctx->opt_prefilter > 3)
        return set_err(ctx, MMRS_ERR_ARG,
                       "mmrs_sweep_upload: prefilter must be 0 (auto), 1 (off), 2 (tensor-core tier) or 3 (expanded-form tier)");
    if (b->n_units == 0) {
        ctx->grids.clear();
        ctx->grid_of_unit.clear();
        ctx->tgrids.clear();
        ctx->tgrid_of_unit.clear();
        ctx->h_units.clear();
        ctx->h_work.clear();
        ctx->total_cands = 0;
        ctx->ready = true;
        return MMRS_OK;
    }
    int rc = upload_points(ctx, b);
    if (rc != MMRS_OK) return rc;
    rc = apply_grids(ctx, b->grids, b->n_grids, b->grid_of_unit, tgrids, n_tgrids, tgrid_of_unit);
    if (rc != MMRS_OK) return rc;
    // The host arrays (and our own staging vectors) must outlive the async copies.
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->ready = true;
    return MMRS_OK;
}

extern "C" int mmrs_sweep_upload(mmrs_ctx* ctx, const mmrs_sweep_batch* b, const mmrs_sweep_opts* o) {
    return upload_impl(ctx, b, o, nullptr, 0, nullptr, "mmrs_sweep_upload");
}

extern "C" int mmrs_rigid_sweep_upload(mmrs_ctx* ctx, const mmrs_sweep_batch* b, const mmrs_tgrid* tgrids, int64_t n_tgrids,
                                       const int32_t* tgrid_of_unit, const mmrs_sweep_opts* o) {
    if (!tgrids && ctx) return set_err(ctx, MMRS_ERR_ARG, "mmrs_rigid_sweep_upload: bad translation grids");
    return upload_impl(ctx, b, o, tgrids, n_tgrids, tgrid_of_unit, "mmrs_rigid_sweep_upload");
}

extern "C" int mmrs_partial_sweep_upload(mmrs_ctx* ctx, const mmrs_sweep_batch* b, const mmrs_tgrid* tgrids,
                                         int64_t n_tgrids, const int32_t* tgrid_of_unit, double inlier_fraction,
                                         const mmrs_sweep_opts* o) {
    if (!ctx) return set_err(nullptr, MMRS_ERR_ARG, "mmrs_partial_sweep_upload: ctx is NULL");
    if (!std::isfinite(inlier_fraction) || !(inlier_fraction > 0.0) || inlier_fraction > 1.0)
        return set_err(ctx, MMRS_ERR_ARG, "mmrs_partial_sweep_upload: inlier_fraction must be finite with 0 < f <= 1");
    if (!tgrids && (n_tgrids || tgrid_of_unit)) return set_err(ctx, MMRS_ERR_ARG, "mmrs_partial_sweep_upload: bad translation grids");
    return upload_impl(ctx, b, o, tgrids, n_tgrids, tgrid_of_unit,
                       inlier_fraction < 1.0 ? "mmrs_partial_sweep_upload"
                       : tgrids              ? "mmrs_rigid_sweep_upload"
                                             : "mmrs_sweep_upload",
                       inlier_fraction < 1.0 ? kCostPartial : kCostFull, inlier_fraction);
}

extern "C" int mmrs_mean_sweep_upload(mmrs_ctx* ctx, const mmrs_sweep_batch* b, const mmrs_tgrid* tgrids,
                                      int64_t n_tgrids, const int32_t* tgrid_of_unit, const mmrs_sweep_opts* o) {
    if (!ctx) return set_err(nullptr, MMRS_ERR_ARG, "mmrs_mean_sweep_upload: ctx is NULL");
    if (!tgrids && (n_tgrids || tgrid_of_unit)) return set_err(ctx, MMRS_ERR_ARG, "mmrs_mean_sweep_upload: bad translation grids");
    return upload_impl(ctx, b, o, tgrids, n_tgrids, tgrid_of_unit, "mmrs_mean_sweep_upload", kCostMean);
}

static int regrid_impl(mmrs_ctx* ctx, const mmrs_grid* grids, int64_t n_grids, const int32_t* grid_of_unit,
                       const mmrs_tgrid* tgrids, int64_t n_tgrids, const int32_t* tgrid_of_unit, double tie_margin,
                       const char* fn) {
    if (!ctx) return set_err(nullptr, MMRS_ERR_ARG, std::string(fn) + ": ctx is NULL");
    if (!ctx->ready) return set_err(ctx, MMRS_ERR_STATE, std::string(fn) + ": no batch uploaded");
    if (tgrids || n_tgrids)
        if (int rc = check_tgrids(ctx, fn, ctx->n_units, tgrids, n_tgrids, tgrid_of_unit)) return rc;
    if (ctx->n_units == 0) return MMRS_OK;
    if (!grids || n_grids < 1) return set_err(ctx, MMRS_ERR_ARG, std::string(fn) + ": bad grids");
    ENTER_DEVICE(ctx);
    ctx->ready = false;
    ctx->ran = false;
    ctx->tie_margin = tie_margin > 0 ? tie_margin : 0.0;
    ctx->upload_launches = 0;
    int rc = apply_grids(ctx, grids, n_grids, grid_of_unit, tgrids, n_tgrids, tgrid_of_unit);
    if (rc != MMRS_OK) return rc;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->ready = true;
    return MMRS_OK;
}

extern "C" int mmrs_sweep_regrid(mmrs_ctx* ctx, const mmrs_grid* grids, int64_t n_grids, const int32_t* grid_of_unit,
                                 double tie_margin) {
    return regrid_impl(ctx, grids, n_grids, grid_of_unit, nullptr, 0, nullptr, tie_margin, "mmrs_sweep_regrid");
}

extern "C" int mmrs_rigid_sweep_regrid(mmrs_ctx* ctx, const mmrs_grid* grids, int64_t n_grids, const int32_t* grid_of_unit,
                                       const mmrs_tgrid* tgrids, int64_t n_tgrids, const int32_t* tgrid_of_unit,
                                       double tie_margin) {
    if (!tgrids) return set_err(ctx, MMRS_ERR_ARG, "mmrs_rigid_sweep_regrid: bad translation grids");
    return regrid_impl(ctx, grids, n_grids, grid_of_unit, tgrids, n_tgrids, tgrid_of_unit, tie_margin,
                       "mmrs_rigid_sweep_regrid");
}

// ---- run ------------------------------------------------------------------------------
// K3 launch shape: both point sets of an item in shared memory (f64), or — sets too large for it — the rotated points in
// a per-CTA scratch row in global memory (d_exact_scratch) and the reference set read in place.
struct ExactPlan {
    int smem, grid;
    double2* scratch;
    double* mins = nullptr;   // partial and mean costs: the CTAs' row minima in global memory (with scratch)
};
// The partial and mean costs also keep the row minima of one direction (max_pts doubles per CTA).
static int exact_plan(mmrs_ctx* ctx, Cost cost, int max_pts, int want_grid, ExactPlan* p) {
    const bool mins = cost != kCostFull;
    const long long smem = 64 + 2LL * max_pts * 16 + (mins ? (long long)max_pts * 8 : 0);
    if (smem <= kMaxDynSmem) {
        *p = ExactPlan{(int)smem, want_grid, nullptr};
        return MMRS_OK;
    }
    const int grid = std::max(1, std::min(want_grid, ctx->n_sm * 2));
    const size_t rot = (size_t)grid * max_pts * 16;
    ENSURE(ctx->d_exact_scratch, mins ? (size_t)grid * max_pts * 24 : rot);
    char* base = (char*)ctx->d_exact_scratch.p;
    *p = ExactPlan{64, grid, (double2*)base, mins ? (double*)(base + rot) : nullptr};
    return MMRS_OK;
}

// K3 of a cost (k_exact<COST>, and k_exact_dense<COST> for a whole unit), its shared-memory limit raised once.
using ExactKernel = decltype(&k_exact<kCostFull>);
using ExactDenseKernel = decltype(&k_exact_dense<kCostFull>);
static cudaError_t exact_kernel(Cost c, ExactKernel* k) {
    switch (c) {
        case kCostPartial: *k = k_exact<kCostPartial>; return RAISE_SMEM(k_exact<kCostPartial>);
        case kCostMean: *k = k_exact<kCostMean>; return RAISE_SMEM(k_exact<kCostMean>);
        default: *k = k_exact<kCostFull>; return RAISE_SMEM(k_exact<kCostFull>);
    }
}
static cudaError_t exact_kernel(Cost c, ExactDenseKernel* k) {
    switch (c) {
        case kCostPartial: *k = k_exact_dense<kCostPartial>; return RAISE_SMEM(k_exact_dense<kCostPartial>);
        case kCostMean: *k = k_exact_dense<kCostMean>; return RAISE_SMEM(k_exact_dense<kCostMean>);
        default: *k = k_exact_dense<kCostFull>; return RAISE_SMEM(k_exact_dense<kCostFull>);
    }
}

// f64 recheck of every candidate of `unit` (shortlist overflow): leftmost arg-min on the host
// over device-computed reference-arithmetic distances.
static int full_f64_unit(mmrs_ctx* ctx, int64_t u, UnitResultDev& r) {
    const UnitDesc& d = ctx->h_units[u];
    ENSURE(ctx->d_tmp, (size_t)d.n_cand * 8);
    ExactPlan ep;
    if (int rc = exact_plan(ctx, ctx->cost, ctx->max_pts, std::min(d.n_cand, ctx->n_sm * 8), &ep)) return rc;
    ExactDenseKernel k3;
    CUDA_TRY(ctx, exact_kernel(ctx->cost, &k3));
    k3<<<ep.grid, 256, ep.smem, ctx->stream>>>((const UnitDesc*)ctx->d_units.p, (int)u, (const double*)ctx->d_test.p,
                                               (const double*)ctx->d_ref.p, (const double2*)ctx->d_cs64.p,
                                               (const unsigned char*)ctx->d_zero.p, d.cand_off, d.n_cand,
                                               (double*)ctx->d_tmp.p, ctx->max_pts, ep.scratch, ep.mins,
                                               ctx->rigid ? (const double2*)ctx->d_t64.p : nullptr, false);
    CUDA_TRY(ctx, cudaGetLastError());
    std::vector<double> h(d.n_cand);
    CUDA_TRY(ctx, cudaMemcpyAsync(h.data(), ctx->d_tmp.p, (size_t)d.n_cand * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->launches += 1;
    int best = 0;
    for (int c = 1; c < d.n_cand; ++c)
        if (h[c] < h[best]) best = c;
    const double lim = h[best] + ctx->tie_margin * std::fmax(1.0, (double)ctx->h_rmax[u]);
    int ties = 1;
    const double* cs = ctx->h_cs.data() + 2 * d.cand_off;
    const int T = d.n_trans;   // rigid candidates: a tie is a different (cos, sin) or a different (tx, ty)
    const double* tt = ctx->rigid ? ctx->h_t.data() + 2 * d.t_off : nullptr;
    const int bi = best / T, bj = best % T;
    for (int c = 0; c < d.n_cand; ++c) {
        if (c == best || h[c] > lim) continue;
        const int i = c / T, j = c % T;
        bool differs = cs[2 * i] != cs[2 * bi] || cs[2 * i + 1] != cs[2 * bi + 1];
        if (tt) differs = differs || tt[2 * j] != tt[2 * bj] || tt[2 * j + 1] != tt[2 * bj + 1];
        if (differs) ++ties;
    }
    r.best_idx = best;
    r.best_dist = h[best];
    r.n_shortlist = d.n_cand;
    r.n_ties = ties;
    r.flags |= MMRS_FLAG_FULL_F64;
    ctx->overflow_dist[u] = std::move(h);
    return MMRS_OK;
}

// Re-scores a candidate list (in d_l1_items) with the exact FP32 sweep: one launch per size class, each scoring the list
// items of its own units. n_items: the list's device counter (NULL: exactly `cap` items); diag: slot of d_l1_n that
// receives the kernel's diagnostic.
static int rescore_list(mmrs_ctx* ctx, const unsigned* n_items, unsigned cap, int chunk, int diag) {
    const ListArgs la{(const int2*)ctx->d_l1_items.p, n_items, cap, chunk, (const unsigned*)ctx->d_rmax.p,
                      (unsigned*)ctx->d_l1_n.p + diag};
    const int grid = (int)(((long long)la.cap + la.chunk - 1) / la.chunk);
    for (const auto& cl : ctx->classes) {
        if (!launch_sweep(cl.ta, cl.multi, cl.tailp, grid, cl.smem, ctx->stream, (const UnitDesc*)ctx->d_units.p, nullptr,
                          (const float4*)ctx->d_lay.p, (const float2*)ctx->d_cs32.p, (float*)ctx->d_dist32.p,
                          (unsigned long long*)ctx->d_key.p, &la))
            return set_err(ctx, MMRS_ERR_ARG, "no sweep kernel for this register tile");
        ctx->launches += 1;
    }
    CUDA_TRY(ctx, cudaGetLastError());
    return MMRS_OK;
}

// Tier 1 and 2 of every tier: the candidates inside the window (rel, abs, k_shortlist `mode`) of each unit's minimum in
// `key` go to the list, which is re-scored with the exact FP32 sweep.
static int rescore_window(mmrs_ctx* ctx, const unsigned long long* key, float rel, float abs, int mode, int chunk, int diag) {
    cudaStream_t s = ctx->stream;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_tc[1], s));
    k_shortlist<<<(unsigned)ctx->n_units, 256, 0, s>>>((const UnitDesc*)ctx->d_units.p, (const float*)ctx->d_dist32.p, key,
                                                       (const unsigned*)ctx->d_rmax.p, rel, abs, ctx->l1_cap,
                                                       (int*)ctx->d_l1_count.p, (unsigned*)ctx->d_l1_base.p,
                                                       (int2*)ctx->d_l1_items.p, (unsigned*)ctx->d_l1_n.p, mode, nullptr);
    CUDA_TRY(ctx, cudaGetLastError());
    ctx->launches += 1;
    if (int rc = rescore_list(ctx, (const unsigned*)ctx->d_l1_n.p, ctx->l1_cap, chunk, diag)) return rc;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_tc[2], s));
    return MMRS_OK;
}

// Lower-bound pruning (K1p): bounds of every candidate; the candidate with the smallest bound is scored first, and only
// the candidates whose bound is within the window of that exact distance are scored after it.
static int run_prune(mmrs_ctx* ctx) {
    const int64_t U = ctx->n_units;
    cudaStream_t s = ctx->stream;
    const UnitDesc* units = (const UnitDesc*)ctx->d_units.p;
    // tier 0: lower bounds of every candidate (rows-only passes over R strided points of each set)
    const UnitDesc* lbu = (const UnitDesc*)ctx->d_units_lb.p;
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_dist32.p, 0, (size_t)ctx->total_cands * 4, s));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_l1_n.p, 0, 16, s));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_tc[0], s));
    if (ctx->lb_R == 128) {
        CUDA_TRY(ctx, RAISE_SMEM((k_lb<4, 2>)));
        k_lb<4, 2><<<(unsigned)ctx->h_work_lb.size(), kThreads, ctx->smem_lb, s>>>(
            lbu, (const WorkItem*)ctx->d_work_lb.p, (const float4*)ctx->d_lay_lb.p, (const float2*)ctx->d_cs32.p,
            (float*)ctx->d_dist32.p);
    } else {
        CUDA_TRY(ctx, RAISE_SMEM((k_lb<1, 8>)));
        k_lb<1, 8><<<(unsigned)ctx->h_work_lb.size(), kThreads, ctx->smem_lb, s>>>(
            lbu, (const WorkItem*)ctx->d_work_lb.p, (const float4*)ctx->d_lay_lb.p, (const float2*)ctx->d_cs32.p,
            (float*)ctx->d_dist32.p);
    }
    CUDA_TRY(ctx, cudaGetLastError());
    // the candidate with the smallest bound is scored first: its exact FP32 distance bounds the minimum from above
    k_lb_argmin<<<(unsigned)U, 256, 0, s>>>(units, (const float*)ctx->d_dist32.p, (int*)ctx->d_l1_count.p,
                                            (unsigned*)ctx->d_l1_base.p, (int2*)ctx->d_l1_items.p);
    CUDA_TRY(ctx, cudaGetLastError());
    ctx->launches += 2;
    if (int rc = rescore_list(ctx, nullptr, (unsigned)U, 1, 2)) return rc;   // k_lb_argmin's list: one item per unit
    // survivors: bound <= that distance + twice the FP32 window; everything else cannot be the arg-min
    return rescore_window(ctx, (const unsigned long long*)ctx->d_key.p, 4e-6f, 4e-6f, 0, 32, 2);
}

// MMRS_TC_TRACE (experiments): the per-tile clock stamps of K1t's CTA 0, as a text file at `path`.
static int dump_tc_trace(mmrs_ctx* ctx, const long long* d_trace, const char* path) {
    cudaStream_t s = ctx->stream;
    std::vector<long long> h(8 * 256 + 64 * 8);
    CUDA_TRY(ctx, cudaMemcpyAsync(h.data(), d_trace, h.size() * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    if (FILE* f = std::fopen(path, "w")) {
        std::fprintf(f, "tile wg issuer_ready issuer_committed epi_woken epi_released\n");
        for (int g = 0; g < 2; ++g)
            for (int t = 0; t < 256; ++t)
                std::fprintf(f, "%d %d %lld %lld %lld %lld\n", t, g, h[(g * 4 + 0) * 256 + t], h[(g * 4 + 1) * 256 + t],
                             h[(g * 4 + 2) * 256 + t], h[(g * 4 + 3) * 256 + t]);
        std::fprintf(f, "fine stamps (wg 0, quarter 0): tile start ld0_done fold0_done wait1_done wait3_done fold3_done fenced\n");
        for (int t = 0; t < 64; ++t) {
            std::fprintf(f, "%d", t);
            for (int k = 0; k < 7; ++k) std::fprintf(f, " %lld", h[2048 + t * 8 + k] - h[2048 + t * 8]);
            std::fprintf(f, " | woken->start %lld, fenced->released %lld\n", h[2048 + t * 8] - h[(0 * 4 + 2) * 256 + t],
                         h[(0 * 4 + 3) * 256 + t] - h[2048 + t * 8 + 6]);
        }
        std::fclose(f);
    }
    return MMRS_OK;
}

// Tensor-core prefilter (K1t): every candidate on the tensor cores, then the candidates inside its window re-scored.
static int run_tc(mmrs_ctx* ctx) {
    const int64_t U = ctx->n_units;
    cudaStream_t s = ctx->stream;
    // tier 0: every candidate on the tensor cores (bf16x3, FP32 accumulate) -> approximate dist32 + per-unit minimum
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_key_tc.p, 0xff, U * 8, s));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_l1_n.p, 0, 16, s));
    CUDA_TRY(ctx, RAISE_SMEM(k_tc_sweep));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_tc[0], s));
    const char* trace_path = std::getenv("MMRS_TC_TRACE");  // experiments: per-tile clock stamps of CTA 0
    long long* d_trace = nullptr;
    if (trace_path && *trace_path) {
        ENSURE(ctx->d_tmp, (8 * 256 + 64 * 8) * 8);
        d_trace = (long long*)ctx->d_tmp.p;
        CUDA_TRY(ctx, cudaMemsetAsync(d_trace, 0, (8 * 256 + 64 * 8) * 8, s));
    }
    k_tc_sweep<<<(unsigned)ctx->h_work_tc.size(), kTcThreads, ctx->smem_tc, s>>>(
        (const UnitDesc*)ctx->d_units.p, (const WorkItem*)ctx->d_work_tc.p, (const double*)ctx->d_test.p,
        (const double*)ctx->d_ref.p, (const float2*)ctx->d_cs32.p, (float*)ctx->d_dist32.p,
        (unsigned long long*)ctx->d_key_tc.p, d_trace);
    CUDA_TRY(ctx, cudaGetLastError());
    ctx->launches += 1;
    if (d_trace)
        if (int rc = dump_tc_trace(ctx, d_trace, trace_path)) return rc;
    return rescore_window(ctx, (const unsigned long long*)ctx->d_key_tc.p, 1e-6f, (float)ctx->tc_abs, 1, 8, 1);
}

// Expanded-form tier (K1x): every candidate in the expanded form, then the candidates inside its window re-scored in
// direct form.
static int run_xf(mmrs_ctx* ctx) {
    const int64_t U = ctx->n_units;
    cudaStream_t s = ctx->stream;
    // tier 0: every candidate in the expanded form (K1x) -> FP32 distances with a bounded ABSOLUTE error on d^2
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_key_tc.p, 0xff, U * 8, s));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_l1_n.p, 0, 16, s));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_tc[0], s));
    for (const auto& cl : ctx->classes) {
        if (!cl.work_count) continue;
        if (!launch_sweep(cl.ta, cl.multi, cl.tailp, (int)cl.work_count, cl.smem, s, (const UnitDesc*)ctx->d_units.p,
                          (const WorkItem*)ctx->d_work.p + cl.work_begin, (const float4*)ctx->d_lay.p,
                          (const float2*)ctx->d_cs32.p, (float*)ctx->d_dist32.p, (unsigned long long*)ctx->d_key_tc.p,
                          nullptr, true))
            return set_err(ctx, MMRS_ERR_ARG, "no sweep kernel for this register tile");
        CUDA_TRY(ctx, cudaGetLastError());
        ctx->launches += 1;
    }
    return rescore_window(ctx, (const unsigned long long*)ctx->d_key_tc.p, 4e-6f, (float)ctx->xf_abs, 2, 16, 1);
}

// The dense sweep of one size class: K1b (k_sweep_big) for units beyond K1's shared-memory staging, else K1e-partial
// for the partial cost, K1e where the class takes it, or K1 (its mean form for the mean cost). t32 != NULL: rigid
// candidates.
static int sweep_class(mmrs_ctx* ctx, const mmrs_ctx::SweepClass& cl, const float2* t32) {
    cudaStream_t s = ctx->stream;
    const UnitDesc* units = (const UnitDesc*)ctx->d_units.p;
    const WorkItem* work = (const WorkItem*)ctx->d_work.p + cl.work_begin;
    const float4* lay = (const float4*)ctx->d_lay.p;
    const float2* cs32 = (const float2*)ctx->d_cs32.p;
    float* dist32 = (float*)ctx->d_dist32.p;
    unsigned long long* key = (unsigned long long*)ctx->d_key.p;
    if (cl.big) {
        const int grid = (int)std::min<size_t>(cl.work_count, (size_t)ctx->n_sm * 2);
        ENSURE(ctx->d_big_rows, (size_t)grid * kWarpsPerCta * ctx->big_scratch_per_warp * 4);
        auto big = t32 ? k_sweep_big<true> : k_sweep_big<false>;
        big<<<grid, kThreads, 0, s>>>(units, work, (int)cl.work_count, lay, cs32, dist32, key, (float*)ctx->d_big_rows.p,
                                      ctx->big_scratch_per_warp, t32);
    } else if (ctx->cost == kCostPartial || cl.eb) {
        if (!ctx->eb_ran) {   // one counter of the pair distances the early-break kernels evaluate in this run
            ENSURE(ctx->d_eb_pairs, 8);
            CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_eb_pairs.p, 0, 8, s));
            ctx->eb_ran = true;
        }
        unsigned long long* pairs = (unsigned long long*)ctx->d_eb_pairs.p;
        // K1e-partial for the partial cost (every class: big units are refused at upload), else K1e
        const bool partial = ctx->cost == kCostPartial;
        if (partial) CUDA_TRY(ctx, t32 ? RAISE_SMEM((k_sweep_eb<true, true>)) : RAISE_SMEM((k_sweep_eb<false, true>)));
        else CUDA_TRY(ctx, t32 ? RAISE_SMEM((k_sweep_eb<true, false>)) : RAISE_SMEM((k_sweep_eb<false, false>)));
        auto eb = partial ? (t32 ? k_sweep_eb<true, true> : k_sweep_eb<false, true>)
                               : (t32 ? k_sweep_eb<true, false> : k_sweep_eb<false, false>);
        eb<<<(unsigned)cl.work_count, cl.eb_warps * 32, cl.smem_eb, s>>>(units, work, lay, cs32, dist32, key, pairs, t32,
                                                                          ctx->eb_env != 0 ? 1 : 0);
        ctx->eb_cands += cl.live;
    } else if (!launch_sweep(cl.ta, cl.multi, cl.tailp, (int)cl.work_count, cl.smem, s, units, work, lay, cs32, dist32,
                             key, nullptr, false, t32, ctx->cost == kCostMean)) {
        return set_err(ctx, MMRS_ERR_ARG, "no sweep kernel for this register tile");
    }
    CUDA_TRY(ctx, cudaGetLastError());
    ctx->launches += 1;
    return MMRS_OK;
}

extern "C" int mmrs_sweep_run(mmrs_ctx* ctx) {
    if (!ctx) return set_err(nullptr, MMRS_ERR_ARG, "mmrs_sweep_run: ctx is NULL");
    if (!ctx->ready) return set_err(ctx, MMRS_ERR_STATE, "mmrs_sweep_run: no batch uploaded");
    ENTER_DEVICE(ctx);
    const int64_t U = ctx->n_units;
    ctx->launches = 0;
    ctx->ran = true;
    ctx->overflow_dist.clear();
    if (U == 0) return MMRS_OK;
    cudaStream_t s = ctx->stream;
    const UnitDesc* units = (const UnitDesc*)ctx->d_units.p;
    // rigid candidates: translation tables, and R_eff in place of Rmax wherever the FP32 error bound enters
    const float2* t32 = ctx->rigid ? (const float2*)ctx->d_t32.p : nullptr;
    const double2* t64 = ctx->rigid ? (const double2*)ctx->d_t64.p : nullptr;
    const unsigned* rbits = (const unsigned*)(ctx->rigid ? ctx->d_reff.p : ctx->d_rmax.p);
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_key.p, 0xff, U * 8, s));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_nitems.p, 0, 16, s));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[0], s));
    // the planned tier, or the dense sweep when the tier has no work
    const bool has_work = ctx->tier == kTierTc      ? !ctx->h_work_tc.empty()
                          : ctx->tier == kTierXf    ? !ctx->h_work.empty()
                          : ctx->tier == kTierPrune ? !ctx->h_work_lb.empty()
                                                    : true;
    ctx->tier_ran = has_work ? ctx->tier : kTierDense;
    ctx->eb_ran = false;
    ctx->eb_cands = 0;
    int rc = MMRS_OK;
    switch (ctx->tier_ran) {
        case kTierPrune: rc = run_prune(ctx); break;
        case kTierTc: rc = run_tc(ctx); break;
        case kTierXf: rc = run_xf(ctx); break;
        case kTierDense:
            for (const auto& cl : ctx->classes)   // one launch per size class (register tile / chunked / exact tiling)
                if (cl.work_count && (rc = sweep_class(ctx, cl, t32)) != MMRS_OK) break;
            break;
    }
    if (rc != MMRS_OK) return rc;
    // after K1t / K1x, K2 passes a unit whose tier-1 list overflowed (never re-scored in FP32) on as an overflow
    const bool listed = ctx->tier_ran == kTierTc || ctx->tier_ran == kTierXf;
    if (ctx->part_active == 2) {
        // candidate axis: the global FP32 minimum of every unit = min over ranks of the packed (distance, index) keys
        NcclApi& nc = nccl_api();
        const int rc = nc.AllReduce(ctx->d_key.p, ctx->d_key.p, (size_t)U, kNcclUint64, kNcclMin, ctx->comm, s);
        if (rc != kNcclSuccess) return set_err(ctx, MMRS_ERR_CUDA, nccl_err(rc));
        ctx->collectives += 1;
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], s));
    k_shortlist<<<(unsigned)U, 256, 0, s>>>(units, (const float*)ctx->d_dist32.p,
                                            (const unsigned long long*)ctx->d_key.p, rbits,
                                            (float)ctx->opt_rel, (float)ctx->opt_abs, ctx->pool_cap,
                                            (int*)ctx->d_sl_count.p, (unsigned*)ctx->d_sl_base.p, (int2*)ctx->d_items.p,
                                            (unsigned*)ctx->d_nitems.p, 0, listed ? (const int*)ctx->d_l1_count.p : nullptr);
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[2], s));
    {
        ExactPlan ep;
        if (int rc = exact_plan(ctx, ctx->cost, ctx->max_pts, ctx->n_sm * 8, &ep)) return rc;
        ExactKernel k3;
        CUDA_TRY(ctx, exact_kernel(ctx->cost, &k3));
        k3<<<ep.grid, 256, ep.smem, s>>>(units, (const double*)ctx->d_test.p, (const double*)ctx->d_ref.p,
                                         (const double2*)ctx->d_cs64.p, (const unsigned char*)ctx->d_zero.p,
                                         (const int2*)ctx->d_items.p, (const unsigned*)ctx->d_nitems.p, ctx->pool_cap,
                                         (double*)ctx->d_sl_dist.p, ctx->max_pts, ep.scratch, ep.mins, t64);
        CUDA_TRY(ctx, cudaGetLastError());
        k_select<<<(unsigned)((U + 7) / 8), 256, 0, s>>>(units, (int)U, (const double2*)ctx->d_cs64.p,
                                                         (const int2*)ctx->d_items.p,
                                                         (const double*)ctx->d_sl_dist.p, (const int*)ctx->d_sl_count.p,
                                                         (const unsigned*)ctx->d_sl_base.p,
                                                         (const unsigned long long*)ctx->d_key.p, rbits,
                                                         ctx->tie_margin, (UnitResultDev*)ctx->d_res.p, t64);
        CUDA_TRY(ctx, cudaGetLastError());
    }
    ctx->launches += 3;
    if (ctx->part_active && ctx->comm) {
        NcclApi& nc = nccl_api();
        if (ctx->part_active == 1) {
            // whole units: entries of the other ranks are zero, so ONE sum over the 32-byte results is an exact merge
            static_assert(sizeof(UnitResultDev) == 32, "the merge works on 4 int64 words per unit");
            const int rc = nc.AllReduce(ctx->d_res.p, ctx->d_res.p, (size_t)U * 4, kNcclInt64, kNcclSum, ctx->comm, s);
            if (rc != kNcclSuccess) return set_err(ctx, MMRS_ERR_CUDA, nccl_err(rc));
            ctx->collectives += 1;
        } else {
            const int W = ctx->shard_world;
            ENSURE(ctx->d_res_all, (size_t)W * U * sizeof(UnitResultDev));
            ENSURE(ctx->d_cnt, (size_t)U * 16);
            int rc = nc.AllGather(ctx->d_res.p, ctx->d_res_all.p, (size_t)U * 4, kNcclInt64, ctx->comm, s);
            if (rc != kNcclSuccess) return set_err(ctx, MMRS_ERR_CUDA, nccl_err(rc));
            k_merge_angle<<<(unsigned)((U + 7) / 8), 256, 0, s>>>(
                units, (int)U, W, (const UnitResultDev*)ctx->d_res_all.p, (const double2*)ctx->d_cs64.p,
                (const int2*)ctx->d_items.p, (const double*)ctx->d_sl_dist.p, (const int*)ctx->d_sl_count.p,
                (const unsigned*)ctx->d_sl_base.p, (const unsigned long long*)ctx->d_key.p,
                (const unsigned*)ctx->d_rmax.p, ctx->tie_margin, (UnitResultDev*)ctx->d_res.p, (int4*)ctx->d_cnt.p);
            CUDA_TRY(ctx, cudaGetLastError());
            rc = nc.AllReduce(ctx->d_cnt.p, ctx->d_cnt.p, (size_t)U * 4, kNcclInt32, kNcclSum, ctx->comm, s);
            if (rc != kNcclSuccess) return set_err(ctx, MMRS_ERR_CUDA, nccl_err(rc));
            k_finish_angle<<<(unsigned)((U + 255) / 256), 256, 0, s>>>((int)U, (const int4*)ctx->d_cnt.p,
                                                                       (UnitResultDev*)ctx->d_res.p);
            CUDA_TRY(ctx, cudaGetLastError());
            ctx->launches += 2;
            ctx->collectives += 2;
        }
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[3], s));
    return MMRS_OK;
}

// ---- download ------------------------------------------------------------------------
// out: the per-unit results (best_idx = the flattened candidate index i T + j of a rigid run, best_angle = angle i);
// rout (rigid download): the same plus the angle / translation indices and the translation of the winner.
static int download_impl(mmrs_ctx* ctx, mmrs_unit_result* out, mmrs_rigid_result* rout, const char* fn) {
    if (!ctx) return set_err(nullptr, MMRS_ERR_ARG, std::string(fn) + ": ctx is NULL");
    if (!ctx->ready || !ctx->ran) return set_err(ctx, MMRS_ERR_STATE, std::string(fn) + ": nothing has been run");
    const int64_t U = ctx->n_units;
    if (U == 0) return MMRS_OK;
    if (!out && !rout) return set_err(ctx, MMRS_ERR_ARG, std::string(fn) + ": out is NULL");
    ENTER_DEVICE(ctx);
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_res, ctx->d_res.p, U * sizeof(UnitResultDev), cudaMemcpyDeviceToHost,
                                  ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (std::getenv("MMRS_TRACE")) {  // device time of this run on stderr
        static const char* const kTierLabel[] = {"dense;", "tc:", "pruned:", "expanded:"};
        float t[4] = {0, 0, 0, 0}, a = 0, b = 0;
        cudaEventElapsedTime(&t[0], ctx->ev[0], ctx->ev[1]);
        cudaEventElapsedTime(&t[1], ctx->ev[1], ctx->ev[2]);
        cudaEventElapsedTime(&t[2], ctx->ev[2], ctx->ev[3]);
        if (ctx->tier_ran != kTierDense) {
            cudaEventElapsedTime(&a, ctx->ev_tc[0], ctx->ev_tc[1]);
            cudaEventElapsedTime(&b, ctx->ev_tc[1], ctx->ev_tc[2]);
        }
        long long scored = 0;
        int worst = 0;
        if (ctx->tier_ran != kTierDense) {
            std::vector<int> cnt((size_t)U);
            cudaMemcpy(cnt.data(), ctx->d_l1_count.p, (size_t)U * 4, cudaMemcpyDeviceToHost);
            for (int c : cnt) scored += c > 0 ? c : 0, worst = std::max(worst, c);
        }
        std::fprintf(stderr, "[mmrs]   run: %lld units, %lld candidates, sweep %.2f ms (%s tier0 %.2f + tier1 %.2f; %lld scored exactly, "
                     "largest unit list %d), shortlist %.2f, recheck %.2f\n",
                     (long long)U, ctx->total_cands, t[0], kTierLabel[ctx->tier_ran], a, b, scored,
                     worst, t[1], t[2]);
    }
    if (ctx->part_active == 1 && !ctx->comm && ctx->exchange) {
        // host transport: the same exact sum-merge through the caller's all-reduce
        if (ctx->exchange(ctx->exchange_user, reinterpret_cast<int64_t*>(ctx->h_res), (int64_t)U * 4) != 0)
            return set_err(ctx, MMRS_ERR_CUDA, "mmrs: the exchange callback (all-reduce of per-unit results) failed");
        ctx->collectives += 1;
    }
    const UnitResultDev* hr = (const UnitResultDev*)ctx->h_res;
    bool need_rmax = false;
    for (int64_t u = 0; u < U; ++u)
        if (hr[u].n_shortlist < 0) need_rmax = true;
    if (need_rmax) {   // tie margin of the full f64 recheck: R_eff for rigid candidates
        ctx->h_rmax.resize(U);
        CUDA_TRY(ctx, cudaMemcpy(ctx->h_rmax.data(), ctx->rigid ? ctx->d_reff.p : ctx->d_rmax.p, U * 4, cudaMemcpyDeviceToHost));
    }
    for (int64_t u = 0; u < U; ++u) {
        UnitResultDev r = hr[u];
        const mmrs_grid& g = ctx->grids[ctx->grid_of_unit[u]];
        const int T = ctx->h_units[u].n_trans;
        mmrs_unit_result o;
        if (r.flags & MMRS_FLAG_DEGENERATE) {
            o = mmrs_unit_result{-1, g.fallback, 0.0, 0.0f, 0, 0, r.flags};
        } else if (r.flags & MMRS_FLAG_EMPTY) {  // every candidate costs 0.0 -> leftmost wins (process_utils.rs:86-88)
            o = mmrs_unit_result{0, mmrs_grid_angle(&g, 0), 0.0, 0.0f, 0, (int32_t)(g.n_cand * T), r.flags};
        } else {
            if (r.n_shortlist < 0) {
                int rc = full_f64_unit(ctx, u, r);
                if (rc != MMRS_OK) return rc;
            }
            o.best_idx = r.best_idx;
            o.best_angle = mmrs_grid_angle(&g, r.best_idx / T);
            o.best_dist = r.best_dist;
            o.best_dist_f32 = r.best_d32;
            o.n_shortlist = r.n_shortlist;
            o.n_ties = r.n_ties;
            o.flags = r.flags;
        }
        if (out) out[u] = o;
        if (rout) {
            mmrs_rigid_result& q = rout[u];
            q.r = o;
            q.pad = 0;
            if (o.best_idx < 0) {   // degenerate angle grid: the fallback angle at the translation grid's centre
                q.angle_idx = -1, q.trans_idx = -1;
                q.best_tx = ctx->rigid ? ctx->tgrids[ctx->tgrid_of_unit[u]].t0x : 0.0;
                q.best_ty = ctx->rigid ? ctx->tgrids[ctx->tgrid_of_unit[u]].t0y : 0.0;
            } else {
                q.angle_idx = o.best_idx / T, q.trans_idx = (int32_t)(o.best_idx % T);
                q.best_tx = ctx->rigid ? ctx->h_t[2 * (ctx->h_units[u].t_off + q.trans_idx)] : 0.0;
                q.best_ty = ctx->rigid ? ctx->h_t[2 * (ctx->h_units[u].t_off + q.trans_idx) + 1] : 0.0;
            }
        }
    }
    return MMRS_OK;
}

extern "C" int mmrs_sweep_download(mmrs_ctx* ctx, mmrs_unit_result* out) {
    return download_impl(ctx, out, nullptr, "mmrs_sweep_download");
}

extern "C" int mmrs_rigid_sweep_download(mmrs_ctx* ctx, mmrs_rigid_result* out) {
    return download_impl(ctx, nullptr, out, "mmrs_rigid_sweep_download");
}

extern "C" int mmrs_rigid_sweep_batched(mmrs_ctx* ctx, const mmrs_sweep_batch* batch, const mmrs_tgrid* tgrids,
                                        int64_t n_tgrids, const int32_t* tgrid_of_unit, const mmrs_sweep_opts* opts,
                                        mmrs_rigid_result* out) {
    int rc = mmrs_rigid_sweep_upload(ctx, batch, tgrids, n_tgrids, tgrid_of_unit, opts);
    if (rc != MMRS_OK) return rc;
    rc = mmrs_sweep_run(ctx);
    if (rc != MMRS_OK) return rc;
    return mmrs_rigid_sweep_download(ctx, out);
}

extern "C" int mmrs_sweep_batched(mmrs_ctx* ctx, const mmrs_sweep_batch* batch, const mmrs_sweep_opts* opts,
                                  mmrs_unit_result* out) {
    int rc = mmrs_sweep_upload(ctx, batch, opts);
    if (rc != MMRS_OK) return rc;
    rc = mmrs_sweep_run(ctx);
    if (rc != MMRS_OK) return rc;
    return mmrs_sweep_download(ctx, out);
}

// ---- diagnostics -----------------------------------------------------------------------
extern "C" int mmrs_sweep_get_dist32(mmrs_ctx* ctx, int64_t unit, float* out, int64_t cap) {
    if (!ctx || !ctx->ready || !ctx->ran) return set_err(ctx, MMRS_ERR_STATE, "mmrs_sweep_get_dist32: nothing has been run");
    if (unit < 0 || unit >= ctx->n_units) return set_err(ctx, MMRS_ERR_ARG, "unit out of range");
    const UnitDesc& d = ctx->h_units[unit];
    const int64_t n = std::min<int64_t>(cap, d.n_cand);
    ENTER_DEVICE(ctx);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (n > 0)
        CUDA_TRY(ctx, cudaMemcpy(out, (const float*)ctx->d_dist32.p + d.dist_off, n * 4, cudaMemcpyDeviceToHost));
    return MMRS_OK;
}

extern "C" int mmrs_sweep_get_shortlist(mmrs_ctx* ctx, int64_t unit, int64_t* idx_out, double* dist_out, int32_t cap,
                                        int32_t* n_out) {
    if (!ctx || !ctx->ready || !ctx->ran)
        return set_err(ctx, MMRS_ERR_STATE, "mmrs_sweep_get_shortlist: nothing has been run");
    if (unit < 0 || unit >= ctx->n_units) return set_err(ctx, MMRS_ERR_ARG, "unit out of range");
    ENTER_DEVICE(ctx);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    auto ov = ctx->overflow_dist.find(unit);
    if (ov != ctx->overflow_dist.end()) {  // the whole unit was rechecked
        const int n = (int)ov->second.size();
        *n_out = n;
        for (int i = 0; i < n && i < cap; ++i) {
            idx_out[i] = i;
            dist_out[i] = ov->second[i];
        }
        return MMRS_OK;
    }
    int n = 0;
    unsigned base = 0;
    CUDA_TRY(ctx, cudaMemcpy(&n, (const int*)ctx->d_sl_count.p + unit, 4, cudaMemcpyDeviceToHost));
    CUDA_TRY(ctx, cudaMemcpy(&base, (const unsigned*)ctx->d_sl_base.p + unit, 4, cudaMemcpyDeviceToHost));
    if (n < 0) return set_err(ctx, MMRS_ERR_STATE, "shortlist pool overflowed; call mmrs_sweep_download first");
    *n_out = n;
    const int k = std::min(n, cap);
    std::vector<int2> it(k);
    if (k > 0) {
        CUDA_TRY(ctx, cudaMemcpy(it.data(), (const int2*)ctx->d_items.p + base, (size_t)k * 8, cudaMemcpyDeviceToHost));
        CUDA_TRY(ctx, cudaMemcpy(dist_out, (const double*)ctx->d_sl_dist.p + base, (size_t)k * 8, cudaMemcpyDeviceToHost));
    }
    for (int i = 0; i < k; ++i) idx_out[i] = it[i].y;
    return MMRS_OK;
}

extern "C" int mmrs_sweep_plan(mmrs_ctx* ctx, int64_t plan_out[5]) {
    if (!ctx || !plan_out) return set_err(ctx, MMRS_ERR_ARG, "mmrs_sweep_plan: NULL argument");
    if (!ctx->ready) return set_err(ctx, MMRS_ERR_STATE, "mmrs_sweep_plan: no batch uploaded");
    // the size class that carries most of the work
    const mmrs_ctx::SweepClass* top = nullptr;
    for (const auto& cl : ctx->classes)
        if (!top || cl.cost > top->cost) top = &cl;
    plan_out[0] = top ? top->ta : 0;
    plan_out[1] = top ? (top->multi ? 1 : 0) | (top->tailp ? 2 : 0) | (top->big ? 4 : 0) : 0;
    plan_out[2] = (int64_t)ctx->h_work.size();
    plan_out[3] = top ? (int64_t)top->smem : 0;
    plan_out[4] = (int64_t)ctx->classes.size();
    return MMRS_OK;
}

extern "C" int mmrs_last_timings(mmrs_ctx* ctx, float ms_out[4], int32_t* launches_out) {
    if (!ctx || !ctx->ran) return set_err(ctx, MMRS_ERR_STATE, "mmrs_last_timings: nothing has been run");
    ENTER_DEVICE(ctx);
    for (int i = 0; i < 4; ++i) ms_out[i] = 0.f;
    if (ctx->n_units > 0) {
        CUDA_TRY(ctx, cudaEventSynchronize(ctx->ev[3]));
        CUDA_TRY(ctx, cudaEventElapsedTime(&ms_out[0], ctx->ev[0], ctx->ev[1]));
        CUDA_TRY(ctx, cudaEventElapsedTime(&ms_out[1], ctx->ev[1], ctx->ev[2]));
        CUDA_TRY(ctx, cudaEventElapsedTime(&ms_out[2], ctx->ev[2], ctx->ev[3]));
        CUDA_TRY(ctx, cudaEventElapsedTime(&ms_out[3], ctx->ev[0], ctx->ev[3]));
    }
    if (launches_out) *launches_out = ctx->launches;
    return MMRS_OK;
}

// ---- explicit-angle exact evaluation ----------------------------------------------------
// txy == NULL: rotation only; otherwise candidate k is (angles[k], txy[2k], txy[2k+1]).
// The partial (inlier_fraction) and mean costs: on the finite points of each set (as the sweep uploads them).
static int eval_exact_impl(mmrs_ctx* ctx, const double* test_xy, int64_t n_test, const double* ref_xy, int64_t n_ref,
                           double cx, double cy, int32_t mode, const double* angles, const double* txy, int64_t n_angles,
                           double* dist_out, const char* fn, Cost cost = kCostFull, double inlier_fraction = 1.0) {
    if (!ctx) return set_err(nullptr, MMRS_ERR_ARG, std::string(fn) + ": ctx is NULL");
    if (n_test < 0 || n_ref < 0 || n_angles < 0 || (n_angles > 0 && (!angles || !dist_out)))
        return set_err(ctx, MMRS_ERR_ARG, std::string(fn) + ": bad arguments");
    std::vector<double> f_test, f_ref;
    if (cost != kCostFull) {
        if ((n_test > 0 && !test_xy) || (n_ref > 0 && !ref_xy)) return set_err(ctx, MMRS_ERR_ARG, std::string(fn) + ": bad arguments");
        auto finite = [](const double* xy, int64_t n, std::vector<double>& out) {
            for (int64_t i = 0; i < n; ++i)
                if (std::isfinite(xy[2 * i]) && std::isfinite(xy[2 * i + 1])) out.push_back(xy[2 * i]), out.push_back(xy[2 * i + 1]);
        };
        finite(test_xy, n_test, f_test);
        finite(ref_xy, n_ref, f_ref);
        test_xy = f_test.data(), n_test = (int64_t)f_test.size() / 2;
        ref_xy = f_ref.data(), n_ref = (int64_t)f_ref.size() / 2;
        if (n_test > (1 << 24) || n_ref > (1 << 24)) return set_err(ctx, MMRS_ERR_ARG, std::string(fn) + ": too many points");
    }
    if (n_angles == 0) return MMRS_OK;
    if (n_test == 0 || n_ref == 0) {  // process_utils.rs:86-88
        for (int64_t i = 0; i < n_angles; ++i) dist_out[i] = 0.0;
        return MMRS_OK;
    }
    ENTER_DEVICE(ctx);
    cudaStream_t s = ctx->stream;
    std::vector<double> cs(2 * n_angles);
    std::vector<unsigned char> zero(n_angles);
    for (int64_t i = 0; i < n_angles; ++i) {
        cs[2 * i] = std::cos(angles[i]);
        cs[2 * i + 1] = std::sin(angles[i]);
        zero[i] = (mode == 0 && angles[i] == 0.0) ? 1 : 0;
    }
    // private scratch (does not disturb an uploaded batch)
    const size_t b_pts = (size_t)(n_test + n_ref) * 16, b_cs = (size_t)n_angles * 16, b_out = (size_t)n_angles * 8;
    const size_t o_cs = (b_pts + 255) / 256 * 256, o_zero = o_cs + (b_cs + 255) / 256 * 256,
                 o_out = o_zero + ((size_t)n_angles + 255) / 256 * 256, o_unit = o_out + (b_out + 255) / 256 * 256,
                 o_t = o_unit + 256;
    ENSURE(ctx->d_tmp, o_t + (txy ? b_cs : 0));
    unsigned char* base = (unsigned char*)ctx->d_tmp.p;
    UnitDesc d{};
    d.test_off = 0;
    d.ref_off = 0;
    d.n = (int)n_test;
    d.m = (int)n_ref;
    d.cx = cx;
    d.cy = cy;
    d.n_trans = 1;
    d.q_fwd = (short)partial_q(inlier_fraction, d.m);
    d.q_bwd = (short)partial_q(inlier_fraction, d.n);
    if (txy) CUDA_TRY(ctx, cudaMemcpyAsync(base + o_t, txy, b_cs, cudaMemcpyHostToDevice, s));
    CUDA_TRY(ctx, cudaMemcpyAsync(base, test_xy, (size_t)n_test * 16, cudaMemcpyHostToDevice, s));
    CUDA_TRY(ctx, cudaMemcpyAsync(base + (size_t)n_test * 16, ref_xy, (size_t)n_ref * 16, cudaMemcpyHostToDevice, s));
    CUDA_TRY(ctx, cudaMemcpyAsync(base + o_cs, cs.data(), b_cs, cudaMemcpyHostToDevice, s));
    CUDA_TRY(ctx, cudaMemcpyAsync(base + o_zero, zero.data(), (size_t)n_angles, cudaMemcpyHostToDevice, s));
    CUDA_TRY(ctx, cudaMemcpyAsync(base + o_unit, &d, sizeof(UnitDesc), cudaMemcpyHostToDevice, s));
    const int max_n = (int)std::max(n_test, n_ref);
    ExactPlan ep;
    const int want_grid = (int)std::min<int64_t>(n_angles, (int64_t)ctx->n_sm * 8);
    if (int rc = exact_plan(ctx, cost, max_n, want_grid, &ep)) return rc;
    ExactDenseKernel k3;
    CUDA_TRY(ctx, exact_kernel(cost, &k3));
    k3<<<ep.grid, 256, ep.smem, s>>>((const UnitDesc*)(base + o_unit), 0, (const double*)base,
                                     (const double*)(base + (size_t)n_test * 16), (const double2*)(base + o_cs),
                                     (const unsigned char*)(base + o_zero), 0, (int)n_angles, (double*)(base + o_out),
                                     max_n, ep.scratch, ep.mins, txy ? (const double2*)(base + o_t) : nullptr, true);
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemcpyAsync(dist_out, base + o_out, b_out, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    ctx->eval_launches += 1;
    return MMRS_OK;
}

extern "C" int mmrs_eval_exact(mmrs_ctx* ctx, const double* test_xy, int64_t n_test, const double* ref_xy,
                               int64_t n_ref, double cx, double cy, int32_t mode, const double* angles,
                               int64_t n_angles, double* dist_out) {
    return eval_exact_impl(ctx, test_xy, n_test, ref_xy, n_ref, cx, cy, mode, angles, nullptr, n_angles, dist_out,
                           "mmrs_eval_exact");
}

extern "C" int mmrs_eval_exact_rigid(mmrs_ctx* ctx, const double* test_xy, int64_t n_test, const double* ref_xy,
                                     int64_t n_ref, double cx, double cy, int32_t mode, const double* angles,
                                     const double* txy, int64_t n_cand, double* dist_out) {
    if (n_cand > 0 && !txy) return set_err(ctx, MMRS_ERR_ARG, "mmrs_eval_exact_rigid: txy is NULL");
    return eval_exact_impl(ctx, test_xy, n_test, ref_xy, n_ref, cx, cy, mode, angles, txy, n_cand, dist_out,
                           "mmrs_eval_exact_rigid");
}

extern "C" int mmrs_eval_exact_partial(mmrs_ctx* ctx, const double* test_xy, int64_t n_test, const double* ref_xy,
                                       int64_t n_ref, double cx, double cy, int32_t mode, const double* angles,
                                       const double* txy, int64_t n_cand, double inlier_fraction, double* dist_out) {
    if (!std::isfinite(inlier_fraction) || !(inlier_fraction > 0.0) || inlier_fraction > 1.0)
        return set_err(ctx, MMRS_ERR_ARG, "mmrs_eval_exact_partial: inlier_fraction must be finite with 0 < f <= 1");
    return eval_exact_impl(ctx, test_xy, n_test, ref_xy, n_ref, cx, cy, mode, angles, txy, n_cand, dist_out,
                           "mmrs_eval_exact_partial", inlier_fraction < 1.0 ? kCostPartial : kCostFull, inlier_fraction);
}

extern "C" int mmrs_eval_exact_mean(mmrs_ctx* ctx, const double* test_xy, int64_t n_test, const double* ref_xy,
                                    int64_t n_ref, double cx, double cy, int32_t mode, const double* angles,
                                    const double* txy, int64_t n_cand, double* dist_out) {
    return eval_exact_impl(ctx, test_xy, n_test, ref_xy, n_ref, cx, cy, mode, angles, txy, n_cand, dist_out,
                           "mmrs_eval_exact_mean", kCostMean);
}

// ---- FP32 peak probe ------------------------------------------------------------------------
extern "C" int mmrs_fp32_probe(mmrs_ctx* ctx, int32_t iters, double* tflops_out) {
    if (!ctx || !tflops_out) return set_err(ctx, MMRS_ERR_ARG, "mmrs_fp32_probe: bad arguments");
    ENTER_DEVICE(ctx);
    const int blocks = ctx->n_sm * 8;
    ENSURE(ctx->d_tmp, (size_t)blocks * 256 * 4);
    cudaEvent_t a, b;
    CUDA_TRY(ctx, cudaEventCreate(&a));
    CUDA_TRY(ctx, cudaEventCreate(&b));
    k_fp32_probe<<<blocks, 256, 0, ctx->stream>>>((float*)ctx->d_tmp.p, iters / 4 + 1, 1.0000001f, 1e-9f);  // warm-up
    CUDA_TRY(ctx, cudaEventRecord(a, ctx->stream));
    k_fp32_probe<<<blocks, 256, 0, ctx->stream>>>((float*)ctx->d_tmp.p, iters, 1.0000001f, 1e-9f);
    CUDA_TRY(ctx, cudaEventRecord(b, ctx->stream));
    CUDA_TRY(ctx, cudaEventSynchronize(b));
    CUDA_TRY(ctx, cudaGetLastError());
    float ms = 0;
    CUDA_TRY(ctx, cudaEventElapsedTime(&ms, a, b));
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    const double flops = (double)blocks * 256 * (double)iters * 16 * 8 * 2;
    *tflops_out = flops / (ms * 1e-3) / 1e12;
    return MMRS_OK;
}

// ---- tensor-core prefilter diagnostics -----------------------------------------------------------
extern "C" int mmrs_sweep_prefilter_info(mmrs_ctx* ctx, double out[6]) {
    if (!ctx || !out) return set_err(ctx, MMRS_ERR_ARG, "mmrs_sweep_prefilter_info: NULL argument");
    if (!ctx->ran) return set_err(ctx, MMRS_ERR_STATE, "mmrs_sweep_prefilter_info: nothing has been run");
    for (int i = 0; i < 6; ++i) out[i] = 0.0;
    out[5] = ctx->tc_abs;
    if (ctx->tier_ran == kTierDense && ctx->eb_ran) {   // the dense sweep ran K1e: [3] pairs evaluated, [4] candidates
        ENTER_DEVICE(ctx);
        CUDA_TRY(ctx, cudaEventSynchronize(ctx->ev[3]));
        unsigned long long pairs = 0;
        CUDA_TRY(ctx, cudaMemcpy(&pairs, ctx->d_eb_pairs.p, 8, cudaMemcpyDeviceToHost));
        out[3] = (double)pairs;
        out[4] = (double)ctx->eb_cands;
        return MMRS_OK;
    }
    if (ctx->tier_ran == kTierDense || ctx->n_units == 0) return MMRS_OK;
    ENTER_DEVICE(ctx);
    CUDA_TRY(ctx, cudaEventSynchronize(ctx->ev[3]));
    float a = 0.f, b = 0.f;
    CUDA_TRY(ctx, cudaEventElapsedTime(&a, ctx->ev_tc[0], ctx->ev_tc[1]));
    CUDA_TRY(ctx, cudaEventElapsedTime(&b, ctx->ev_tc[1], ctx->ev_tc[2]));
    unsigned h[2] = {0u, 0u};
    CUDA_TRY(ctx, cudaMemcpy(h, ctx->d_l1_n.p, 8, cudaMemcpyDeviceToHost));
    float err;
    std::memcpy(&err, &h[1], 4);
    out[0] = (double)ctx->tier_ran;
    if (ctx->tier_ran == kTierXf) out[5] = ctx->xf_abs;
    out[1] = a;
    out[2] = b;
    out[3] = (double)h[0];
    out[4] = (double)err;
    return MMRS_OK;
}

// ---- communicator ---------------------------------------------------------------------------------------------
extern "C" int mmrs_comm_unique_id(uint8_t id_out[MMRS_COMM_ID_BYTES]) {
    if (!id_out) return set_err(nullptr, MMRS_ERR_ARG, "mmrs_comm_unique_id: id_out is NULL");
    NcclApi& nc = nccl_api();
    if (!nc.ok()) return set_err(nullptr, MMRS_ERR_STATE, nc.error);
    static_assert(sizeof(nccl_unique_id) == MMRS_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
    nccl_unique_id id;
    const int rc = nc.GetUniqueId(&id);
    if (rc != kNcclSuccess) return set_err(nullptr, MMRS_ERR_CUDA, nccl_err(rc));
    std::memcpy(id_out, &id, sizeof id);
    return MMRS_OK;
}

extern "C" int mmrs_ctx_comm_init(mmrs_ctx* ctx, const uint8_t id[MMRS_COMM_ID_BYTES], int32_t rank, int32_t world) {
    if (!ctx || !id) return set_err(ctx, MMRS_ERR_ARG, "mmrs_ctx_comm_init: NULL argument");
    if (world < 1 || rank < 0 || rank >= world) return set_err(ctx, MMRS_ERR_ARG, "mmrs_ctx_comm_init: bad rank / world");
    NcclApi& nc = nccl_api();
    if (!nc.ok()) return set_err(ctx, MMRS_ERR_STATE, nc.error);
    ENTER_DEVICE(ctx);
    if (ctx->comm) {
        nc.CommDestroy(ctx->comm);
        ctx->comm = nullptr;
    }
    nccl_unique_id uid;
    std::memcpy(&uid, id, sizeof uid);
    nccl_comm_t comm = nullptr;
    const int rc = nc.CommInitRank(&comm, world, uid, rank);
    if (rc != kNcclSuccess) return set_err(ctx, MMRS_ERR_CUDA, nccl_err(rc));
    ctx->comm = comm;
    ctx->shard_rank = rank;
    ctx->shard_world = world;
    return MMRS_OK;
}

extern "C" int mmrs_ctx_set_partition(mmrs_ctx* ctx, int32_t axis) {
    if (!ctx) return set_err(nullptr, MMRS_ERR_ARG, "mmrs_ctx_set_partition: ctx is NULL");
    if (axis < 0 || axis > 2) return set_err(ctx, MMRS_ERR_ARG, "mmrs_ctx_set_partition: axis must be 0, 1 or 2");
    ctx->part_axis = axis;
    return MMRS_OK;
}

extern "C" int mmrs_ctx_comm_info(const mmrs_ctx* ctx, int32_t out[4]) {
    if (!ctx || !out) return MMRS_ERR_ARG;
    out[0] = ctx->shard_rank, out[1] = ctx->shard_world, out[2] = ctx->part_axis, out[3] = ctx->comm ? 1 : 0;
    return MMRS_OK;
}

// Broadcast of a host buffer from `root` to every rank through the communicator (device staging, NCCL broadcast on the
// context's stream). Used by mmrs_process_cases to hand the aligned pullbacks of one rank to the others.
int mmrs::comm_broadcast(mmrs_ctx* ctx, void* host, size_t bytes, int root) {
    if (!ctx->comm) return set_err(ctx, MMRS_ERR_STATE, "no communicator bound");
    if (bytes == 0) return MMRS_OK;
    NcclApi& nc = nccl_api();
    ENTER_DEVICE(ctx);
    ENSURE(ctx->d_bcast, bytes);
    if (ctx->shard_rank == root)
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_bcast.p, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    const int rc = nc.Broadcast(ctx->d_bcast.p, ctx->d_bcast.p, bytes, /*ncclInt8*/ 0, root, ctx->comm, ctx->stream);
    if (rc != kNcclSuccess) return set_err(ctx, MMRS_ERR_CUDA, nccl_err(rc));
    if (ctx->shard_rank != root)
        CUDA_TRY(ctx, cudaMemcpyAsync(host, ctx->d_bcast.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->collectives += 1;
    return MMRS_OK;
}

extern "C" int mmrs_ctx_set_prune(mmrs_ctx* ctx, int32_t on) {
    if (!ctx) return set_err(nullptr, MMRS_ERR_ARG, "mmrs_ctx_set_prune: ctx is NULL");
    ctx->ctx_prune = on ? 1 : 0;
    return MMRS_OK;
}
