// =============================================================================
// sweep_kernels.cuh — sm_100a device code of the Hausdorff rotation sweep.
//
//   K0  k_prep        f64 points -> centred FP32 staging layout (+ Rmax)
//   K1  k_sweep<TA>   FP32 sweep: one CTA = one unit x one tile of candidate
//                     angles, one warp = one candidate; reference contour
//                     staged in shared memory by a TMA bulk copy; test points
//                     rotated into registers; symmetric directed Hausdorff as
//                     a register-tiled min-over-M / max-over-N with packed
//                     f32x2 arithmetic (FADD2/FMUL2/FFMA2), 3-input FMNMX and
//                     warp REDUX; fused per-unit arg-min on a packed
//                     (distance, index) 64-bit key with atomicMin. Also re-scores
//                     candidate lists (LIST), runs the expanded-form tier K1x (XF) and scores the mean cost (MEAN).
//   K1e k_sweep_eb<RIGID, false>
//                     the dense sweep with early-break directed passes: every candidate's FP32 distance,
//                     bit-identical to K1, from ~1 % of the pair distances (default wherever it fits)
//   K1e-partial k_sweep_eb<RIGID, true>
//                     the same passes for the partial (rank-K) cost: per direction the q + 1 largest exact minima
//   K1b k_sweep_big   the FP32 sweep for units beyond K1's shared-memory staging (reference set streamed in blocks)
//   K1p k_prep_lb, k_lb, k_lb_argmin
//                     exact lower-bound pruning tier: candidates bounded above the best are never scored
//   K2  k_shortlist   candidates within the FP32 error window of the minimum
//   K3  k_exact<COST> the reference's f64 arithmetic, literally, on those (full, partial or mean cost)
//   K4  k_select      leftmost f64 arg-min + tie count per unit
//
// Replaces (reference paths): search_range + hausdorff_distance +
// directed_hausdorff, src/intravascular/processing/process_utils.rs:33-121, and
// the cost closures align_within.rs:99-105/:200-206, align_between.rs:189-216.
// =============================================================================
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cuda/std/type_traits>

#include "mmrs_internal.hpp"

namespace mmrs {

#ifndef MMRS_TRIP_UNROLL
#define MMRS_TRIP_UNROLL 1   // trips (four reference points each) per loop iteration of the sweep's main loop
#endif
#ifndef MMRS_EXP_NOTAIL   // timing experiments only (wrong results): skip the tail pass / the seed loads of exact tiling
#define MMRS_EXP_NOTAIL 0
#endif
#ifndef MMRS_EXP_NOSEED
#define MMRS_EXP_NOSEED 0
#endif
constexpr int kWarpsPerCta = 8;
constexpr int kThreads = kWarpsPerCta * 32;

// ---- packed FP32 helpers (Blackwell-only PTX: *.f32x2, 3-input min.f32) --------
__device__ __forceinline__ uint64_t pk(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk(uint64_t v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t sub2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ float min3(float a, float b, float c) {
    float r;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}

// ---- mbarrier + TMA bulk copy (cp.async.bulk -> SASS UBLKCP) --------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
    uint32_t ok = 0;
    while (!ok) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(phase)
            : "memory");
    }
}

// =============================================================================
// K0: f64 (x,y) -> centred FP32 staging layout.
// A block (test points, the set that is rotated; register side of K1):
//   S = ceil(TA/2) float4 slots per lane and chunk; slot k < TA/2 at (c*S+k)*32 + l holds the
//   points i0 = c*32*TA + 2k*32 + l and i1 = i0 + 32 as (x0, x1, y0, y1); for odd TA the last
//   slot holds the single point i0 = c*32*TA + (TA-1)*32 + l as (x, x, y, y).
// B block (reference points; streamed from shared memory in K1):
//   float4 j = (bx0, by0, bx1, by1) = reference points 2j and 2j+1, j < m_pairs. The packed f32x2
//   instructions take these as scalar operands broadcast to both halves (one 32-bit register
//   read instead of a 64-bit pair: the sweep is register-file-bandwidth bound, DESIGN.md §4).
// Indices past the end repeat the last point (a duplicate never changes a
// min-over-points or a max-over-points).
// NB block (after the B block): float2 j = (|b_2j|^2, |b_2j+1|^2), the squared norms the expanded-form tier adds.
// Tail block (exact tiling, UnitDesc.n_tail > 0; after the NB block): the n mod 32 test points that do not fill a
// register slot, two per float4 (x0, y0, x1, y1). K1 scores them in a short pass of its own instead of a padded slot.
// =============================================================================
// Block sizes of one unit's staging image in float4. The B block of exact tiling (n_tail > 0) is padded to 16 (TA + 1)
// float4 so that the tail pass can address its reference points lane + 32 q without clamping.
struct StageLayout {
    int a, b, nb, t;   // A, B, NB (float2 per pair of reference points, rounded up to float4) and tail blocks
    __host__ __device__ int total() const { return a + b + nb + t; }
};
__host__ __device__ inline StageLayout stage_layout(int ta, int n_chunks, int n_tail, int m_pairs) {
    const int b = n_tail > 0 ? 16 * (ta + 1) : m_pairs;
    return StageLayout{n_chunks * ((ta + 1) / 2) * 32, b, (b + 1) / 2, (n_tail + 1) / 2};
}

__global__ void k_prep(const UnitDesc* __restrict__ units, const double* __restrict__ test_xy,
                       const double* __restrict__ ref_xy, float4* __restrict__ lay, unsigned* __restrict__ rmax_bits) {
    const UnitDesc ud = units[blockIdx.x];
    if (ud.n <= 0 || ud.m <= 0) return;
    const int TA = ud.ta;
    const int half = (TA + 1) / 2, pairs = TA / 2;
    const StageLayout sl = stage_layout(TA, ud.n_chunks, ud.n_tail, ud.m_pairs);
    // exact tiling (n_tail > 0): the register slots hold the first 32 TA points only, the rest is the tail block
    const int n_main = ud.n - ud.n_tail;
    float4* A = lay + ud.lay_off;
    float4* B = A + sl.a;
    float2* NB = reinterpret_cast<float2*>(B + sl.b);
    float4* T = B + sl.b + sl.nb;
    float rmax = 0.f;
    for (int e = threadIdx.x; e < sl.a; e += blockDim.x) {
        int l = e & 31, ck = e >> 5;
        int c = ck / half, k = ck - c * half;
        int i0 = c * 32 * TA + 2 * k * 32 + l, i1 = (k < pairs) ? i0 + 32 : i0;
        i0 = min(i0, n_main - 1);
        i1 = min(i1, n_main - 1);
        const double* p0 = test_xy + 2 * (ud.test_off + i0);
        const double* p1 = test_xy + 2 * (ud.test_off + i1);
        float4 v;
        v.x = (float)(p0[0] - ud.cx);
        v.y = (float)(p1[0] - ud.cx);
        v.z = (float)(p0[1] - ud.cy);
        v.w = (float)(p1[1] - ud.cy);
        A[e] = v;
        rmax = fmaxf(rmax, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
    }
    for (int j = threadIdx.x; j < sl.b; j += blockDim.x) {
        const int j0 = min(2 * j, ud.m - 1), j1 = min(2 * j + 1, ud.m - 1);
        const double* p0 = ref_xy + 2 * (ud.ref_off + j0);
        const double* p1 = ref_xy + 2 * (ud.ref_off + j1);
        const float4 v = make_float4((float)(p0[0] - ud.cx), (float)(p0[1] - ud.cy), (float)(p1[0] - ud.cx),
                                     (float)(p1[1] - ud.cy));
        B[j] = v;
        // squared norms of the ROUNDED coordinates, formed in f64 and rounded once (expanded-form tier, K1x)
        NB[j] = make_float2((float)((double)v.x * v.x + (double)v.y * v.y), (float)((double)v.z * v.z + (double)v.w * v.w));
        rmax = fmaxf(rmax, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
    }
    if (threadIdx.x == 0 && (sl.b & 1)) NB[sl.b] = make_float2(0.f, 0.f);   // padding of the odd float4
    // tail block: float4 t = tail points 2t and 2t+1 as (x0, y0, x1, y1) (an odd count repeats the last point)
    for (int t = threadIdx.x; t < (ud.n_tail + 1) / 2; t += blockDim.x) {
        const int i0 = n_main + min(2 * t, ud.n_tail - 1), i1 = n_main + min(2 * t + 1, ud.n_tail - 1);
        const double* p0 = test_xy + 2 * (ud.test_off + i0);
        const double* p1 = test_xy + 2 * (ud.test_off + i1);
        const float4 v = make_float4((float)(p0[0] - ud.cx), (float)(p0[1] - ud.cy), (float)(p1[0] - ud.cx),
                                     (float)(p1[1] - ud.cy));
        T[t] = v;
        rmax = fmaxf(rmax, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
    }
    unsigned rb = __reduce_max_sync(0xffffffffu, __float_as_uint(rmax));
    if ((threadIdx.x & 31) == 0) atomicMax(&rmax_bits[blockIdx.x], rb);
}

// f64 (cos, sin) table -> FP32 table for K1.
__global__ void k_cs32(const double2* __restrict__ cs64, float2* __restrict__ cs32, long long n) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) cs32[i] = make_float2((float)cs64[i].x, (float)cs64[i].y);
}

// =============================================================================
// K1: the FP32 sweep.
// =============================================================================
// LIST = false: the dense sweep, work item = (unit, first candidate, candidates in this tile).
// LIST = true : exact re-scoring of a candidate list (after lower-bound pruning, or after the tensor-core prefilter of
//               tc_kernels.cuh). The list is ONE global array of (unit, candidate) items, contiguous per unit; CTA b owns
//               positions [b * l_chunk, (b + 1) * l_chunk) whatever units they belong to (it re-stages per run of equal
//               units), so the SMs stay busy however unevenly the survivors are spread over the units. Same arithmetic;
//               overwrites the dist32 entries and records the largest |d_old^2 - d_fp32^2| / Rmax^2 (the tensor-core
//               prefilter's error, checked against its window).
// TAILP = true : exact tiling for a test set of 32 TA + R points (0 < R < 32, single chunk). The R tail points would
//               waste most of a padded register slot (520 points: slot 17 carries 8 points and 24 duplicates, 4.4 % of
//               the launch), so per candidate the warp first runs a short pass with the roles swapped: every lane
//               holds ceil(M / 32) reference points in registers, the rotated tail points are broadcast two at a time;
//               the tail's row minima are finished with one REDUX each and its column minima — lane-local, no REDUX —
//               go to a per-warp shared-memory array from which the main loop seeds its column accumulators (one
//               broadcast LDS.64 per two reference points; the seed takes the free slot of the first 3-input minimum).
// XF = true    : K1x, the EXPANDED-FORM tier (dense launches only). |a - b|^2 = |b|^2 - 2 a.b + |a|^2: per packed pair of
//               test points and reference point two FFMA2 give r = |b|^2 - 2 a.b (what the row minima need: |a|^2 is
//               constant along a row and is added after the minimum) and one FADD2 gives r + |a|^2 (what the column
//               minima need) — 6 packed FP32 instructions per 2 x 2 block instead of 8 (-7 % per block measured,
//               profiles/r02_microbench_expanded_forms.txt). The price is cancellation: with Rn the largest point norm
//               the result carries an ABSOLUTE error of at most 13 u Rn^2 (u = 2^-24; one rounding each for |b|^2
//               (u), the two FMAs (3 u + 3 u: the partial sums stay below 3 Rn^2), the final add (4 u) and two for
//               |a|^2) <= 1.6e-6 Rmax^2, instead of the direct form's relative 3e-7. So K1x is a FILTER tier exactly like
//               K1 is a filter for the f64 recheck: every candidate is scored, the candidates within the error window
//               of the minimum are re-scored by the direct-form kernel (LIST), and K2/K3/K4 run unchanged on exact
//               FP32 values — the selection is bit-identical to the dense direct path. The tail pass and the odd
//               scalar slot stay in direct form (their values are exact, the seeds and minima mix freely).
// RIGID = true: rigid candidates (dense launches, direct form). Candidate c = i n_trans + j is angle i of the unit's
//               grid and translation j of its translation grid (t32, FP32); every rotated test point gets the
//               translation added once (one FADD2 per packed pair and coordinate, one FADD for the unpaired point).
// MEAN = true : the mean cost (include/mmrs_b200.h "mean cost"; dense direct-form launches). Same pairs, staging, tail
//               pass and chunk walk; only the reductions change. Each lane sums sqrtf of its completed row minima in
//               f64 (per chunk; lane 0 also takes the tail pass's REDUX'ed minima); the final column minima go, like a
//               chunked unit's intermediate ones, from lane 0 to the warp's shared row, and after the walk each lane
//               sums sqrtf of every 32nd. Then a fixed shuffle tree, one division per direction, one rounding to FP32.
//               Every padding duplicate of the staging image stays out of both sums: register slots at or past
//               n - n_tail, the last chunk's padding, the repeated last point of an odd tail and column indices at or
//               past m (an odd m's repeated last reference point, the B-block padding of exact tiling).
template <int TA, bool MULTI, bool LIST, bool TAILP, bool XF, bool RIGID = false, bool MEAN = false>
__global__ void __launch_bounds__(kThreads, 2)
    k_sweep(const UnitDesc* __restrict__ units, const WorkItem* __restrict__ work, const float4* __restrict__ lay,
            const float2* __restrict__ cs32, float* __restrict__ dist32, unsigned long long* __restrict__ key,
            const int2* __restrict__ l_items, const unsigned* __restrict__ l_nitems, unsigned l_cap, int l_chunk,
            const unsigned* __restrict__ rmax_bits, unsigned* __restrict__ diag, const float2* __restrict__ t32) {
    static_assert(TA >= 2 && TA <= 18, "register tile out of range");
    static_assert(!(TAILP && MULTI), "the tail pass is for single-chunk units");
    static_assert(!(XF && LIST), "the expanded form is a dense tier; lists are re-scored in direct form");
    static_assert(!(RIGID && (XF || LIST)), "rigid candidates run the dense direct-form sweep");
    static_assert(!(MEAN && (XF || LIST)), "the mean cost runs the dense direct-form sweep");
    constexpr int SB = TA + 1;         // TAILP: reference points per lane of the tail pass (M <= 32 SB)
    constexpr int H = TA / 2;          // packed pairs of test points per lane
    constexpr bool TAIL = (TA & 1);    // plus one unpaired point when TA is odd
    constexpr int S = H + (TAIL ? 1 : 0);
    constexpr int TU = MMRS_TRIP_UNROLL;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
    unsigned long long* s_key = reinterpret_cast<unsigned long long*>(smem_raw + 8);
    float4* sA = reinterpret_cast<float4*>(smem_raw + 16);

    // LIST: this CTA owns the global list positions [g_pos, g_hi); they may span several units (runs of equal .x).
    unsigned g_pos = 0, g_hi = 0;
    if (LIST) {
        const unsigned n_items = l_nitems ? min(*l_nitems, l_cap) : l_cap;
        g_pos = blockIdx.x * (unsigned)l_chunk;
        g_hi = min(g_pos + (unsigned)l_chunk, n_items);
        if (g_pos >= g_hi) return;  // nothing for this CTA (uniform: before any barrier)
    }
    const WorkItem w = LIST ? WorkItem{0, 0, 0, 0} : work[blockIdx.x];
    const int lane = threadIdx.x & 31, wid = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // warp-uniform for ptxas: the B-block and seed pointers live in uniform registers
    if (threadIdx.x == 0) mbar_init(bar, 1);
    uint32_t phase = 0;
    const float INF = __int_as_float(0x7f800000);
    float worst = 0.f;
    for (;;) {  // one pass for the dense sweep; one pass per run of equal units in LIST mode
    int unit = w.unit, total = w.count;
    const int2* my_items = nullptr;
    unsigned run_end = 0;
    if (LIST) {
        unit = l_items[g_pos].x;
        run_end = g_pos + 1;
        while (run_end < g_hi && l_items[run_end].x == unit) ++run_end;
        total = (int)(run_end - g_pos);
        my_items = l_items + g_pos;
        if (unit < 0) {  // neutralised entries of an overflowed reservation
            g_pos = run_end;
            if (g_pos >= g_hi) break;
            continue;
        }
    }
    const UnitDesc ud = units[unit];
    if (LIST && (ud.ta != TA || (ud.n_chunks > 1) != MULTI || (ud.n_tail > 0) != TAILP)) {
        // a run of another size class: the launch of that class scores it (uniform per CTA: before any barrier use)
        g_pos = run_end;
        if (g_pos >= g_hi) break;
        continue;
    }
    const int a_elems = ud.n_chunks * S * 32;
    const int b_elems = TAILP ? 16 * SB : ud.m_pairs;   // float4 per PAIR of reference points (exact tiling: padded)
    const int b_pts = 2 * ud.m_pairs;
    const int nb_elems = (b_elems + 1) / 2;                // float2 per PAIR of reference points: their squared norms
    const int t_elems = TAILP ? (ud.n_tail + 1) / 2 : 0;   // float4 per PAIR of tail points
    float4* sB = sA + a_elems;
    const float2* sNB = reinterpret_cast<const float2*>(sB + b_elems);
    const float4* sT = sB + b_elems + nb_elems;
    unsigned* s_col = reinterpret_cast<unsigned*>(sB + b_elems + nb_elems + t_elems);  // MULTI, MEAN: [warp][b_pts rounded up to 4]; TAILP: [warp][32 SB]

    if (threadIdx.x == 0) {
        *s_key = ~0ull;
        const uint32_t bytes = (uint32_t)(a_elems + b_elems + nb_elems + t_elems) * 16u;
        mbar_expect_tx(bar, bytes);
        tma_bulk_g2s(sA, lay + ud.lay_off, bytes, bar);
    }
    __syncthreads();
    mbar_wait(bar, phase);
    phase ^= 1u;

    unsigned long long best = ~0ull;
    unsigned* my_col = s_col + wid * (TAILP ? 32 * SB : ((b_pts + 3) & ~3));   // 16-byte aligned rows: four seeds per LDS.128
    // LIST: squared give-up threshold from the unit's best exact distance so far (bits; 0xffffffff = none yet)
    unsigned give_up = 0xffffffffu;
    if (LIST) {
        const unsigned ub_bits = (unsigned)(key[unit] >> 32);
        if (ub_bits != 0xffffffffu) {
            const float t = __uint_as_float(ub_bits) * (1.0f + 4e-6f) + 4e-6f * __uint_as_float(rmax_bits[unit]);
            give_up = __float_as_uint(t * t * (1.0f + 1e-6f));
        }
    }

    for (int ci = wid; ci < total; ci += kWarpsPerCta) {
        const int c = LIST ? my_items[ci].y : w.begin + ci;
        float2 tr = make_float2(0.f, 0.f);   // RIGID: translation of this candidate
        int ia = c;                          // RIGID: its angle index
        if (RIGID) {
            ia = c / ud.n_trans;
            tr = __ldg(&t32[ud.t_off + (c - ia * ud.n_trans)]);
        }
        const float2 cs = __ldg(&cs32[ud.cand_off + ia]);
        const uint64_t C2 = pk(cs.x, cs.x), S2 = pk(cs.y, cs.y), NS2 = pk(-cs.y, -cs.y);
        const uint64_t TX2 = pk(tr.x, tr.x), TY2 = pk(tr.y, tr.y);
        unsigned rowmax = 0u, colmax = 0u;  // bit patterns of non-negative floats order like unsigned ints
        double rsum = 0.0;                  // MEAN: this lane's sum of row values
        bool gave_up = false;

        if (TAILP) {
            // Tail pass, roles swapped: this lane's reference points lane, lane + 32, ... in registers (indices past the
            // end repeat the last stored point), the rotated tail points broadcast two at a time.
            const float2* sBp = reinterpret_cast<const float2*>(sB) + lane;
            float bx[SB], by[SB], tc[SB];
#pragma unroll
            for (int q = 0; q < SB; ++q) {
                const float2 b = sBp[32 * q];   // one base register, immediate offsets (the B block is padded to 32 SB points)
                bx[q] = b.x;
                by[q] = b.y;
                tc[q] = INF;
            }
#if MMRS_EXP_NOTAIL
            for (int t = 0; t < 0; ++t) {
#else
#pragma unroll 1
            for (int t = 0; t < t_elems; ++t) {
#endif
                const float4 a = sT[t];  // (x0, y0, x1, y1): broadcast
                const uint64_t X2 = pk(a.x, a.z), Y2 = pk(a.y, a.w);
                uint64_t PX = fma2(Y2, NS2, mul2(X2, C2)), PY = fma2(X2, S2, mul2(Y2, C2));
                if (RIGID) PX = add2(PX, TX2), PY = add2(PY, TY2);
                float r0 = INF, r1 = INF;   // row minima of the two tail points over this lane's reference points
#pragma unroll
                for (int q = 0; q < SB; q += 2) {
                    const uint64_t dxa = sub2(PX, pk(bx[q], bx[q])), dya = sub2(PY, pk(by[q], by[q]));
                    const uint64_t da = fma2(dxa, dxa, mul2(dya, dya));   // (|t0 - b_q|^2, |t1 - b_q|^2)
                    float a0, a1;
                    upk(da, a0, a1);
                    tc[q] = min3(tc[q], a0, a1);
                    if (q + 1 < SB) {
                        const uint64_t dxb = sub2(PX, pk(bx[q + 1], bx[q + 1])), dyb = sub2(PY, pk(by[q + 1], by[q + 1]));
                        const uint64_t db = fma2(dxb, dxb, mul2(dyb, dyb));
                        float b0, b1;
                        upk(db, b0, b1);
                        tc[q + 1] = min3(tc[q + 1], b0, b1);
                        r0 = min3(r0, a0, b0);
                        r1 = min3(r1, a1, b1);
                    } else {
                        r0 = fminf(r0, a0);
                        r1 = fminf(r1, a1);
                    }
                }
                const unsigned m0 = __reduce_min_sync(0xffffffffu, __float_as_uint(r0));
                const unsigned m1 = __reduce_min_sync(0xffffffffu, __float_as_uint(r1));
                if constexpr (MEAN) {
                    if (lane == 0) {   // an odd tail repeats its last point as tail point 2t + 1
                        rsum += (double)sqrtf(__uint_as_float(m0));
                        if (2 * t + 1 < ud.n_tail) rsum += (double)sqrtf(__uint_as_float(m1));
                    }
                } else {
                    rowmax = max(rowmax, max(m0, m1));
                }
            }
            __syncwarp();  // the previous candidate's main loop is done reading the seeds
#pragma unroll
            for (int q = 0; q < SB; ++q) my_col[lane + 32 * q] = __float_as_uint(tc[q]);
            __syncwarp();
        }

        for (int ch = 0; ch < ud.n_chunks; ++ch) {
            uint64_t AX[H], AY[H];           // XF: (-2 x', -2 y')
            uint64_t NA[XF ? H : 1];         // XF: |a'|^2 of the rotated FP32 points
            float row[TA];
            float tx = 0.f, ty = 0.f;
            if (TAIL) {
                const float4 a = sA[(ch * S + H) * 32 + lane];
                tx = fmaf(a.z, -cs.y, a.x * cs.x);
                ty = fmaf(a.x, cs.y, a.z * cs.x);
                if (RIGID) tx = __fadd_rn(tx, tr.x), ty = __fadd_rn(ty, tr.y);
                row[TA - 1] = INF;
            }
#pragma unroll
            for (int k = 0; k < H; ++k) {
                const float4 a = sA[(ch * S + k) * 32 + lane];
                const uint64_t X2 = pk(a.x, a.y), Y2 = pk(a.z, a.w);
                AX[k] = fma2(Y2, NS2, mul2(X2, C2));  // x' = x cos - y sin
                AY[k] = fma2(X2, S2, mul2(Y2, C2));   // y' = x sin + y cos
                if (RIGID) {                          // + t, rounded once
                    AX[k] = add2(AX[k], TX2);
                    AY[k] = add2(AY[k], TY2);
                }
                if (XF) {
                    NA[k] = fma2(AX[k], AX[k], mul2(AY[k], AY[k]));
                    const uint64_t M2 = pk(-2.f, -2.f);
                    AX[k] = mul2(AX[k], M2);          // exact scaling
                    AY[k] = mul2(AY[k], M2);
                }
                row[2 * k] = INF;
                row[2 * k + 1] = INF;
            }
            // One step = one float4 of the B block = two reference points against this lane's TA test points; c0 / c1 enter
            // holding the seeds of the two column minima (INF, the tail pass's minima, or the previous chunks' minima).
            auto step = [&](auto last_tag, const float4 B, float c0, float c1, unsigned* col_out) {
                constexpr bool LASTC = decltype(last_tag)::value;   // all test points seen after this chunk
                const uint64_t bx0 = pk(B.x, B.x), by0 = pk(B.y, B.y);
                const uint64_t bx1 = pk(B.z, B.z), by1 = pk(B.w, B.w);
                if (TAIL) {  // scalar FP32 ops for the unpaired point
                    const float ex0 = tx - B.x, ey0 = ty - B.y, ex1 = tx - B.z, ey1 = ty - B.w;
                    const float t0 = fmaf(ex0, ex0, ey0 * ey0), t1 = fmaf(ex1, ex1, ey1 * ey1);
                    row[TA - 1] = min3(row[TA - 1], t0, t1);
                    c0 = (MULTI || TAILP) ? fminf(c0, t0) : t0;  // plain single-chunk: these distances seed the column minima
                    c1 = (MULTI || TAILP) ? fminf(c1, t1) : t1;
                }
                if (XF) {
                    const float2 nb = sNB[(int)(col_out - my_col) >> 1];
                    const uint64_t n0 = pk(nb.x, nb.x), n1 = pk(nb.y, nb.y);
#pragma unroll
                    for (int k = 0; k < H; ++k) {
                        const uint64_t r0 = fma2(AX[k], bx0, fma2(AY[k], by0, n0));  // |b0|^2 - 2 a.b0 for (a0, a1)
                        const uint64_t r1 = fma2(AX[k], bx1, fma2(AY[k], by1, n1));
                        const uint64_t d0 = add2(r0, NA[k]), d1 = add2(r1, NA[k]);   // + |a|^2: the squared distances
                        float r00, r10, r01, r11, d00, d10, d01, d11;
                        upk(r0, r00, r10);
                        upk(r1, r01, r11);
                        upk(d0, d00, d10);
                        upk(d1, d01, d11);
                        row[2 * k] = min3(row[2 * k], r00, r01);
                        row[2 * k + 1] = min3(row[2 * k + 1], r10, r11);
                        c0 = min3(c0, d00, d10);
                        c1 = min3(c1, d01, d11);
                    }
                    c0 = fmaxf(c0, 0.f);   // cancellation can leave a tiny negative value: the bit-pattern order needs >= 0
                    c1 = fmaxf(c1, 0.f);
                } else {
#pragma unroll
                    for (int k = 0; k < H; ++k) {
                        const uint64_t dx0 = sub2(AX[k], bx0), dy0 = sub2(AY[k], by0);
                        const uint64_t dx1 = sub2(AX[k], bx1), dy1 = sub2(AY[k], by1);
                        const uint64_t d0 = fma2(dx0, dx0, mul2(dy0, dy0));  // (|a0-b0|^2, |a1-b0|^2)
                        const uint64_t d1 = fma2(dx1, dx1, mul2(dy1, dy1));  // (|a0-b1|^2, |a1-b1|^2)
                        float d00, d10, d01, d11;
                        upk(d0, d00, d10);
                        upk(d1, d01, d11);
                        row[2 * k] = min3(row[2 * k], d00, d01);
                        row[2 * k + 1] = min3(row[2 * k + 1], d10, d11);
                        c0 = min3(c0, d00, d10);
                        c1 = min3(c1, d01, d11);
                    }
                }
                const unsigned r0 = __reduce_min_sync(0xffffffffu, __float_as_uint(c0));
                const unsigned r1 = __reduce_min_sync(0xffffffffu, __float_as_uint(c1));
                if (LASTC && !MEAN) {
                    colmax = max(colmax, max(r0, r1));  // these are the column minima
                } else if (lane == 0) {
                    *reinterpret_cast<uint2*>(col_out) = make_uint2(r0, r1);
                }
            };
            // The B block is walked two float4 (four reference points) per trip with running pointers: one LDS.128 brings
            // the four seeds, and the addresses cost two pointer increments instead of an index computation per array.
            // Specialised on (last chunk, seeded) so that a chunked unit's loop carries no per-step branches.
            auto walk = [&](auto last_tag, auto seeded_tag) {
                constexpr bool SEEDED = decltype(seeded_tag)::value;   // MULTI: lane 0 alone carries the seeds
                const float4* pB = sB;
                unsigned* pC = my_col;
                const float4* const pB_end2 = sB + (ud.m_pairs & ~1);
#pragma unroll TU
                for (; pB != pB_end2; pB += 2, pC += 4) {
                    const float4 B0 = pB[0], B1 = pB[1];
                    float s0 = INF, s1 = INF, s2 = INF, s3 = INF;
                    if (SEEDED && (TAILP || lane == 0)) {
                        const uint4 sd = *reinterpret_cast<const uint4*>(pC);
                        s0 = __uint_as_float(sd.x), s1 = __uint_as_float(sd.y), s2 = __uint_as_float(sd.z), s3 = __uint_as_float(sd.w);
                    }
                    step(last_tag, B0, s0, s1, pC);
                    // LIST: a column minimum above the unit's best exact distance (+ window) already proves that this
                    // candidate cannot win: stop, and keep the proven lower bound (uniform across the warp)
                    if (LIST && colmax > give_up) {
                        gave_up = true;
                        break;
                    }
                    step(last_tag, B1, s2, s3, pC + 2);
                    if (LIST && colmax > give_up) {
                        gave_up = true;
                        break;
                    }
                }
                if ((ud.m_pairs & 1) && !(LIST && gave_up)) {   // the odd last float4
                    float s0 = INF, s1 = INF;
                    if (SEEDED && (TAILP || lane == 0)) {
                        const uint2 sd = *reinterpret_cast<const uint2*>(pC);
                        s0 = __uint_as_float(sd.x), s1 = __uint_as_float(sd.y);
                    }
                    step(last_tag, *pB, s0, s1, pC);
                    if (LIST && colmax > give_up) gave_up = true;
                }
            };
            using T_ = cuda::std::true_type;
            using F_ = cuda::std::false_type;
            if (!MULTI) {
                if (TAILP && !MMRS_EXP_NOSEED) walk(T_{}, T_{});
                else walk(T_{}, F_{});
            } else if (ud.n_chunks == 1) {
                walk(T_{}, F_{});
            } else if (ch == 0) {
                walk(F_{}, F_{});
            } else if (ch < ud.n_chunks - 1) {
                walk(F_{}, T_{});
            } else {
                walk(T_{}, T_{});
            }
            if (LIST && gave_up) break;  // the row minima are incomplete: only the column bound counts
            if constexpr (MEAN) {   // row[k] is test point ch 32 TA + 32 k + lane; from n - n_tail on, padding
                const int i0 = ch * 32 * TA + lane, n_main = ud.n - ud.n_tail;
#pragma unroll
                for (int k = 0; k < TA; ++k)
                    if (i0 + 32 * k < n_main) rsum += (double)sqrtf(row[k]);
                continue;
            }
            if (XF) {   // row minima of r -> squared distances: + |a|^2 (the odd scalar slot is already a distance)
#pragma unroll
                for (int k = 0; k < H; ++k) {
                    float n0, n1;
                    upk(NA[k], n0, n1);
                    row[2 * k] += n0;
                    row[2 * k + 1] += n1;
                }
            }
            float rm = XF ? fmaxf(row[0], 0.f) : row[0];
#pragma unroll
            for (int k = 1; k < TA; ++k) rm = fmaxf(rm, row[k]);
            rowmax = max(rowmax, __float_as_uint(rm));
        }
        if (MULTI) __syncwarp();  // the next candidate reuses my_col
        float d;
        if constexpr (MEAN) {
            __syncwarp();   // lane 0 stored the column minima
            double csum = 0.0;
            for (int j = lane; j < ud.m; j += 32) csum += (double)sqrtf(__uint_as_float(my_col[j]));
            __syncwarp();   // the next candidate reuses my_col
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                rsum += __shfl_xor_sync(0xffffffffu, rsum, o);
                csum += __shfl_xor_sync(0xffffffffu, csum, o);
            }
            // an FP32 overflow of d^2 makes a term, and so the cost, +inf, as it makes the full cost's maximum
            d = (float)fmax(csum / (double)ud.m, rsum / (double)ud.n);
        } else {
            const unsigned h2 = __reduce_max_sync(0xffffffffu, max(rowmax, colmax));
            d = sqrtf(__uint_as_float(h2));
        }
        if (lane == 0) {
            // A candidate that gave up holds only a proven LOWER BOUND (above the unit's window): it is stored as such
            // (mmrs_b200.h: dist32 of pruned / given-up candidates is a bound) but enters neither the error diagnostic
            // nor the unit's key.
            if (LIST && !gave_up) {
                const float old = dist32[ud.dist_off + c];
                worst = fmaxf(worst, fabsf(d * d - old * old));
            }
            dist32[ud.dist_off + c] = d;
            if (!LIST || !gave_up) {
                const unsigned long long k64 = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)c;
                best = min(best, k64);
            }
        }
    }
    if (LIST && lane == 0 && worst > 0.f) {
        const float r = fmaxf(__uint_as_float(rmax_bits[unit]), 1e-30f);
        atomicMax(diag, __float_as_uint(worst / (r * r)));
        worst = 0.f;
    }
    if (lane == 0 && best != ~0ull) atomicMin(s_key, best);
    __syncthreads();
    if (threadIdx.x == 0 && *s_key != ~0ull) atomicMin(&key[unit], *s_key);
    if (!LIST) break;
    g_pos = run_end;
    if (g_pos >= g_hi) break;
    __syncthreads();  // every warp is done with the staged unit and s_key before the next run re-stages
    }
}

// =============================================================================
// K1e (k_sweep_eb<RIGID, false>): the dense sweep with EARLY-BREAK directed passes. Same work items, staging image (one
// TMA bulk copy) and outputs (dist32, the packed (distance, index) key) as K1, but a candidate no longer costs all N M
// pair distances:
//     H^2 = max( max_a min_b d^2 , max_b min_a d^2 ),
// and once L, an exactly computed row or column minimum of THIS candidate, is known, a row that meets one b with
// d^2 <= L cannot raise the maximum and stops there. Per warp, over a contiguous run of the tile's candidates:
//   rotate  the N test points into a per-warp shared-memory row A'[N];
//   seed    L = max(exact minimum of row ra, exact minimum of column cb), where ra / cb defined the previous
//           candidate's maximum (the warp's first candidate: the points farthest from the rotation centre);
//   rows    lane l takes rows l, l + 32, ...: kEbTries positions of a zig-zag scan around the row's hint (the index
//           where it stopped for the previous candidate); rows still open are then finished one at a time by the
//           whole warp (32 positions per round, one REDUX.MIN), stopping at the first round whose minimum is <= L;
//           a row that runs to its end has an exact minimum > L, which becomes L;
//   columns the same with the reference points as rows and A' as the set.
// Every pair distance is K1's operation sequence (x' = fma(y, -s, x c), y' = fma(x, s, y c), d^2 = fma(dx, dx, dy dy)),
// pinned against contraction; the column pass reads the same A' (|a - b|^2 and |b - a|^2 round alike). L only ever
// holds exact minima of the current candidate: earlier candidates decide the ORDER of the scans, never a threshold. So
// the final L is max over every row and column minimum, and dist32 is bit-identical to K1's. An overflowed d^2 = inf
// never passes <= L: that row scans to its exact minimum, as K1 computes it.
// =============================================================================
constexpr int kEbTries = 4;   // zig-zag positions a lane tries on its own before the warp takes its row over

// per-warp shared memory of K1e: A'[n] (float2), then the row hints [n] and column hints [m] (16-bit indices)
__host__ __device__ constexpr int eb_warp_bytes(int n, int m) { return (8 * n + 2 * (n + m) + 15) & ~15; }

__device__ __forceinline__ float eb_d2(float2 a, float2 b) {
    const float dx = __fsub_rn(a.x, b.x), dy = __fsub_rn(a.y, b.y);
    return __fmaf_rn(dx, dx, __fmul_rn(dy, dy));
}
// t-th position (t < n: every index exactly once) of a scan over n points that starts at h and zig-zags outward:
// h, h + 1, h - 1, h + 2, ... modulo n (contours are closed)
__device__ __forceinline__ int eb_zig(int h, int t, int n) {
    int j = h + ((t & 1) ? (t + 1) >> 1 : -(t >> 1));
    j = j < 0 ? j + n : j;
    return j >= n ? j - n : j;
}
// Minimum of d^2(a, P[j]) over the n points of P, the whole warp together along the zig-zag from h (call it with the
// full warp, warp-uniform arguments). early: stop after the first round whose running minimum is <= L. Returns the bit
// pattern of the minimum found (the exact minimum whenever it is > L) and, in arg, where it was found.
__device__ __forceinline__ unsigned eb_warp_min(const float2* P, int n, float2 a, int h, unsigned L, bool early, int lane,
                                                int& arg, unsigned& pairs) {
    unsigned best = ~0u, m = ~0u;
    int bj = h;
    for (int t0 = 0; t0 < n; t0 += 32) {
        const int t = t0 + lane;
        if (t < n) {
            const int j = eb_zig(h, t, n);
            const unsigned d = __float_as_uint(eb_d2(a, P[j]));
            if (d < best) best = d, bj = j;
            ++pairs;
        }
        m = __reduce_min_sync(0xffffffffu, best);
        if (early && m <= L) break;
    }
    arg = __shfl_sync(0xffffffffu, bj, __ffs(__ballot_sync(0xffffffffu, best == m)) - 1);
    return m;
}
// Index of the largest v over the warp (v: non-negative float bits; ties -> lowest lane).
__device__ __forceinline__ int eb_warp_argmax(unsigned v, int idx) {
    const unsigned m = __reduce_max_sync(0xffffffffu, v);
    return __shfl_sync(0xffffffffu, idx, __ffs(__ballot_sync(0xffffffffu, v == m)) - 1);
}

// Rows g .. g + 31 of one direction of the early-break passes (call it with the full warp): rows R[i] against the n_set
// points of P, with the rows' hints h; open: row g + lane takes part. Lane l first tries kEbTries positions of the
// zig-zag around the hint of row g + l; the rows still open are then finished one at a time by the whole warp. A row
// stops at its first d^2 <= L and keeps that position as its hint; a row that scans to its end has an exact minimum
// mn > L, and L becomes exact(mn, i).
template <class Exact>
__device__ __forceinline__ void eb_rows(const float2* R, int g, bool open, const float2* P, int n_set, unsigned short* h,
                                        unsigned& L, Exact exact, int lane, unsigned& pairs) {
    if (open) {
        const int i = g + lane;
        const float2 a = R[i];
        const int h0 = h[i];
        for (int t = 0; t < kEbTries && t < n_set; ++t) {
            const int j = eb_zig(h0, t, n_set);
            ++pairs;
            if (__float_as_uint(eb_d2(a, P[j])) <= L) {
                h[i] = (unsigned short)j;
                open = false;
                break;
            }
        }
    }
    for (unsigned open_mask = __ballot_sync(0xffffffffu, open); open_mask; open_mask &= open_mask - 1) {
        const int ii = g + __ffs(open_mask) - 1;
        int arg;
        const unsigned mn = eb_warp_min(P, n_set, R[ii], h[ii], L, true, lane, arg, pairs);
        __syncwarp();
        if (lane == 0) h[ii] = (unsigned short)arg;
        if (mn > L) L = exact(mn, ii);
    }
}

// =============================================================================
// K1e-partial (k_sweep_eb<RIGID, true>): the early-break sweep for the PARTIAL cost (include/mmrs_b200.h "partial
// cost"). In each direction the directed value is the (q + 1)-th largest row minimum instead of the largest, so the q
// worst points of each set do not count. Same work items, staging image and outputs as K1e; per warp, over its
// contiguous run:
//   lists   per direction the q + 1 largest EXACT minima found so far (float bits + point index) in per-warp shared
//           memory; kth = the smallest of them when the list is full, else 0; L = max(kth_rows, kth_cols);
//   seed    the rows of the previous candidate's list in the direction that defined its value (the run's first
//           candidate: the q + 1 points farthest from the centre, both directions), each scanned to its end by one
//           lane; they enter the list and are marked so that the main pass skips them;
//   rows    K1e's pass (eb_rows) with the seeded rows left out: a row that scans to its end has an exact minimum > L
//           and enters its list (replacing the smallest entry when full); L is recomputed;
//   columns the same with the reference points as rows.
// Exactness (F = max(V_r, V_c), V the true (q + 1)-th largest FP32 minimum of a direction): L is always the (q + 1)-th
// largest of a subset of exact minima, so L <= F; a row that was not collected has a minimum <= L at that time <=
// L_final; if V_r > L_final, all q + 1 rows of the true top q + 1 were collected and the list's kth is V_r; otherwise
// kth_r <= V_r <= L_final. Hence L_final = F, bit for bit, and with q = 0 this is K1e. early = 0 (MMRS_EARLY_BREAK=0):
// no row stops early (every row is scanned to its end by one lane), the bit-for-bit test partner.
// =============================================================================
constexpr int kPartialMaxQ = 255;   // points per direction and unit that may be left out (the list holds q + 1 <= 256)

// per-warp shared memory of K1e-partial: K1e's block (A', row / column hints), then for rows and for columns the list
// (q + 1 float bits, q + 1 indices) and a bit set of the seeded points
__host__ __device__ constexpr int ebp_warp_bytes(int n, int m, int q_r, int q_c) {
    return (eb_warp_bytes(n, m) + 8 * (q_r + 1) + 8 * (q_c + 1) + 4 * ((n + 31) / 32 + (m + 31) / 32) + 15) & ~15;
}

// The q + 1 largest exact minima of one direction found so far. cnt, kth and at are warp-uniform.
struct EbList {
    unsigned* val;
    int* idx;
    int cap, cnt;
    unsigned kth;   // smallest entry when the list is full, else 0
    int at;         // its slot
};
__device__ __forceinline__ void ebl_refresh(EbList& l, int lane) {
    __syncwarp();
    if (l.cnt < l.cap) {
        l.kth = 0u;
        return;
    }
    unsigned mn = ~0u;
    int at = 0;
    for (int k = lane; k < l.cap; k += 32)
        if (l.val[k] < mn) mn = l.val[k], at = k;
    const unsigned m = __reduce_min_sync(0xffffffffu, mn);
    l.at = __shfl_sync(0xffffffffu, at, __ffs(__ballot_sync(0xffffffffu, mn == m)) - 1);
    l.kth = m;
}
// v: an exact minimum > kth (warp-uniform arguments)
__device__ __forceinline__ void ebl_insert(EbList& l, unsigned v, int i, int lane) {
    const int k = l.cnt < l.cap ? l.cnt++ : l.at;
    if (lane == 0) l.val[k] = v, l.idx[k] = i;
    ebl_refresh(l, lane);
}
// Exact minimum of d^2(a, P[j]) over the n points of P by ONE lane, in index order (the warp's lanes read the same P[j]:
// a broadcast); arg = where it was first found.
__device__ __forceinline__ unsigned eb_lane_min(const float2* P, int n, float2 a, int& arg, unsigned& pairs) {
    unsigned best = ~0u;
    int bj = 0;
    for (int j = 0; j < n; ++j) {
        const unsigned d = __float_as_uint(eb_d2(a, P[j]));
        if (d < best) best = d, bj = j;
    }
    pairs += (unsigned)n;
    arg = bj;
    return best;
}

// RIGID = true: rigid candidates, c = i n_trans + j (see k_sweep): A'[k] = R a_k + t, the translation added once with
// __fadd_rn when the row is materialised; the column pass reads the same A', so K1e stays bit-identical to K1.
// PARTIAL = false: K1e, kWarpsPerCta warps per CTA; early is not read.
// PARTIAL = true: K1e-partial, blockDim.x / 32 warps per CTA (the host picks 8, 4, 2 or 1 per size class).
template <bool RIGID, bool PARTIAL>
__global__ void __launch_bounds__(kThreads, PARTIAL ? 2 : 3)
    k_sweep_eb(const UnitDesc* __restrict__ units, const WorkItem* __restrict__ work, const float4* __restrict__ lay,
               const float2* __restrict__ cs32, float* __restrict__ dist32, unsigned long long* __restrict__ key,
               unsigned long long* __restrict__ pairs_out, const float2* __restrict__ t32, int early) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
    unsigned long long* s_key = reinterpret_cast<unsigned long long*>(smem_raw + 8);
    float4* sA = reinterpret_cast<float4*>(smem_raw + 16);
    const WorkItem w = work[blockIdx.x];
    const UnitDesc ud = units[w.unit];
    const int n_warps = PARTIAL ? blockDim.x >> 5 : kWarpsPerCta;
    const int lane = threadIdx.x & 31, wid = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int TA = ud.ta, S = (TA + 1) / 2, N = ud.n, M = ud.m, n_main = N - ud.n_tail;
    const StageLayout sl = stage_layout(TA, ud.n_chunks, ud.n_tail, ud.m_pairs);
    const float2* sB = reinterpret_cast<const float2*>(sA + sl.a);                        // reference point j
    const float2* sT = reinterpret_cast<const float2*>(sA + sl.a + sl.b + sl.nb);         // tail point t
    unsigned char* my = reinterpret_cast<unsigned char*>(sA + sl.a + sl.b + sl.nb + sl.t) +
                        wid * (PARTIAL ? ebp_warp_bytes(N, M, ud.q_bwd, ud.q_fwd) : eb_warp_bytes(N, M));
    float2* sR = reinterpret_cast<float2*>(my);                                           // A': rotated test points
    // direction 0, rows: A' against the reference points; direction 1, columns: the reference points against A'
    const float2* pts[2] = {sR, sB};
    const int n_rows[2] = {N, M};
    unsigned short* hint[2];
    hint[0] = reinterpret_cast<unsigned short*>(sR + N);
    hint[1] = hint[0] + N;
    EbList lst[2];       // PARTIAL: the lists of the two directions
    unsigned* bits[2];   // PARTIAL: the seeded rows of the two directions
    if constexpr (PARTIAL) {
        unsigned* lp = reinterpret_cast<unsigned*>(my + eb_warp_bytes(N, M));
        lst[0].cap = ud.q_bwd + 1, lst[1].cap = ud.q_fwd + 1;
        lst[0].val = lp;
        lst[0].idx = reinterpret_cast<int*>(lp + lst[0].cap);
        lst[1].val = lp + 2 * lst[0].cap;
        lst[1].idx = reinterpret_cast<int*>(lst[1].val + lst[1].cap);
        bits[0] = lp + 2 * (lst[0].cap + lst[1].cap);
        bits[1] = bits[0] + (N + 31) / 32;
    }
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        *s_key = ~0ull;
        const uint32_t bytes = (uint32_t)sl.total() * 16u;
        mbar_expect_tx(bar, bytes);
        tma_bulk_g2s(sA, lay + ud.lay_off, bytes, bar);
    }
    __syncthreads();
    mbar_wait(bar, 0);

    // test point i of the staging image (K0's layout: register slots, then the exact-tiling tail block)
    auto test_pt = [&](int i) -> float2 {
        if (i >= n_main) return sT[i - n_main];
        const int c = i / (32 * TA), r = i - c * 32 * TA;
        const float4 v = sA[(c * S + (r >> 6)) * 32 + (r & 31)];
        return (r & 32) ? make_float2(v.y, v.w) : make_float2(v.x, v.z);
    };
    // this warp's contiguous run of candidates: neighbouring angles keep the hints valid
    const int per = (w.count + n_warps - 1) / n_warps;
    const int c_begin = w.begin + min(w.count, wid * per), c_end = w.begin + min(w.count, (wid + 1) * per);
    unsigned long long best = ~0ull;
    unsigned pairs = 0;
    if (c_begin < c_end) {
        int ra = 0, cb = 0;            // K1e: the row and the column that defined the previous candidate's value
        bool seed[2] = {true, true};   // PARTIAL: the directions whose lists seed the next candidate
        if constexpr (PARTIAL) {
#pragma unroll
            for (int dir = 0; dir < 2; ++dir) {
                const int n = n_rows[dir];
                for (int k = lane; k < (n + 31) / 32; k += 32) bits[dir][k] = 0u;
                for (int r = lane; r < n; r += 32)
                    hint[dir][r] = (unsigned short)(((long long)r * n_rows[1 - dir]) / n);
                __syncwarp();
                // first candidate's seeds: the q + 1 points farthest from the rotation centre (unrotated)
                EbList& l = lst[dir];
                for (int k = 0; k < l.cap; ++k) {
                    unsigned far = 0u;
                    int at = 0;
                    for (int r = lane; r < n; r += 32) {
                        if ((bits[dir][r >> 5] >> (r & 31)) & 1u) continue;
                        const float2 p = dir ? sB[r] : test_pt(r);
                        const unsigned r2 = __float_as_uint(p.x * p.x + p.y * p.y) + 1u;   // > 0: not yet taken
                        if (r2 > far) far = r2, at = r;
                    }
                    const int r = eb_warp_argmax(far, at);
                    if (lane == 0) {
                        l.idx[k] = r;
                        bits[dir][r >> 5] |= 1u << (r & 31);
                    }
                    __syncwarp();
                }
                l.cnt = l.cap;
            }
        } else {
            // first candidate: hints on the index diagonal, seeds at the points farthest from the rotation centre
            unsigned far_a = 0u, far_b = 0u;
            int ia = 0, ib = 0;
            for (int i = lane; i < N; i += 32) {
                const float2 p = test_pt(i);
                const unsigned r2 = __float_as_uint(p.x * p.x + p.y * p.y);
                if (r2 > far_a) far_a = r2, ia = i;
                hint[0][i] = (unsigned short)(((long long)i * M) / N);
            }
            for (int j = lane; j < M; j += 32) {
                const float2 p = sB[j];
                const unsigned r2 = __float_as_uint(p.x * p.x + p.y * p.y);
                if (r2 > far_b) far_b = r2, ib = j;
                hint[1][j] = (unsigned short)(((long long)j * N) / M);
            }
            ra = eb_warp_argmax(far_a, ia), cb = eb_warp_argmax(far_b, ib);
        }
        for (int c = c_begin; c < c_end; ++c) {
            float2 tr = make_float2(0.f, 0.f);
            int ia = c;
            if (RIGID) {
                ia = c / ud.n_trans;
                tr = __ldg(&t32[ud.t_off + (c - ia * ud.n_trans)]);
            }
            const float2 cs = __ldg(&cs32[ud.cand_off + ia]);
            __syncwarp();   // the previous candidate is done with A', the hints and the lists
            for (int i = lane; i < N; i += 32) {
                const float2 p = test_pt(i);
                float2 r = make_float2(__fmaf_rn(p.y, -cs.y, __fmul_rn(p.x, cs.x)), __fmaf_rn(p.x, cs.y, __fmul_rn(p.y, cs.x)));
                if (RIGID) r = make_float2(__fadd_rn(r.x, tr.x), __fadd_rn(r.y, tr.y));
                sR[i] = r;
            }
            __syncwarp();
            unsigned L;
            if constexpr (PARTIAL) {
                // seeds: the listed rows of the seeded directions, one lane each, scanned to the end
#pragma unroll
                for (int dir = 0; dir < 2; ++dir) {
                    EbList& l = lst[dir];
                    if (!seed[dir]) {
                        l.cnt = 0;
                        l.kth = 0u;
                        continue;
                    }
                    for (int k = lane; k < l.cnt; k += 32) {
                        const int r = l.idx[k];
                        int arg;
                        l.val[k] = eb_lane_min(pts[1 - dir], n_rows[1 - dir], pts[dir][r], arg, pairs);
                        hint[dir][r] = (unsigned short)arg;
                        atomicOr(&bits[dir][r >> 5], 1u << (r & 31));
                    }
                    ebl_refresh(l, lane);
                }
                L = max(lst[0].kth, lst[1].kth);
#pragma unroll
                for (int dir = 0; dir < 2; ++dir) {
                    const float2* R = pts[dir];
                    const float2* P = pts[1 - dir];
                    const int n = n_rows[dir], n_set = n_rows[1 - dir];
                    unsigned short* h = hint[dir];
                    const unsigned* seeded = bits[dir];
                    for (int g = 0; g < n; g += 32) {
                        const int i = g + lane;
                        const bool open = i < n && !((seeded[i >> 5] >> (i & 31)) & 1u);
                        if (early) {
                            eb_rows(R, g, open, P, n_set, h, L,
                                    [&](unsigned mn, int r) {
                                        ebl_insert(lst[dir], mn, r, lane);
                                        return max(lst[0].kth, lst[1].kth);
                                    },
                                    lane, pairs);
                            continue;
                        }
                        // every open row scanned to its end by its lane; the exact minima > L enter the list in lane order
                        unsigned mn = ~0u;
                        if (open) {
                            int arg;
                            mn = eb_lane_min(P, n_set, R[i], arg, pairs);
                            h[i] = (unsigned short)arg;
                        }
                        for (unsigned m = __ballot_sync(0xffffffffu, open); m; m &= m - 1) {
                            const int src = __ffs(m) - 1;
                            const unsigned v = __shfl_sync(0xffffffffu, mn, src);
                            if (v > L) {
                                ebl_insert(lst[dir], v, g + src, lane);
                                L = max(lst[0].kth, lst[1].kth);
                            }
                        }
                    }
                }
            } else {
                // seeds: the exact minima of the row and the column that defined the previous candidate's value
                int arg;
                L = eb_warp_min(sB, M, sR[ra], hint[0][ra], 0u, false, lane, arg, pairs);
                const int h_ra = arg;
                const unsigned lc = eb_warp_min(sR, N, sB[cb], hint[1][cb], 0u, false, lane, arg, pairs);
                __syncwarp();
                if (lane == 0) hint[0][ra] = (unsigned short)h_ra, hint[1][cb] = (unsigned short)arg;
                L = max(L, lc);
                __syncwarp();
                for (int g = 0; g < N; g += 32)   // rows: test point i against the reference points
                    eb_rows(sR, g, g + lane < N, sB, M, hint[0], L, [&](unsigned mn, int i) { ra = i; return mn; }, lane, pairs);
                for (int g = 0; g < M; g += 32)   // columns: reference point j against A'
                    eb_rows(sB, g, g + lane < M, sR, N, hint[1], L, [&](unsigned mn, int j) { cb = j; return mn; }, lane, pairs);
            }
            const float d = sqrtf(__uint_as_float(L));
            if (lane == 0) {
                dist32[ud.dist_off + c] = d;
                best = min(best, ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)c);
            }
            if constexpr (PARTIAL) {
                // the next candidate seeds the direction that defined this value (ties: rows) from this list
                seed[0] = lst[0].kth >= lst[1].kth;
                seed[1] = !seed[0];
                __syncwarp();
#pragma unroll
                for (int dir = 0; dir < 2; ++dir)
                    for (int k = lane; k < (n_rows[dir] + 31) / 32; k += 32) bits[dir][k] = 0u;
            }
        }
    }
    const unsigned warp_pairs = __reduce_add_sync(0xffffffffu, pairs);
    if (lane == 0 && pairs_out && warp_pairs) atomicAdd(pairs_out, (unsigned long long)warp_pairs);
    if (lane == 0 && best != ~0ull) atomicMin(s_key, best);
    __syncthreads();
    if (threadIdx.x == 0 && *s_key != ~0ull) atomicMin(&key[w.unit], *s_key);
}

// =============================================================================
// K1b: the FP32 sweep for units that do not fit K1's shared-memory staging (more than ~4 000 points per set; the
// reference has no size limit, process_utils.rs:84-121). Same arithmetic as K1's chunked flavour (one warp = one
// candidate, TA = 16 test points per lane and chunk, packed f32x2, 3-input minima, one REDUX per reference point), but
//   * the REFERENCE set is streamed through shared memory in blocks of kBigBlock points (all warps of the CTA walk the
//     blocks together, each with its own candidate); the per-warp column-minimum array only spans one block;
//   * the TEST set is read chunk by chunk from the staging image in global memory (L2) and rotated again per block;
//   * the ROW minima of a candidate persist across the blocks in a per-warp scratch row in global memory
//     ([CTA][warp][slot][lane] floats, coalesced, L2-resident: 2 x 4 B per test point and block).
// Persistent grid: CTA b walks the work items b, b + gridDim.x, ... (its scratch rows are reused).
// =============================================================================
constexpr int kBigBlock = 1024;   // reference points per shared-memory block
constexpr int kBigTA = 16;

// RIGID = true: rigid candidates, c = i n_trans + j (see k_sweep).
template <bool RIGID = false>
__global__ void __launch_bounds__(kThreads, 2)
    k_sweep_big(const UnitDesc* __restrict__ units, const WorkItem* __restrict__ work, int n_work,
                const float4* __restrict__ lay, const float2* __restrict__ cs32, float* __restrict__ dist32,
                unsigned long long* __restrict__ key, float* __restrict__ row_scratch, long long scratch_per_warp,
                const float2* __restrict__ t32) {
    constexpr int TA = kBigTA, H = TA / 2;
    __shared__ __align__(16) float4 sB[kBigBlock / 2];
    __shared__ unsigned s_col[kWarpsPerCta][kBigBlock];
    const int lane = threadIdx.x & 31, wid = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // warp-uniform for ptxas
    const float INF = __int_as_float(0x7f800000);
    float* my_rows = row_scratch + ((long long)blockIdx.x * kWarpsPerCta + wid) * scratch_per_warp;
    unsigned* my_col = s_col[wid];
    for (int wi = blockIdx.x; wi < n_work; wi += gridDim.x) {
        const WorkItem w = work[wi];
        const UnitDesc ud = units[w.unit];
        const float4* gA = lay + ud.lay_off;
        const float4* gB = gA + (long long)ud.n_chunks * H * 32;
        const int n_blocks = (ud.m_pairs + kBigBlock / 2 - 1) / (kBigBlock / 2);
        for (int c0 = 0; c0 < w.count; c0 += kWarpsPerCta) {   // one candidate per warp and round; every warp walks the blocks
            const bool live = c0 + wid < w.count;
            const int c = w.begin + min(c0 + wid, w.count - 1);
            float2 tr = make_float2(0.f, 0.f);
            int ia = c;
            if (RIGID) {
                ia = c / ud.n_trans;
                tr = __ldg(&t32[ud.t_off + (c - ia * ud.n_trans)]);
            }
            const float2 cs = __ldg(&cs32[ud.cand_off + ia]);
            const uint64_t C2 = pk(cs.x, cs.x), S2 = pk(cs.y, cs.y), NS2 = pk(-cs.y, -cs.y);
            const uint64_t TX2 = pk(tr.x, tr.x), TY2 = pk(tr.y, tr.y);
            unsigned rowmax = 0u, colmax = 0u;
            for (int bb = 0; bb < n_blocks; ++bb) {
                const int j0 = bb * (kBigBlock / 2), jn = min(kBigBlock / 2, ud.m_pairs - j0);
                __syncthreads();   // every warp is done with the previous block
                for (int j = threadIdx.x; j < jn; j += kThreads) sB[j] = gB[j0 + j];
                __syncthreads();
                const bool last_block = bb == n_blocks - 1;
                for (int ch = 0; ch < ud.n_chunks; ++ch) {
                    uint64_t AX[H], AY[H];
                    float row[TA];
#pragma unroll
                    for (int k = 0; k < H; ++k) {
                        const float4 a = __ldg(&gA[(ch * H + k) * 32 + lane]);
                        const uint64_t X2 = pk(a.x, a.y), Y2 = pk(a.z, a.w);
                        AX[k] = fma2(Y2, NS2, mul2(X2, C2));
                        AY[k] = fma2(X2, S2, mul2(Y2, C2));
                        if (RIGID) {
                            AX[k] = add2(AX[k], TX2);
                            AY[k] = add2(AY[k], TY2);
                        }
                        if (bb == 0) {
                            row[2 * k] = INF;
                            row[2 * k + 1] = INF;
                        } else {   // the row minima over the previous blocks
                            const float2 r = *reinterpret_cast<const float2*>(&my_rows[((ch * H + k) * 32 + lane) * 2]);
                            row[2 * k] = r.x;
                            row[2 * k + 1] = r.y;
                        }
                    }
                    const bool last_chunk = ch == ud.n_chunks - 1;
#pragma unroll 2
                    for (int j = 0; j < jn; ++j) {
                        const float4 B = sB[j];
                        const uint64_t bx0 = pk(B.x, B.x), by0 = pk(B.y, B.y), bx1 = pk(B.z, B.z), by1 = pk(B.w, B.w);
                        float q0 = INF, q1 = INF;
                        if (ch > 0 && lane == 0) {
                            const uint2 prev = *reinterpret_cast<const uint2*>(&my_col[2 * j]);
                            q0 = __uint_as_float(prev.x);
                            q1 = __uint_as_float(prev.y);
                        }
#pragma unroll
                        for (int k = 0; k < H; ++k) {
                            const uint64_t dx0 = sub2(AX[k], bx0), dy0 = sub2(AY[k], by0);
                            const uint64_t dx1 = sub2(AX[k], bx1), dy1 = sub2(AY[k], by1);
                            const uint64_t d0 = fma2(dx0, dx0, mul2(dy0, dy0));
                            const uint64_t d1 = fma2(dx1, dx1, mul2(dy1, dy1));
                            float d00, d10, d01, d11;
                            upk(d0, d00, d10);
                            upk(d1, d01, d11);
                            row[2 * k] = min3(row[2 * k], d00, d01);
                            row[2 * k + 1] = min3(row[2 * k + 1], d10, d11);
                            q0 = min3(q0, d00, d10);
                            q1 = min3(q1, d01, d11);
                        }
                        const unsigned r0 = __reduce_min_sync(0xffffffffu, __float_as_uint(q0));
                        const unsigned r1 = __reduce_min_sync(0xffffffffu, __float_as_uint(q1));
                        if (last_chunk) colmax = max(colmax, max(r0, r1));
                        else if (lane == 0) *reinterpret_cast<uint2*>(&my_col[2 * j]) = make_uint2(r0, r1);
                    }
                    if (last_block) {
                        float rm = row[0];
#pragma unroll
                        for (int k = 1; k < TA; ++k) rm = fmaxf(rm, row[k]);
                        rowmax = max(rowmax, __float_as_uint(rm));
                    } else {
#pragma unroll
                        for (int k = 0; k < H; ++k)
                            *reinterpret_cast<float2*>(&my_rows[((ch * H + k) * 32 + lane) * 2]) = make_float2(row[2 * k], row[2 * k + 1]);
                    }
                    __syncwarp();   // the next chunk reads the column minima lane 0 just stored
                }
            }
            const unsigned h2 = __reduce_max_sync(0xffffffffu, max(rowmax, colmax));
            const float d = sqrtf(__uint_as_float(h2));
            if (lane == 0 && live) {
                dist32[ud.dist_off + c] = d;
                atomicMin(&key[w.unit], ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)c);
            }
        }
    }
}

// =============================================================================
// K1p: exact lower-bound pruning tier (opt-in, mmrs_sweep_opts.prune). For ANY subsets A' of the test points and B'
// of the reference points,
//     H(A, B) = max( max_{a in A} min_{b in B} |a - b| , max_{b in B} min_{a in A} |a - b| )
//            >= max( max_{a in A'} min_{b in B} |a - b| , max_{b in B'} min_{a in A} |a - b| ) =: LB,
// because a maximum over fewer rows can only be smaller while every row minimum still runs over ALL points of the
// other set. LB costs (|A'| M + |B'| N) pair distances instead of N M. A candidate whose LB exceeds the exact distance
// of any evaluated candidate (plus the FP32 window) cannot be the arg-min and is never scored; every other candidate is
// scored by the exact FP32 kernel (k_sweep LIST) and continues to K2/K3/K4 unchanged, so the selected candidate, its
// angle and its f64 distance are identical to the dense path's.
//   k_prep_lb   per unit two staging images: rows = R sampled test points / columns = all reference points, and
//               rows = R sampled reference points / columns = all test points (rotated by -theta instead). The sample
//               is, per window of n/R consecutive points, the point farthest from the rotation centre: the directed
//               maxima sit where a contour sticks out (measured: 4x fewer survivors than plain striding).
//   k_lb<RS,CB> rows-only sweep of those images, 32 RS rows x CB candidates per warp: row minima + max, no column minima,
//               no REDUX per column; result max-combined into dist32 with atomicMax on the (non-negative) float bits.
//               32 rows for sets below 1 024 points, 128 rows above (dense 2 000-point lumina of consecutive frames
//               differ so little that a coarser sample lets half of the candidates through).
//   k_lb_argmin the candidate with the smallest LB of each unit (scored first: its exact distance is the bound).
// =============================================================================
constexpr int kLbNegSin = 0x100;  // UnitDesc.flags of a lower-bound unit: rotate its rows by -theta

__global__ void k_prep_lb(const UnitDesc* __restrict__ units, const UnitDesc* __restrict__ lb_units, int n_units,
                          const double* __restrict__ test_xy, const double* __restrict__ ref_xy,
                          float4* __restrict__ lay, int R, int R_eff, int pick_mode) {
    const int u = blockIdx.x;
    const UnitDesc ud = units[u];
    if (ud.n <= 0 || ud.m <= 0) return;
    for (int pass = 0; pass < 2; ++pass) {
        const UnitDesc lb = lb_units[u + pass * n_units];
        const double* rows = pass == 0 ? test_xy + 2 * ud.test_off : ref_xy + 2 * ud.ref_off;
        const double* cols = pass == 0 ? ref_xy + 2 * ud.ref_off : test_xy + 2 * ud.test_off;
        const int nr = pass == 0 ? ud.n : ud.m, nc = pass == 0 ? ud.m : ud.n;
        float2* A = reinterpret_cast<float2*>(lay + lb.lay_off);   // R rows (x, y); lane l of k_lb owns row l
        float4* B = lay + lb.lay_off + R / 2;
        // R_eff < R (experiments): only R_eff distinct rows, repeated, to measure how the bound degrades
        auto pick = [&](int r) { return nr <= R ? min(r, nr - 1) : (int)(((long long)(r % R_eff) * nr) / R_eff); };
        for (int r = threadIdx.x; r < R; r += blockDim.x) {
            int i = pick(r);
            if (pick_mode == 3 && nr > R) {
                // half strided, half farthest: windows of 2 nr / R points; even rows take the window's first point,
                // odd rows its point farthest from the rotation centre
                const int w = r >> 1, W = R >> 1;
                const int lo = (int)(((long long)w * nr) / W), hi = (int)(((long long)(w + 1) * nr) / W);
                i = lo;
                if (r & 1) {
                    double best = -1.0;
                    for (int k = lo; k < hi; ++k) {
                        const double dx = rows[2 * k] - ud.cx, dy = rows[2 * k + 1] - ud.cy, rr = dx * dx + dy * dy;
                        if (rr > best) best = rr, i = k;
                    }
                }
            } else if (pick_mode != 0 && nr > R) {
                // Any subset gives a valid bound; the directed maxima sit where a contour sticks out or caves in, so
                // take, per index window, the point farthest from (even windows / mode 2: all) or nearest to (odd
                // windows) the rotation centre instead of the window's first point.
                const int lo = (int)(((long long)r * nr) / R), hi = (int)(((long long)(r + 1) * nr) / R);
                const bool want_max = pick_mode == 2 || (r & 1) == 0;
                double best = want_max ? -1.0 : 1e300;
                for (int k = lo; k < hi; ++k) {
                    const double dx = rows[2 * k] - ud.cx, dy = rows[2 * k + 1] - ud.cy, rr = dx * dx + dy * dy;
                    if (want_max ? rr > best : rr < best) best = rr, i = k;
                }
            }
            A[r] = make_float2((float)(rows[2 * i] - ud.cx), (float)(rows[2 * i + 1] - ud.cy));
        }
        for (int j = threadIdx.x; j < lb.m_pairs; j += blockDim.x) {
            const int j0 = min(2 * j, nc - 1), j1 = min(2 * j + 1, nc - 1);
            B[j] = make_float4((float)(cols[2 * j0] - ud.cx), (float)(cols[2 * j0 + 1] - ud.cy), (float)(cols[2 * j1] - ud.cx),
                               (float)(cols[2 * j1 + 1] - ud.cy));
        }
    }
}

// One warp = CB consecutive candidates x 32 RS sampled rows (lane l owns rows l, l + 32, ...): the packed f32x2 lanes
// carry TWO CANDIDATES of the same row, so one broadcast LDS.128 of two column points feeds RS CB/2 = 4 blocks of
// 8 packed FP32 + 2 FMNMX3 — the instruction mix of K1's inner loop without its column side.
template <int RS, int CB>
__global__ void __launch_bounds__(kThreads, 2)
    k_lb(const UnitDesc* __restrict__ lb_units, const WorkItem* __restrict__ work, const float4* __restrict__ lay,
         const float2* __restrict__ cs32, float* __restrict__ dist32) {
    constexpr int P = CB / 2;
    static_assert(RS * CB == 8 && CB >= 2, "rows per lane x candidates per warp");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
    float4* sA = reinterpret_cast<float4*>(smem_raw + 16);
    const WorkItem w = work[blockIdx.x];
    const UnitDesc ud = lb_units[w.unit];
    const int a_elems = 16 * RS, b_elems = ud.m_pairs;   // 32 RS rows x 8 B
    float4* sB = sA + a_elems;
    const int lane = threadIdx.x & 31, wid = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // warp-uniform for ptxas
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        const uint32_t bytes = (uint32_t)(a_elems + b_elems) * 16u;
        mbar_expect_tx(bar, bytes);
        tma_bulk_g2s(sA, lay + ud.lay_off, bytes, bar);
    }
    __syncthreads();
    mbar_wait(bar, 0);
    const float INF = __int_as_float(0x7f800000);
    const float sgn = (ud.flags & kLbNegSin) ? -1.f : 1.f;
    unsigned* out = reinterpret_cast<unsigned*>(dist32 + ud.dist_off);
    uint64_t X2[RS], Y2[RS];
#pragma unroll
    for (int r = 0; r < RS; ++r) {
        const float2 a = reinterpret_cast<const float2*>(sA)[lane + 32 * r];
        X2[r] = pk(a.x, a.x);
        Y2[r] = pk(a.y, a.y);
    }
    for (int g = wid * CB; g < w.count; g += kWarpsPerCta * CB) {
        uint64_t AX[RS][P], AY[RS][P];
        float row[RS][CB];
#pragma unroll
        for (int p = 0; p < P; ++p) {
            const int c0 = w.begin + min(g + 2 * p, w.count - 1), c1 = w.begin + min(g + 2 * p + 1, w.count - 1);
            const float2 s0 = __ldg(&cs32[ud.cand_off + c0]), s1 = __ldg(&cs32[ud.cand_off + c1]);
            const uint64_t C2 = pk(s0.x, s1.x), S2 = pk(s0.y * sgn, s1.y * sgn), NS2 = pk(-s0.y * sgn, -s1.y * sgn);
#pragma unroll
            for (int r = 0; r < RS; ++r) {
                AX[r][p] = fma2(Y2[r], NS2, mul2(X2[r], C2));   // (x cos0 - y sin0, x cos1 - y sin1)
                AY[r][p] = fma2(X2[r], S2, mul2(Y2[r], C2));
                row[r][2 * p] = INF;
                row[r][2 * p + 1] = INF;
            }
        }
#pragma unroll 2
        for (int j = 0; j < ud.m_pairs; ++j) {
            const float4 B = sB[j];
            const uint64_t bx0 = pk(B.x, B.x), by0 = pk(B.y, B.y), bx1 = pk(B.z, B.z), by1 = pk(B.w, B.w);
#pragma unroll
            for (int r = 0; r < RS; ++r) {
#pragma unroll
                for (int p = 0; p < P; ++p) {
                    const uint64_t dx0 = sub2(AX[r][p], bx0), dy0 = sub2(AY[r][p], by0);
                    const uint64_t dx1 = sub2(AX[r][p], bx1), dy1 = sub2(AY[r][p], by1);
                    const uint64_t d0 = fma2(dx0, dx0, mul2(dy0, dy0));  // column point 0: (candidate 2p, candidate 2p+1)
                    const uint64_t d1 = fma2(dx1, dx1, mul2(dy1, dy1));  // column point 1
                    float d00, d01, d10, d11;
                    upk(d0, d00, d01);
                    upk(d1, d10, d11);
                    row[r][2 * p] = min3(row[r][2 * p], d00, d10);
                    row[r][2 * p + 1] = min3(row[r][2 * p + 1], d01, d11);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < CB; ++k) {
            float rm = row[0][k];
#pragma unroll
            for (int r = 1; r < RS; ++r) rm = fmaxf(rm, row[r][k]);
            const unsigned h2 = __reduce_max_sync(0xffffffffu, __float_as_uint(rm));
            if (lane == k && g + k < w.count) atomicMax(&out[w.begin + g + k], __float_as_uint(sqrtf(__uint_as_float(h2))));
        }
    }
}

// One CTA per unit: the candidate with the smallest lower bound (ties -> lowest index) becomes the unit's one-item list.
__global__ void k_lb_argmin(const UnitDesc* __restrict__ units, const float* __restrict__ dist32, int* __restrict__ l_count,
                            unsigned* __restrict__ l_base, int2* __restrict__ l_items) {
    __shared__ unsigned long long s_best;
    const int u = blockIdx.x;
    const UnitDesc ud = units[u];
    if (threadIdx.x == 0) s_best = ~0ull;
    __syncthreads();
    if (ud.flags || ud.n_cand <= 0) {
        if (threadIdx.x == 0) l_count[u] = 0, l_base[u] = (unsigned)u, l_items[u] = make_int2(-1, 0);
        return;
    }
    unsigned long long best = ~0ull;
    const float* d = dist32 + ud.dist_off;
    for (int c = threadIdx.x; c < ud.n_cand; c += blockDim.x) {
        const unsigned long long k = ((unsigned long long)__float_as_uint(d[c]) << 32) | (unsigned)c;
        best = best < k ? best : k;
    }
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
        best = best < other ? best : other;
    }
    if ((threadIdx.x & 31) == 0) atomicMin(&s_best, best);
    __syncthreads();
    if (threadIdx.x == 0) {
        l_items[u] = make_int2(u, (int)(s_best & 0xffffffffu));
        l_base[u] = (unsigned)u;
        l_count[u] = 1;
    }
}

// =============================================================================
// K2: shortlist = candidates whose FP32 distance lies inside the FP32 error window above the
// minimum. Two scans of the unit's FP32 row (L2-resident): count, reserve a contiguous range of
// the global item pool with one atomicAdd, then write (unit, candidate) items. A unit may take
// any number of items; only when the POOL is exhausted is it flagged for the dense f64 path.
// =============================================================================
// mode 0: the FP32 window  d <= dmin (1 + rel) + abs_scale Rmax  (tier 2 -> f64 recheck).
// mode 1: the tensor-core prefilter's window in SQUARED distance  d^2 <= dmin^2 + abs_scale Rmax^2  (tier 1 -> exact
//         FP32 re-scoring); `key` is then the prefilter's own minimum.
// prev_count (mode 0, optional): a unit whose tier-1 list overflowed its pool (< 0) was never re-scored in FP32; it is
// passed on as an overflow so the host rechecks all of its candidates in f64.
__global__ void k_shortlist(const UnitDesc* __restrict__ units, const float* __restrict__ dist32,
                            const unsigned long long* __restrict__ key, const unsigned* __restrict__ rmax_bits,
                            float rel, float abs_scale, unsigned pool_cap, int* __restrict__ sl_count,
                            unsigned* __restrict__ sl_base, int2* __restrict__ items, unsigned* __restrict__ n_items,
                            int mode, const int* __restrict__ prev_count) {
    __shared__ int s_n, s_pos;
    __shared__ unsigned s_base;
    const int u = blockIdx.x;
    const UnitDesc ud = units[u];
    if (ud.n_cand <= 0 || ud.n <= 0 || ud.m <= 0 || ud.c_hi <= ud.c_lo) {   // nothing of this unit is swept here
        if (threadIdx.x == 0) {
            sl_count[u] = 0;
            sl_base[u] = 0;
        }
        return;
    }
    if (prev_count && prev_count[u] < 0) {
        if (threadIdx.x == 0) {
            sl_count[u] = -ud.n_cand;
            sl_base[u] = 0;
        }
        return;
    }
    if (threadIdx.x == 0) s_n = 0, s_pos = 0;
    __syncthreads();
    const float dmin = __uint_as_float((unsigned)(key[u] >> 32));
    const float rmax = __uint_as_float(rmax_bits[u]);
    // mode 2 (expanded-form tier): the window of the tier's own absolute error on d^2 (abs_scale Rmax^2), widened by the
    // whole FP32 window of the stage behind it (4e-6 relative + 4e-6 Rmax: twice what k_shortlist mode 0 uses), so that
    // every candidate the exact FP32 values would shortlist is among the re-scored ones whatever the distance is.
    const float thr = mode == 2   ? sqrtf(fmaf(dmin, dmin, abs_scale * rmax * rmax)) * (1.0f + rel) + 4e-6f * rmax
                      : mode == 1 ? sqrtf(fmaf(dmin, dmin, abs_scale * rmax * rmax)) * (1.0f + rel)
                                  : dmin * (1.0f + rel) + abs_scale * rmax;
    const float* d = dist32 + ud.dist_off;
    int mine = 0;
    for (int c = ud.c_lo + threadIdx.x; c < ud.c_hi; c += blockDim.x) mine += (d[c] <= thr) ? 1 : 0;
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&s_n, mine);
    __syncthreads();
    const int n = s_n;
    if (threadIdx.x == 0) s_base = atomicAdd(n_items, (unsigned)n);
    __syncthreads();
    const unsigned base = s_base;
    const bool fits = (unsigned long long)base + (unsigned)n <= pool_cap;
    if (threadIdx.x == 0) {
        sl_base[u] = base;
        sl_count[u] = fits ? n : -n;  // negative: pool exhausted, the host rechecks the whole unit in f64
    }
    if (!fits) {  // neutralise the part of the reservation that lies inside the pool
        for (unsigned k = base + threadIdx.x; k < pool_cap && k < base + (unsigned)n; k += blockDim.x)
            items[k] = make_int2(-1, 0);
        return;
    }
    for (int c = ud.c_lo + threadIdx.x; c < ud.c_hi; c += blockDim.x)
        if (d[c] <= thr) items[base + atomicAdd(&s_pos, 1)] = make_int2(u, c);
}

// =============================================================================
// K3: the reference's f64 arithmetic, literally (no FMA contraction: explicit
// __dmul_rn/__dadd_rn/__dsub_rn; IEEE sqrt). cos/sin come from the HOST's glibc
// (what Rust's f64::sin/cos call), passed as a table, because CUDA's double
// sin/cos are not bit-identical to glibc's.
//   rotate     : contour_point.rs:38-52 (mode 0, identity iff angle == 0.0) /
//                align_between.rs:193-209 (mode 1)
//   translate  : rigid candidates only: x' = rx + tx, y' = ry + ty (__dadd_rn; + 0.0 is exact, so a zero translation
//                is the rotation-only cost bit for bit)
//   distances  : process_utils.rs:84-121, both directions, sqrt, max
//                (partial cost: the (q + 1)-th largest row minimum of each direction instead of the largest; mean
//                cost: the mean row value sqrt(minimum) of each direction)
// One CTA per (unit, candidate) item; grid-stride over the item list.
// t64 != NULL: rigid candidates, c = i n_trans + j -> angle i of the unit's grid, translation j of its translation grid.
// =============================================================================
__device__ __forceinline__ double block_max(double v, double* s_red) {
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = s_red[0];
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) r = fmax(r, s_red[i]);
    __syncthreads();
    return r;
}

// (q + 1)-th largest of the n non-negative values v (duplicates counted), by the whole CTA: the v_i with
// #{v_j > v_i} <= q < #{v_j >= v_i}. Every i that satisfies this holds the same value, so the result does not depend
// on the order of the threads.
__device__ __forceinline__ double block_kth_largest(const double* v, int n, int q, double* s_red) {
    double sel = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double x = v[i];
        int gt = 0, ge = 0;
        for (int j = 0; j < n && gt <= q; ++j) {
            const double y = v[j];
            gt += y > x ? 1 : 0;
            ge += y >= x ? 1 : 0;
        }
        if (gt <= q && q < ge) sel = x;
    }
    return block_max(sel, s_red);
}

// Stages the transformed test set in s_rot and, with copy_ref, the reference set in s_ref_in; returns where the
// reference set is read from. s_rot / s_ref_in: shared memory, or (units too large for it) a per-CTA scratch row in
// global memory for the transformed points and the caller's reference array itself (copy_ref = false).
__device__ __forceinline__ const double2* exact_stage(const UnitDesc& ud, const double* __restrict__ test_xy,
                                                      const double* __restrict__ ref_xy, double cosv, double sinv,
                                                      bool identity, double2* s_rot, const double2* s_ref_in,
                                                      bool copy_ref, bool rigid, double2 t) {
    double2* s_ref_w = const_cast<double2*>(s_ref_in);
    const double2* s_ref = copy_ref ? s_ref_in : reinterpret_cast<const double2*>(ref_xy + 2 * ud.ref_off);
    for (int i = threadIdx.x; i < ud.n; i += blockDim.x) {
        const double px = test_xy[2 * (ud.test_off + i)], py = test_xy[2 * (ud.test_off + i) + 1];
        double rx = px, ry = py;
        if (!identity) {
            const double x = __dsub_rn(px, ud.cx), y = __dsub_rn(py, ud.cy);
            rx = __dadd_rn(__dsub_rn(__dmul_rn(x, cosv), __dmul_rn(y, sinv)), ud.cx);
            ry = __dadd_rn(__dadd_rn(__dmul_rn(x, sinv), __dmul_rn(y, cosv)), ud.cy);
        }
        if (rigid) rx = __dadd_rn(rx, t.x), ry = __dadd_rn(ry, t.y);
        s_rot[i] = make_double2(rx, ry);
    }
    if (copy_ref)
        for (int j = threadIdx.x; j < ud.m; j += blockDim.x)
            s_ref_w[j] = make_double2(ref_xy[2 * (ud.ref_off + j)], ref_xy[2 * (ud.ref_off + j) + 1]);
    __syncthreads();
    return s_ref;
}

// The cost of one candidate. Each directed value is the largest row minimum (a non-finite minimum is skipped); for the
// partial cost the (q + 1)-th largest (a non-finite minimum counts as 0); for the mean cost the sum of the row values
// sqrt(minimum) (a non-finite minimum counts as 0), sequential in point order on thread 0, over the count. s_min: n
// (or m) doubles of the CTA (shared memory or a global scratch row) that hold the row minima of the partial cost, the
// row values of the mean cost.
template <Cost COST>
__device__ __forceinline__ double exact_cost(const UnitDesc& ud, const double* __restrict__ test_xy,
                                             const double* __restrict__ ref_xy, double cosv, double sinv, bool identity,
                                             double2* s_rot, const double2* s_ref_in, double* s_red, double* s_min,
                                             bool copy_ref, bool rigid, double2 t) {
    const double2* s_ref = exact_stage(ud, test_xy, ref_xy, cosv, sinv, identity, s_rot, s_ref_in, copy_ref, rigid, t);
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    auto directed = [&](const double2* rows, int nr, const double2* set, int ns, int q) {
        double lmax = 0.0;
        for (int i = threadIdx.x; i < nr; i += blockDim.x) {
            const double2 a = rows[i];
            double mn = INF;
            for (int j = 0; j < ns; ++j) {
                const double2 b = set[j];
                const double dx = __dsub_rn(a.x, b.x), dy = __dsub_rn(a.y, b.y);
                const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
                if (d2 < mn) mn = d2;
            }
            if (COST == kCostPartial) s_min[i] = isfinite(mn) ? mn : 0.0;
            else if (COST == kCostMean) s_min[i] = isfinite(mn) ? __dsqrt_rn(mn) : 0.0;
            else if (isfinite(mn) && mn > lmax) lmax = mn;
        }
        if (COST == kCostFull) return block_max(lmax, s_red);
        __syncthreads();
        if (COST == kCostPartial) return block_kth_largest(s_min, nr, q, s_red);   // ends with a barrier: s_min may be reused
        if (threadIdx.x == 0) {
            double s = 0.0;
            for (int i = 0; i < nr; ++i) s = __dadd_rn(s, s_min[i]);
            s_red[0] = __ddiv_rn(s, (double)nr);
        }
        __syncthreads();
        const double mean = s_red[0];
        __syncthreads();   // s_min and s_red may be reused
        return mean;
    };
    const double fwd = directed(s_ref, ud.m, s_rot, ud.n, ud.q_fwd);   // reference -> transformed
    const double bwd = directed(s_rot, ud.n, s_ref, ud.m, ud.q_bwd);   // transformed -> reference
    if (COST == kCostMean) return fmax(fwd, bwd);
    return fmax(__dsqrt_rn(fwd), __dsqrt_rn(bwd));
}

// Partial and mean costs: g_min != NULL puts the CTA's row minima in a global scratch row (with g_scratch), else shared
// memory after the two staged sets.
template <Cost COST>
__global__ void __launch_bounds__(256)
    k_exact(const UnitDesc* __restrict__ units, const double* __restrict__ test_xy, const double* __restrict__ ref_xy,
            const double2* __restrict__ cs64, const unsigned char* __restrict__ zero_flag,
            const int2* __restrict__ items, const unsigned* __restrict__ n_items, unsigned pool_cap,
            double* __restrict__ sl_dist, int max_n, double2* __restrict__ g_scratch, double* __restrict__ g_min,
            const double2* __restrict__ t64) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* s_red = reinterpret_cast<double*>(smem_raw);
    // g_scratch != NULL: the point sets do not fit shared memory — rotated points in this CTA's global scratch row
    double2* s_rot = g_scratch ? g_scratch + (size_t)blockIdx.x * max_n : reinterpret_cast<double2*>(smem_raw + 64);
    double2* s_ref = g_scratch ? nullptr : s_rot + max_n;
    double* s_min = g_min ? g_min + (size_t)blockIdx.x * max_n : reinterpret_cast<double*>(s_ref + max_n);
    const unsigned total = min(*n_items, pool_cap);
    for (unsigned it = blockIdx.x; it < total; it += gridDim.x) {
        const int2 item = items[it];
        if (item.x < 0) continue;  // uniform per CTA
        const UnitDesc ud = units[item.x];
        const int c = item.y;
        const int i = t64 ? c / ud.n_trans : c;
        const double2 cs = cs64[ud.cand_off + i];
        const bool identity = zero_flag[ud.cand_off + i] != 0;
        const double2 t = t64 ? t64[ud.t_off + (c - i * ud.n_trans)] : make_double2(0.0, 0.0);
        const double d = exact_cost<COST>(ud, test_xy, ref_xy, cs.x, cs.y, identity, s_rot, s_ref, s_red, s_min,
                                             g_scratch == nullptr, t64 != nullptr, t);
        if (threadIdx.x == 0) sl_dist[it] = d;
        __syncthreads();
    }
}

// Dense variant: every candidate [c0, c0+count) of one unit (shortlist overflow
// path and mmrs_eval_exact). t64 != NULL: rigid candidates; paired = true (mmrs_eval_exact_rigid): candidate c takes
// angle c and translation t64[c] instead of the grid product.
template <Cost COST>
__global__ void __launch_bounds__(256)
    k_exact_dense(const UnitDesc* __restrict__ units, int unit, const double* __restrict__ test_xy,
                  const double* __restrict__ ref_xy, const double2* __restrict__ cs64,
                  const unsigned char* __restrict__ zero_flag, long long cs_off, int count, double* __restrict__ out,
                  int max_n, double2* __restrict__ g_scratch, double* __restrict__ g_min, const double2* __restrict__ t64,
                  bool paired) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* s_red = reinterpret_cast<double*>(smem_raw);
    double2* s_rot = g_scratch ? g_scratch + (size_t)blockIdx.x * max_n : reinterpret_cast<double2*>(smem_raw + 64);
    double2* s_ref = g_scratch ? nullptr : s_rot + max_n;
    double* s_min = g_min ? g_min + (size_t)blockIdx.x * max_n : reinterpret_cast<double*>(s_ref + max_n);
    const UnitDesc ud = units[unit];
    for (int c = blockIdx.x; c < count; c += gridDim.x) {
        const int i = (t64 && !paired) ? c / ud.n_trans : c;
        const double2 cs = cs64[cs_off + i];
        const bool identity = zero_flag[cs_off + i] != 0;
        const double2 t = !t64 ? make_double2(0.0, 0.0) : paired ? t64[c] : t64[ud.t_off + (c - i * ud.n_trans)];
        const double d = exact_cost<COST>(ud, test_xy, ref_xy, cs.x, cs.y, identity, s_rot, s_ref, s_red, s_min,
                                             g_scratch == nullptr, t64 != nullptr, t);
        if (threadIdx.x == 0) out[c] = d;
        __syncthreads();
    }
}

// =============================================================================
// K4: per unit, leftmost arg-min over the rechecked candidates in f64 (strict <,
// ties -> lowest candidate index: process_utils.rs:69-74) and the tie count.
// One warp per unit.
// =============================================================================
__global__ void k_select(const UnitDesc* __restrict__ units, int n_units, const double2* __restrict__ cs64,
                         const int2* __restrict__ items, const double* __restrict__ sl_dist,
                         const int* __restrict__ sl_count,
                         const unsigned* __restrict__ sl_base, const unsigned long long* __restrict__ key,
                         const unsigned* __restrict__ rmax_bits, double tie_margin, UnitResultDev* __restrict__ res,
                         const double2* __restrict__ t64) {
    const int u = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (u >= n_units) return;
    const int n = sl_count[u];
    UnitResultDev r;
    if (units[u].flags & kFlagRemote) {   // another rank owns this unit: all-zero entry, the merge is a sum
        if (lane == 0) {
            r.best_idx = 0, r.best_dist = 0.0, r.best_d32 = 0.f, r.n_shortlist = 0, r.n_ties = 0, r.flags = 0;
            res[u] = r;
        }
        return;
    }
    r.best_idx = -1;
    r.best_dist = 0.0;
    r.best_d32 = __uint_as_float((unsigned)(key[u] >> 32));
    r.n_shortlist = n;
    r.n_ties = 0;
    r.flags = units[u].flags;
    if (n > 0) {
        const unsigned base = sl_base[u];
        double bd = __longlong_as_double(0x7ff0000000000000LL);
        int bi = 0x7fffffff;
        for (int k = lane; k < n; k += 32) {
            const double d = sl_dist[base + k];
            const int i = items[base + k].y;
            if (d < bd || (d == bd && i < bi)) {
                bd = d;
                bi = i;
            }
        }
        for (int o = 16; o > 0; o >>= 1) {
            const double od = __shfl_xor_sync(0xffffffffu, bd, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (od < bd || (od == bd && oi < bi)) {
                bd = od;
                bi = oi;
            }
        }
        // Tie count: rechecked candidates within the margin whose ANGLE differs from the winner's. A candidate
        // with the winner's own angle (the -pi / +pi wrap duplicates of a +-180 deg grid) has the winner's cost
        // in any arithmetic, so the lowest index wins there regardless and it is not an ambiguity.
        // Rigid candidates (t64 != NULL): whose TRANSFORM differs, i.e. a different (cos, sin) or a different (tx, ty).
        const double lim = bd + tie_margin * fmax(1.0, (double)__uint_as_float(rmax_bits[u]));
        const long long co = units[u].cand_off, to = units[u].t_off;
        const int nt = t64 ? units[u].n_trans : 1;
        const double2 wcs = cs64[co + bi / nt];
        const double2 wt = t64 ? t64[to + bi % nt] : make_double2(0.0, 0.0);
        int ties = 0;
        for (int k = lane; k < n; k += 32) {
            const int i = items[base + k].y;
            if (i == bi || sl_dist[base + k] > lim) continue;
            const double2 c = cs64[co + i / nt];
            bool differs = c.x != wcs.x || c.y != wcs.y;
            if (t64) {
                const double2 t = t64[to + i % nt];
                differs = differs || t.x != wt.x || t.y != wt.y;
            }
            ties += differs ? 1 : 0;
        }
        for (int o = 16; o > 0; o >>= 1) ties += __shfl_xor_sync(0xffffffffu, ties, o);
        r.best_idx = bi;
        r.best_dist = bd;
        r.n_ties = ties + 1;
    }
    if (lane == 0) res[u] = r;
}

// =============================================================================
// Candidate-axis partition (mmrs_ctx_set_partition 2): every rank swept one contiguous candidate sub-range of every
// unit and holds its LOCAL leftmost f64 arg-min (k_select over its own shortlist, which was cut against the GLOBAL
// FP32 minimum: the packed keys were merged with all-reduce(MIN, uint64) before k_shortlist). res_all = the ranks'
// local results after the all-gather, [world][n_units].
//   k_merge_angle   global leftmost f64 arg-min (lowest distance, ties -> lowest candidate index: process_utils.rs:69-74)
//                   and THIS rank's share of the counts: its shortlist size, its candidates within tie_margin of the
//                   global winner whose angle differs from the winner's, and whether its pool overflowed.
//   k_finish_angle  after the all-reduce(SUM) of those counts.
// One warp per unit.
// =============================================================================
__global__ void k_merge_angle(const UnitDesc* __restrict__ units, int n_units, int world,
                              const UnitResultDev* __restrict__ res_all, const double2* __restrict__ cs64,
                              const int2* __restrict__ items, const double* __restrict__ sl_dist,
                              const int* __restrict__ sl_count, const unsigned* __restrict__ sl_base,
                              const unsigned long long* __restrict__ key, const unsigned* __restrict__ rmax_bits,
                              double tie_margin, UnitResultDev* __restrict__ res, int4* __restrict__ cnt) {
    const int u = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (u >= n_units) return;
    long long bi = -1;
    double bd = 0.0;
    for (int r = 0; r < world; ++r) {   // rank order = candidate order, but compare explicitly
        const UnitResultDev x = res_all[(size_t)r * n_units + u];
        if (x.best_idx < 0) continue;
        if (bi < 0 || x.best_dist < bd || (x.best_dist == bd && x.best_idx < bi)) bi = x.best_idx, bd = x.best_dist;
    }
    const int n = sl_count[u];
    int ties = 0;
    if (bi >= 0 && n > 0) {
        const unsigned base = sl_base[u];
        const double lim = bd + tie_margin * fmax(1.0, (double)__uint_as_float(rmax_bits[u]));
        const long long co = units[u].cand_off;
        const double2 wcs = cs64[co + bi];
        for (int k = lane; k < n; k += 32) {
            const int i = items[base + k].y;
            if (i == bi || sl_dist[base + k] > lim) continue;
            const double2 c = cs64[co + i];
            ties += (c.x != wcs.x || c.y != wcs.y) ? 1 : 0;
        }
        for (int o = 16; o > 0; o >>= 1) ties += __shfl_xor_sync(0xffffffffu, ties, o);
    }
    if (lane == 0) {
        UnitResultDev r;
        r.best_idx = bi;
        r.best_dist = bd;
        r.best_d32 = __uint_as_float((unsigned)(key[u] >> 32));
        r.n_shortlist = 0;
        r.n_ties = 0;
        r.flags = units[u].flags;
        res[u] = r;
        cnt[u] = make_int4(n > 0 ? n : 0, ties, n < 0 ? 1 : 0, 0);
    }
}

__global__ void k_finish_angle(int n_units, const int4* __restrict__ cnt, UnitResultDev* __restrict__ res) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= n_units) return;
    const int4 c = cnt[u];
    // a pool overflow on any rank: every rank rechecks ALL candidates of the unit in f64 at download (negative count)
    res[u].n_shortlist = c.z ? -1 : c.x;
    res[u].n_ties = res[u].best_idx >= 0 ? c.y + 1 : 0;
}

// Rigid runs: R_eff = Rmax + max_j |t_j| per unit (the coordinate magnitude the FP32 error bound scales with), rounded
// up to FP32 bits; used wherever the rotation-only sweep uses Rmax (K2 window, tie margin).
__global__ void k_reff(const unsigned* __restrict__ rmax_bits, const double* __restrict__ tmax, unsigned* __restrict__ reff,
                       int n_units) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u < n_units) reff[u] = __float_as_uint(__double2float_ru((double)__uint_as_float(rmax_bits[u]) + tmax[u]));
}

// =============================================================================
// FP32 peak probe: 8 independent FFMA chains per thread, all SMs busy.
// =============================================================================
__global__ void __launch_bounds__(256) k_fp32_probe(float* out, int iters, float a, float b) {
    float x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            x0 = fmaf(x0, a, b);
            x1 = fmaf(x1, a, b);
            x2 = fmaf(x2, a, b);
            x3 = fmaf(x3, a, b);
            x4 = fmaf(x4, a, b);
            x5 = fmaf(x5, a, b);
            x6 = fmaf(x6, a, b);
            x7 = fmaf(x7, a, b);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

}  // namespace mmrs
