// mmrs_internal.hpp — private state behind the opaque mmrs_ctx of include/mmrs_b200.h.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <map>
#include <string>
#include <vector>

#include "../../include/mmrs_b200.h"

namespace mmrs {
struct UnitDesc {
    long long test_off, ref_off;  // point offsets into the f64 (x,y) arrays
    int n, m;                     // test / reference point counts
    double cx, cy;                // rotation centre
    long long lay_off;            // float4 offset of this unit's staging block (A, B, NB, tail, K1e's grid block)
    int n_chunks;                 // A is stored as n_chunks x (TA/2) x 32 float4
    int m_pairs;                  // B is stored as m_pairs float4 (bx0,by0,bx1,by1)
    long long cand_off;           // offset of this unit's grid in the cos/sin tables
    int n_cand;
    int flags;
    long long dist_off;           // offset of this unit's first candidate in dist32
    int ta;                       // register tile of this unit's size class (test points per lane of K1)
    int n_tail;                   // exact tiling: the last n_tail (< 32) test points live in the tail block, not in a slot
    int c_lo, c_hi;               // candidates [c_lo, c_hi) are swept by THIS rank (all of them unless the batch is
                                  // partitioned across ranks: whole units -> empty range on the other ranks, candidate
                                  // axis -> one contiguous sub-range per rank, global indices kept)
    long long t_off;              // rigid runs: offset of this unit's translation grid in the t64 / t32 tables
    int n_trans;                  // translations per angle (1 without a translation grid): candidate c = i n_trans + j
    short q_fwd, q_bwd;           // partial cost: points that do not count, reference -> test (q(m)) / test -> reference (q(n))
    int eb_grid;                  // K1e: the staging image carries the grid block (sweep_kernels.cuh, K0), else full seed scans
};
constexpr int kFlagRemote = 0x400;  // internal UnitDesc.flags bit: another rank owns this unit (never leaves the library)

// How a run scores its candidates: the dense sweep, or a tier that scores them approximately (or bounds them) and
// re-scores a list with the exact FP32 sweep. The values are the codes mmrs_sweep_prefilter_info reports in out[0].
enum Tier : int { kTierDense = 0, kTierTc = 1, kTierPrune = 2, kTierXf = 3 };

// What a candidate's cost is (include/mmrs_b200.h): the symmetric Hausdorff distance, the partial (rank-K) distance or
// the mean (modified Hausdorff) distance. Partial and mean runs are solo: the dense sweep on one device, no tier.
enum Cost : int { kCostFull = 0, kCostPartial = 1, kCostMean = 2 };

struct WorkItem {
    int unit;
    int begin;  // first candidate
    int count;  // candidates in this tile
    int pad;
};

struct UnitResultDev {
    long long best_idx;
    double best_dist;
    float best_d32;
    int n_shortlist;
    int n_ties;
    int flags;
};

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};
int set_err(mmrs_ctx* ctx, int code, const std::string& msg);
int comm_broadcast(mmrs_ctx* ctx, void* host, size_t bytes, int root);
}  // namespace mmrs

struct mmrs_ctx {
    int device = 0;
    int n_sm = 148;
    int sm_clock_khz = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_tc[3] = {nullptr, nullptr, nullptr};  // tensor-core prefilter: start, after K1t, after tier-2 FP32
    std::string err;

    // batch state
    bool ready = false, ran = false;
    int64_t n_units = 0;
    int mode = 0;
    // size classes of the uploaded units: K1 is launched once per class (register tile, chunked?, exact tiling?)
    struct SweepClass {
        int ta = 2;
        bool multi = false, tailp = false;
        bool big = false;                       // units beyond K1's shared-memory staging: K1b (k_sweep_big)
        size_t smem = 0;
        size_t work_begin = 0, work_count = 0;  // range of h_work / d_work
        long long cost = 0;                     // padded pair evaluations per candidate, summed over the class
        int eb_warps = 0;                       // warps per CTA of the early-break kernel (k_sweep_eb): 8 for K1e,
                                                // 8, 4, 2 or 1 for K1e-partial
        size_t smem_eb = 0;                     // its shared memory per CTA
        bool eb = false;                        // the dense sweep of this class runs K1e (decided per grid set)
        long long live = 0;                     // candidates of this class swept by this rank
    };
    std::vector<SweepClass> classes;
    std::vector<int> class_of_unit;
    long long big_scratch_per_warp = 0;         // K1b: floats of row-minimum scratch per warp (largest padded test set)
    mmrs::DevBuf d_big_rows, d_exact_scratch;   // K1b row minima across reference blocks; K3 rotated points of oversize sets
    int max_pts = 1;
    long long total_cands = 0;
    double opt_rel = 2e-6, opt_abs = 2e-6, tie_margin = 0.0;
    int cap = 64;
    unsigned pool_cap = 0;
    int launches = 0, upload_launches = 0;
    long long eval_launches = 0;
    std::vector<mmrs_grid> grids;
    std::vector<int> grid_of_unit;
    std::vector<mmrs::UnitDesc> h_units;
    std::vector<mmrs::WorkItem> h_work;
    std::vector<double> h_cs;
    std::vector<unsigned char> h_zero;
    std::vector<float> h_rmax;
    std::vector<double> f_test, f_ref;        // the batch without its non-finite points (only when one was found)
    std::vector<int64_t> f_toff, f_roff;
    std::map<int64_t, std::vector<double>> overflow_dist;
    void* h_res = nullptr;  // pinned
    size_t h_res_cap = 0;

    mmrs::DevBuf d_test, d_ref, d_units, d_work, d_lay, d_cs64, d_cs32, d_zero, d_dist32, d_key, d_rmax, d_sl_base,
        d_sl_dist, d_sl_count, d_items, d_nitems, d_res, d_tmp;

    // sweep tiers: K1t, K1x (expanded form, k_sweep<.., XF>) and K1p (lower-bound pruning)
    mmrs::Tier tier = mmrs::kTierDense;       // decided per grid set (apply_grids)
    mmrs::Tier tier_ran = mmrs::kTierDense;   // the last run's: the planned tier, or dense when it had no work

    // tensor-core prefilter tier (tc_kernels.cuh)
    int opt_prefilter = 0;      // mmrs_sweep_opts.prefilter: 0 auto, 1 off, 2 required
    bool tc_shape_ok = false;   // every live unit has kTcMinPts <= n, m <= kTcMaxPts (decided at upload)
    double xf_abs = 8e-6;       // its tier-1 window: d^2 <= dmin^2 + xf_abs * Rmax^2 (>= 4.8x the proven error bound)
    double tc_abs = 4e-6;       // tier-1 window: d^2 <= dmin^2 + tc_abs * Rmax^2
    unsigned l1_cap = 0;
    size_t smem_tc = 0;
    std::vector<mmrs::WorkItem> h_work_tc;
    mmrs::DevBuf d_work_tc, d_key_tc, d_l1_items, d_l1_count, d_l1_base, d_l1_n;

    // exact lower-bound pruning tier (k_lb, sweep_kernels.cuh)
    int opt_prune = 0;          // mmrs_sweep_opts.prune / mmrs_ctx_set_prune: 0 off, 1 on where the batch qualifies
    int ctx_prune = 0;          // context-wide default used when the opts do not say
    bool lb_shape_ok = false;   // every live unit has >= 128 points per set (decided at upload)
    int lb_R = 64;              // rows of a lower-bound unit (32 * TA_lb)
    size_t smem_lb = 0;
    std::vector<mmrs::UnitDesc> h_units_lb;   // [2 U]: pass A (test rows) then pass B (reference rows)
    std::vector<mmrs::WorkItem> h_work_lb;
    mmrs::DevBuf d_units_lb, d_lay_lb, d_work_lb;

    // early-break dense sweep K1e (k_sweep_eb, sweep_kernels.cuh)
    int eb_env = -1;            // MMRS_EARLY_BREAK at upload: -1 unset (K1e where 3 CTAs fit per SM), 0 K1 everywhere, 1 K1e wherever it fits
    bool eb_ran = false;
    long long eb_cands = 0;     // candidates K1e scored in the last run
    mmrs::DevBuf d_eb_pairs;    // pair distances K1e evaluated in the last run (one 64-bit counter)

    // rigid candidates (mmrs_rigid_sweep_*): a translation grid per unit on top of its angle grid
    bool rigid = false;                     // the uploaded grids carry translation grids
    std::vector<mmrs_tgrid> tgrids;
    std::vector<int> tgrid_of_unit;
    std::vector<double> h_t;                // (tx, ty) of every translation of every translation grid
    std::vector<double> h_tmax;             // per unit: largest |t| of its translation grid
    mmrs::DevBuf d_t64, d_t32, d_tmax, d_reff;   // translation tables; per unit R_eff = Rmax + max |t| (float bits)

    // the cost (mmrs_partial_sweep_upload, mmrs_mean_sweep_upload): set with the points, kept across regrids
    mmrs::Cost cost = mmrs::kCostFull;
    double inlier_fraction = 1.0;   // partial cost

    // partition of every batched sweep across ranks (mmrs_ctx_comm_init / mmrs_ctx_set_shard / mmrs_ctx_set_partition)
    int shard_rank = 0, shard_world = 1;
    mmrs_exchange_fn exchange = nullptr;   // host callback (any transport); used when no NCCL communicator is bound
    void* exchange_user = nullptr;
    void* comm = nullptr;                  // ncclComm_t (mmrs_comm.hpp): collectives on device buffers, on `stream`
    int part_axis = 1;                     // 1 = whole units, 2 = candidate sub-ranges of every unit
    int part_active = 0;                   // axis in force for the uploaded batch (0 = not partitioned)
    int opt_partition = 0;                 // mmrs_sweep_opts.partition of the uploaded batch
    long long collectives = 0;             // collectives issued since the context was created
    mmrs::DevBuf d_bcast;                  // staging of comm_broadcast
    mmrs::DevBuf d_res_all, d_cnt;         // candidate axis: the ranks' local results [world][U]; (n_shortlist, ties, overflow) sums

    // counters of the last mmrs_process_cases call
    int64_t stats[5] = {0, 0, 0, 0, 0};
    // host staging of the intrapullback units, kept across calls: 26 MB of FRESH memory per call (config 3) is 6 500
    // page faults, more than sampling the frames costs
    std::vector<double> host_units_test, host_units_ref;

    void free_all();
};
