// msm.cuh — variable-base multi-scalar multiplication on Pallas / Vesta for sm_100a.
//
// Drop-in semantics of ark_ec::VariableBaseMSM::{msm_bigint, msm} as the reference calls them
// (poly-commitment/src/ipa.rs:649-672,943,953,487,497; commitment.rs:382,387 — SURVEY.md §8 rows a1/a2):
//     result = sum_i s_i * P_i       bases affine (x, y Montgomery; identity allowed), scalars canonical 255-bit
// (or Montgomery, converted on the device first), min(len) semantics for msm_bigint.
//
// B200 shape (Pippenger with signed digits, bucket method):
//   * resident bases: an SRS (or a Lagrange basis) is uploaded once and kept in HBM — optionally as a
//     PRECOMPUTED table T[w][i] = 2^(c*w) * P_i (nwin * n affine points; 64 MiB for n = 2^16, c = 16).  With the table
//     all windows share ONE bucket set, so there is no per-window bucket reduction and no Horner doubling chain:
//     180 GB of HBM buys away ~half of the serial tail.  Without a table (one-shot bases) there is one bucket set per
//     window and the host combines the windows.
//   * scalars are recoded to signed base-2^c digits in (-2^(c-1), 2^(c-1)]; (digit != 0) entries are counting-sorted by
//     bucket (histogram -> scan -> scatter, all on device);
//   * accumulation is task based: the histogram is known before any point is touched, so every bucket's sorted entries
//     are cut into ceil(n_b / K) nearly equal tasks; a thread sums one task (<= K XYZZ mixed additions).  The task partials of
//     a bucket are summed thread-parallel in two balanced levels (runs of 4 consecutive partials, then <= 4 run sums per
//     bucket) — thread-serial additions have twice the throughput of the quad-cooperative ones (tools/microbench.py), so the
//     bulk of the reduction stays thread-serial and quads are kept for the short dependent tails.  The rare giant bucket (all
//     points in one bucket — the kimchi witness columns, SURVEY.md §3.1) gets 16 CTAs.  No atomics touch curve points;
//   * bucket reduction sum_b (b+1) B_b in two levels: with b+1 = hi * W + lo the sum is W * sum_hi hi R[hi] + sum_lo lo C[lo]
//     (row / column sums of the bucket grid, one CTA each), then bit slices T_t = sum of the rows / columns whose index has
//     bit t set, and the host finishes with c doublings;
//   * k MSMs over the same bases (the chunks of t, the 15 witness columns, the L/R pair of an IPA round) run as ONE pipeline
//     with k bucket groups: every latency-bound stage is paid once per batch, not once per MSM.
#pragma once
#include <vector>

#include "common.cuh"

namespace zkb {

constexpr unsigned MSM_MAX_WINDOW_BITS = 16;
constexpr uint32_t MSM_MAX_GIANTS = 64;       // buckets with > smax tasks get 16 CTAs each (k_giant_finish)
constexpr unsigned MSM_MAX_BATCH = 16;        // MSMs fused into one pipeline (scalar pointers travel as a kernel parameter)
struct MsmScalarSet {
    const fe* p[MSM_MAX_BATCH];
    uint32_t off[MSM_MAX_BATCH];              // first base of MSM j inside the resident set
};

// A resident set of bases on one device.
struct MsmBases {
    int curve = 0;             // 0 Pallas, 1 Vesta
    size_t n = 0;              // number of points
    unsigned c = 0;            // window bits of the precomputed table (0: no table)
    unsigned nwin = 0;         // windows in the table
    affine_t* d_points = nullptr;  // [max(1,nwin)][n]  row w holds 2^(c*w) * P_i
};

// Growable device scratch of one context/device (sized for the largest call seen so far).
struct MsmWorkspace {
    size_t cap_entries = 0, cap_partials = 0, cap_buckets = 0, cap_bits = 0, cap_hbits = 0;
    int32_t* d_digits = nullptr;      // [k][nwin][n]
    uint32_t* d_entries = nullptr;    // [M]  point index | sign << 31, sorted by bucket
    xyzz_t* d_partials = nullptr;     // [tasks] one partial sum per accumulation task
    uint32_t* d_counts = nullptr;     // [NB]     histogram, then scatter cursors counting down: zero between calls
    uint32_t* d_offsets = nullptr;    // [NB + 1] exclusive scan of the counts
    uint32_t* d_task_off = nullptr;   // [NB + 1] exclusive scan of ceil(count / K)
    xyzz_t* d_buckets = nullptr;      // [NB]
    uint64_t* d_chain = nullptr;      // [tiles] chained scan of k_plan: inclusive (entries << 32 | tasks) per tile
    uint32_t* d_chain_flag = nullptr; // [tiles] epoch stamps of d_chain
    uint32_t epoch = 0;               // bumped per run (no flag memset)
    xyzz_t* d_bitsums = nullptr;      // row/column sums [G][nrows + W], then the slice sums [G][c]
    xyzz_t* h_bitsums = nullptr;      // pinned host copies of [G][c]: two slots (a lane may run ahead of the host tail by one MSM)
    unsigned h_slot = 0;              // slot the next msm_run writes (result at h_bitsums + h_slot * cap_hbits)
    xyzz_t* d_T_out = nullptr;        // when set: the slice sums are copied HERE (device, capacity d_T_cap points) instead of to
    size_t d_T_cap = 0;               // the host, and nothing is synchronised (multi-GPU exchange, zk_msm_partial)
    bool defer_sync = false;          // msm_run returns after enqueueing the D2H copy; the caller synchronises
    uint32_t* d_meta = nullptr;       // [0] sorted entries, [1] tasks, [2] giant buckets
    uint32_t* d_giants = nullptr;     // [MSM_MAX_GIANTS] bucket ids
    xyzz_t* d_giant_slices = nullptr; // [MSM_MAX_GIANTS][GIANT_SLICES] per-CTA slice sums of a giant's partials
    uint32_t* d_giant_tickets = nullptr;  // [MSM_MAX_GIANTS] arrival counters (self-resetting)
    uint32_t chunk = 0;               // K override (0: chosen per call so that the tasks fill the machine once)
    uint32_t wave_threads = 0;        // accumulation threads per SM the task count is sized for (0: built-in default)
    bool tma_gather = false;          // A/B switch: gather the points with the bulk asynchronous copy engine (k_accumulate_tma)
    bool pdl = true;                  // A/B switch: kernels 2.. by programmatic dependent launch, no per-call memsets (false: plain
                                      // launches behind two memsets, the earlier launch shell)
    int sm_count = 148;               // SMs of the device (set by the context)
    bool profile = false;             // record an event after every stage
    cudaEvent_t ev[8] = {};           // MSM_ST_COUNT + 1 stage boundaries
    float stage_ms[8] = {};           // duration of each stage in the last profiled call
};
void msm_workspace_free(MsmWorkspace& ws);

int msm_default_window(size_t n, bool precomputed);
unsigned msm_num_windows(unsigned c);

// Upload n affine points (host or device memory, 16 u32 each) and optionally build the window table.
template <class F> int msm_bases_create(MsmBases& b, const affine_t* pts, bool pts_on_device, size_t n, unsigned c_table, cudaStream_t st);
void msm_bases_free(MsmBases& b);

// Optional per-stage device timing (CUDA events on the launching stream), filled when MsmWorkspace::profile is set.
enum MsmStage { MSM_ST_RECODE = 0, MSM_ST_PLAN, MSM_ST_SCATTER, MSM_ST_ACCUMULATE, MSM_ST_FINISH, MSM_ST_BITSUM, MSM_ST_COUNT };

// What msm_run leaves in ws.h_bitsums: batch x groups x c XYZZ points T[j][g][t]; MSM j is sum_g 2^(c g) sum_t 2^t T[j][g][t].
struct MsmResultShape {
    unsigned c = 0, groups = 0;   // groups == 0: empty MSM (identity)
    unsigned batch = 0;
};

// k <= MSM_MAX_BATCH MSMs in one pipeline, MSM j over bases[offs[j] .. offs[j]+n).  d_scalars[j]: the n scalars of MSM j, already on the device
// (8 u32 each).  window c: 0 = default (ignored when the bases carry a precomputed table).  Synchronises the stream (unless
// ws.defer_sync / ws.d_T_out); the O(c) tail is finished by the caller.
// d_extra / n_extra: n_extra further points that belong to this call only (h and the fresh base U of an IPA round,
// poly-commitment/src/ipa.rs:944,954), laid out like the table — row w holds 2^(c*w) * E_e at d_extra[w * n_extra + e] (one row
// without a table); every scalar vector then carries n_main + n_extra scalars, the extras' last.
// out[i] = sum over r < world of all[r * count + i]   (the cross-rank sum of gathered slice sums, i < count)
template <class F> int msm_sum_partials(const xyzz_t* d_all, size_t world, size_t count, xyzz_t* d_out, cudaStream_t st);

template <class F, class FS>
int msm_run(const MsmBases& b, const size_t* offs, size_t n_main, const fe* const* d_scalars, unsigned k, bool scalars_mont, unsigned c,
            MsmWorkspace& ws, cudaStream_t st, MsmResultShape* shape, unsigned* launches, const affine_t* d_extra = nullptr,
            size_t n_extra = 0);

// group_ntt.cu: Lagrange-basis commitments of the domain of size 2^log_n from the resident generators (SRS::lagrange_basis)
template <class F, class FS> int lagrange_basis_build(const MsmBases& g, unsigned log_n, unsigned chunk, affine_t* d_out, cudaStream_t st, unsigned* launches);

}  // namespace zkb
