// msm.cu — kernels and pipeline of the Pallas/Vesta MSM (see msm.cuh for semantics and reference call sites).
#include "msm.cuh"
#include "quad.cuh"

#include <algorithm>

namespace zkb {

unsigned msm_num_windows(unsigned c) { return (256 + c - 1) / c; }  // top signed digit cannot carry out (scalars < 2^254 + 2^127)

int msm_default_window(size_t n, bool precomputed) {
    // accumulation costs ceil(256/c) * n mixed additions; the bucket side grows with 2^(c-1) (one bucket set with a
    // table, one per window without).  Measured on B200 (tools/sweep.py): 2^16 points -> c = 15 with a table, 12 without.
    unsigned l = 0;
    while (((size_t)1 << (l + 1)) <= n) l++;
    int c = (int)l - (precomputed ? 1 : 4);
    if (c < 4) c = 4;
    if (c > (int)MSM_MAX_WINDOW_BITS) c = MSM_MAX_WINDOW_BITS;
    return c;
}

// ---------------------------------------------------------------------------------------------- table of 2^(cw) P
template <class F> __global__ void k_build_table(affine_t* table, size_t n, unsigned c, unsigned nwin) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    affine_t p = load_affine_nc(table + i);
    xyzz_t acc = xyzz_from_affine<F>(p);
    for (unsigned w = 1; w < nwin; w++) {
        for (unsigned k = 0; k < c; k++) acc = xyzz_dbl<F>(acc);
        store_affine(table + (size_t)w * n + i, xyzz_to_affine<F>(acc));
    }
}

// The same table with ONE field inversion per point instead of one per row (Montgomery's trick over the rows of a point):
// ~255 doublings + 1 inversion + 8 multiplications per row, 3.4x less arithmetic than k_build_table.  nwin <= TABLE_MAX_ROWS.
constexpr unsigned TABLE_MAX_ROWS = 33;   // windows of >= 8 bits
template <class F> __global__ void __launch_bounds__(128) k_build_table_batched(affine_t* table, size_t n, unsigned c, unsigned nwin) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const affine_t p = load_affine_nc(table + i);
    if (affine_is_inf(p)) {
        for (unsigned w = 1; w < nwin; w++) store_affine(table + (size_t)w * n + i, p);
        return;
    }
    xyzz_t pts[TABLE_MAX_ROWS];
    fe pre[TABLE_MAX_ROWS];
    xyzz_t acc = xyzz_from_affine<F>(p);
    for (unsigned w = 1; w < nwin; w++) {
        for (unsigned k = 0; k < c; k++) acc = xyzz_dbl<F>(acc);
        pts[w] = acc;
        const fe z = fe_mul<F>(acc.ZZ, acc.ZZZ);        // never zero: the curve has prime order, doubling a finite point stays finite
        pre[w] = w == 1 ? z : fe_mul<F>(pre[w - 1], z);
    }
    if (nwin < 2) return;
    fe inv = fe_inv<F>(pre[nwin - 1]);
    for (unsigned w = nwin - 1; w >= 1; w--) {
        const fe zi = w == 1 ? inv : fe_mul<F>(inv, pre[w - 1]);          // 1 / (ZZ_w * ZZZ_w)
        inv = fe_mul<F>(inv, fe_mul<F>(pts[w].ZZ, pts[w].ZZZ));
        affine_t r;
        r.x = fe_mul<F>(pts[w].X, fe_mul<F>(zi, pts[w].ZZZ));              // X / ZZ
        r.y = fe_mul<F>(pts[w].Y, fe_mul<F>(zi, pts[w].ZZ));               // Y / ZZZ
        store_affine(table + (size_t)w * n + i, r);
    }
}

template <class F> int msm_bases_create(MsmBases& b, const affine_t* pts, bool pts_on_device, size_t n, unsigned c_table, cudaStream_t st) {
    if (c_table > MSM_MAX_WINDOW_BITS) { zk_set_error("msm: table window %u > %u", c_table, MSM_MAX_WINDOW_BITS); return ZK_ERR_INVALID; }
    b.n = n;
    b.c = c_table;
    b.nwin = c_table ? msm_num_windows(c_table) : 0;
    size_t rows = c_table ? b.nwin : 1;
    ZK_CUDA(cudaMalloc(&b.d_points, std::max<size_t>(rows * n, 1) * sizeof(affine_t)));
    if (n == 0) return ZK_OK;
    ZK_CUDA(cudaMemcpyAsync(b.d_points, pts, n * sizeof(affine_t), pts_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    if (c_table) {
        if (b.nwin <= TABLE_MAX_ROWS) k_build_table_batched<F><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(b.d_points, n, c_table, b.nwin);
        else k_build_table<F><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(b.d_points, n, c_table, b.nwin);
        ZK_CUDA(cudaGetLastError());
    }
    ZK_CUDA(cudaStreamSynchronize(st));
    return ZK_OK;
}

void msm_bases_free(MsmBases& b) {
    if (b.d_points) cudaFree(b.d_points);
    b = MsmBases();
}

// ---------------------------------------------------------------------------------------------- launch chain
// Every kernel of msm_run after the first is launched with programmatic dependent launch (PDL): its CTAs may become resident while
// the previous kernel's last CTAs still run, and wait in pdl_wait() (griddepcontrol.wait) until that kernel has completed and its
// stores are visible.  Two rules make every read of the pipeline ordered:
//   (1) every thread of every kernel after the first executes pdl_wait() before it exits, triggers, or reads the previous kernel's
//       output, and writes no global memory before it.  (The first, k_recode, is an ordinary launch: it starts after everything
//       before it on the stream, the previous call's kernels included.)  So kernel N completes only after kernel N-1 has completed, and by
//       induction after every earlier kernel: reads after the wait see the output of ANY earlier kernel (gridsum reading buckets
//       written by accumulate or the finish kernels, bucket_finish reading offsets from plan, ...);
//   (2) kernel N is launched only once every CTA of kernel N-1 has triggered or exited, which by (1) is after N-1's wait, i.e.
//       after kernel N-2 completed.  So the prologue BEFORE the wait may read what kernel N-2 or earlier wrote: the plan's
//       offsets, task_off and meta in accumulate, run_sum and bucket_finish (plan is at least two kernels back there).
// Without the PDL attribute (profile mode, option msm_pdl = 0) both instructions are no-ops and stream order applies.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------- recode + histogram
// One thread per scalar of one MSM of the batch (blockIdx.y): Montgomery -> canonical if asked (VariableBaseMSM::msm ==
// into_bigint + msm_bigint), then signed base-2^c digits d_w in (-2^(c-1), 2^(c-1)]; digit w of scalar i of MSM j at
// digits[(j*nwin + w)*n + i]; per-bucket counts.  Bucket group of (MSM j, window w): j*gpm + (per_window ? w : 0).
template <class FS>
__global__ void k_recode(MsmScalarSet sc, int scalars_mont, size_t n, unsigned c, unsigned nwin, unsigned gpm, int per_window,
                         int32_t* digits, uint32_t* counts, uint32_t* meta) {
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) meta[2] = 0;   // giant list of this run (k_plan)
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned j = blockIdx.y;
    fe s = load_fe_nc(sc.p[j] + i);
    if (scalars_mont) s = fe_from_mont<FS>(s);
    const uint32_t half = 1u << (c - 1), mask = (1u << c) - 1;
    const uint32_t B = half;
    uint32_t carry = 0;
    for (unsigned w = 0; w < nwin; w++) {
        unsigned off = w * c, limb = off >> 5, sh = off & 31;
        uint32_t v = 0;
        if (limb < 8) {
            v = s.v[limb] >> sh;
            if (sh + c > 32 && limb + 1 < 8) v |= s.v[limb + 1] << (32 - sh);
        }
        uint32_t d = (v & mask) + carry;
        int32_t sd;
        if (d > half) { sd = (int32_t)d - (int32_t)(1u << c); carry = 1; }
        else { sd = (int32_t)d; carry = 0; }
        digits[((size_t)j * nwin + w) * n + i] = sd;
        // warp-aggregated histogram update: lanes that hit the same bucket (kimchi's all-ones columns: all of them) elect
        // one lane to add their count — one atomic per distinct bucket per warp instead of one per lane
        const uint32_t mag = (uint32_t)(sd < 0 ? -sd : sd);
        const uint32_t key = sd != 0 ? (j * gpm + (per_window ? w : 0)) * B + (mag - 1) : 0xffffffffu;
        const uint32_t peers = __match_any_sync(__activemask(), key);
        if (sd != 0 && (threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&counts[key], (uint32_t)__popc(peers));
    }
    pdl_trigger();
}

// Planning pass over the histogram: exclusive scans of the bucket counts (-> offsets of the sorted entry list) and of the
// per-bucket task counts s_b = ceil(n_b / K) (-> task_off).  One CTA per tile of 4096 buckets; the tiles are chained (tile t
// spins on tile t-1's published inclusive total — tiles are dispatched in order, so the predecessor is always resident), which
// keeps the scan a single launch for any batch size.  64-bit lanes carry (entry count << 32 | task count): one scan yields both.
// Buckets with more than smax tasks ("giant": the all-ones witness columns of kimchi put ~n entries in one bucket,
// SURVEY.md §3.1) are listed for k_giant_finish.  Empty buckets get the identity here (all-zero XYZZ): every other bucket is
// written by exactly one of k_accumulate (one task), k_giant_finish, k_bucket_finish(_serial).  The counts stay: k_scatter
// counts them down to zero as its cursors, so every call finds them zeroed.
__device__ __forceinline__ uint64_t block_excl_scan_1024(uint64_t v, uint64_t* warp_sums, uint64_t* tile_total) {
    const unsigned tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    uint64_t x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint64_t y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= (unsigned)d) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
        uint64_t ws = warp_sums[lane], z = ws;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint64_t y = __shfl_up_sync(0xffffffffu, z, d);
            if (lane >= (unsigned)d) z += y;
        }
        warp_sums[lane] = z - ws;
        if (lane == 31) *tile_total = z;
    }
    __syncthreads();
    uint64_t excl = warp_sums[wid] + (x - v);
    __syncthreads();
    return excl;
}

constexpr unsigned PLAN_PER_THREAD = 4, PLAN_TILE = 1024 * PLAN_PER_THREAD;
__global__ void __launch_bounds__(1024) k_plan(uint32_t* counts, uint32_t* offsets, uint32_t* task_off, uint32_t nb, uint32_t K, uint32_t smax,
                                                 uint32_t* meta, uint32_t* giants, uint64_t* chain, uint32_t* chain_flag, uint32_t epoch,
                                                 xyzz_t* buckets) {
    __shared__ uint64_t warp_sums[32];
    __shared__ uint64_t tile_total, prefix_s;
    const unsigned tid = threadIdx.x, tile = blockIdx.x;
    const uint32_t i0 = tile * PLAN_TILE + tid * PLAN_PER_THREAD;
    uint32_t v[PLAN_PER_THREAD];
    uint64_t pk[PLAN_PER_THREAD], sum = 0;
    pdl_wait();
#pragma unroll
    for (unsigned k = 0; k < PLAN_PER_THREAD; k++) {
        v[k] = i0 + k < nb ? counts[i0 + k] : 0;
        if (i0 + k < nb && v[k] == 0) store_xyzz(buckets + i0 + k, xyzz_identity());
        pk[k] = ((uint64_t)v[k] << 32) | ((v[k] + K - 1) / K);
        sum += pk[k];
    }
    uint64_t ex = block_excl_scan_1024(sum, warp_sums, &tile_total);
    if (tid == 0) {
        uint64_t prefix = 0;
        if (tile > 0) {
            volatile uint32_t* f = chain_flag + (tile - 1);
            while (*f != epoch) { }
            __threadfence();
            prefix = *(volatile uint64_t*)(chain + (tile - 1));
        }
        *(volatile uint64_t*)(chain + tile) = prefix + tile_total;
        __threadfence();
        *(volatile uint32_t*)(chain_flag + tile) = epoch;
        prefix_s = prefix;
    }
    __syncthreads();
    ex += prefix_s;
#pragma unroll
    for (unsigned k = 0; k < PLAN_PER_THREAD; k++) {
        if (i0 + k < nb) {
            offsets[i0 + k] = (uint32_t)(ex >> 32);
            task_off[i0 + k] = (uint32_t)ex;
            if ((uint32_t)pk[k] > smax) {
                uint32_t gi = atomicAdd(&meta[2], 1u);
                if (gi < MSM_MAX_GIANTS) giants[gi] = i0 + k;
            }
        }
        ex += pk[k];
    }
    if (tile == gridDim.x - 1 && tid == 0) {
        const uint64_t tot = prefix_s + tile_total;
        offsets[nb] = (uint32_t)(tot >> 32); task_off[nb] = (uint32_t)tot;
        meta[0] = (uint32_t)(tot >> 32); meta[1] = (uint32_t)tot;
    }
    pdl_trigger();
}

// Counting-sort scatter: entry (point index | sign) of every non-zero digit goes to its bucket's range.  The cursors are the
// histogram, counted DOWN: a bucket's slots are handed out from its end, and the counts are zero again when the kernel ends.
__global__ void k_scatter(const int32_t* digits, size_t n, unsigned c, unsigned nwin, unsigned batch, unsigned gpm, int per_window, MsmScalarSet sc,
                          size_t table_stride, int use_table, size_t n_main, size_t n_extra, uint32_t main_count, const uint32_t* offsets,
                          uint32_t* cursors, uint32_t* entries) {
    size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool in_range = id < n * nwin * batch;
    pdl_wait();
    int32_t sd = in_range ? digits[id] : 0;
    const unsigned jw = (unsigned)(id / n), j = jw / nwin, w = jw - j * nwin;
    size_t i = id - (size_t)jw * n;
    const uint32_t B = 1u << (c - 1);
    uint32_t mag = (uint32_t)(sd < 0 ? -sd : sd);
    uint32_t key = sd != 0 ? (j * gpm + (per_window ? w : 0)) * B + (mag - 1) : 0xffffffffu;
    // warp-aggregated cursor bump (see k_recode): the leader reserves a run, every peer takes its rank inside it
    const uint32_t peers = __match_any_sync(0xffffffffu, key);
    const unsigned lane = threadIdx.x & 31, leader = (unsigned)(__ffs(peers) - 1);
    uint32_t base = 0;
    if (sd != 0 && lane == leader) base = atomicSub(&cursors[key], (uint32_t)__popc(peers)) - (uint32_t)__popc(peers);
    base = __shfl_sync(0xffffffffu, base, leader);
    if (sd == 0) return;
    uint32_t pos = offsets[key] + base + (uint32_t)__popc(peers & ((1u << lane) - 1));
    // scalars [0, n_main) belong to the resident bases, [n_main, n) to the call's extra points (their rows behind the table)
    size_t pidx = i < n_main ? (use_table ? (size_t)w * table_stride : 0) + sc.off[in_range ? j : 0] + i
                             : (size_t)main_count + (use_table ? (size_t)w * n_extra : 0) + (i - n_main);
    entries[pos] = (uint32_t)pidx | (sd < 0 ? 0x80000000u : 0u);
    pdl_trigger();
}

// ---------------------------------------------------------------------------------------------- accumulation
// Task t belongs to the bucket b with task_off[b] <= t < task_off[b+1]; the bucket's n_b sorted entries are cut into
// s_b = ceil(n_b / K) nearly equal parts, so no task crosses a bucket boundary and every thread sums <= K points with
// XYZZ mixed additions.  Single-task buckets are written directly, the others leave one partial per task.
template <class F>
__global__ void __launch_bounds__(128) k_accumulate(const affine_t* __restrict__ points, const uint32_t* __restrict__ entries,
                                                    const uint32_t* __restrict__ offsets, const uint32_t* __restrict__ task_off, uint32_t nb,
                                                    uint32_t K, const uint32_t* __restrict__ meta, const affine_t* __restrict__ extra,
                                                    uint32_t main_count, xyzz_t* buckets, xyzz_t* partials) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    // prologue: the plan (two kernels back) is complete when this grid launches
    const bool live = t < __ldg(meta + 1);
    // upper_bound(task_off[0..nb], t) - 1
    uint32_t lo = 0, hi = nb;  // invariant: task_off[lo] <= t < task_off[hi]
    while (live && hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (__ldg(task_off + mid) <= t) lo = mid; else hi = mid;
    }
    pdl_wait();                // the entries of k_scatter
    if (!live) return;
    const uint32_t b = lo;
    const uint32_t e0 = __ldg(offsets + b), nbk = __ldg(offsets + b + 1) - e0;
    const uint32_t sb = (nbk + K - 1) / K, sub = t - __ldg(task_off + b);
    const uint32_t base = nbk / sb, rem = nbk - base * sb;
    uint32_t i = e0 + sub * base + min(sub, rem);
    const uint32_t end = i + base + (sub < rem ? 1u : 0u);
    xyzz_t acc = xyzz_identity();
    // software pipeline: the gather of point i+1 is in flight while point i is added
    // (entries >= main_count address the call's extra points: h and U of an IPA round, ipa.rs:944,954)
    uint32_t e = __ldg(entries + i);
    uint32_t idx = e & 0x7fffffffu;
    affine_t p = load_affine_nc(idx < main_count ? points + idx : extra + (idx - main_count));
    for (; i < end; i++) {
        affine_t q = p;
        const uint32_t sign = e >> 31;
        if (i + 1 < end) {
            e = __ldg(entries + i + 1);
            idx = e & 0x7fffffffu;
            p = load_affine_nc(idx < main_count ? points + idx : extra + (idx - main_count));
        }
        if (sign) q.y = fe_neg<F>(q.y);
        acc = xyzz_madd<F>(acc, q);
    }
    store_xyzz(sb == 1 ? buckets + b : partials + t, acc);
    pdl_trigger();
}

// ---------------------------------------------------------------------------------------------- accumulation, TMA-staged gather
// The same accumulation with the gather moved to the bulk asynchronous copy engine (TMA, `cp.async.bulk`; UBLKCP in SASS): every lane
// asks the copy engine for its next 64-byte point, to be dropped in its own shared-memory slot and signalled on the warp's mbarrier,
// while it adds the current one — two stages per lane.  BASELINE's north star names this staging; on this kernel it is measured,
// not assumed (zk_ctx_set_option "msm_tma", tools/msm_tma_ab.py, profiles/r02_tma_ab.md): the kernel is bound by the FMA-heavy pipe
// (74.9 % busy, LSU 0.7 %), so taking the loads off the LSU path buys nothing and the shared-memory round trip costs a little.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t mbar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(mbar) : "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t mbar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(mbar), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}

template <class F>
__global__ void __launch_bounds__(128) k_accumulate_tma(const affine_t* __restrict__ points, const uint32_t* __restrict__ entries,
                                                        const uint32_t* __restrict__ offsets, const uint32_t* __restrict__ task_off, uint32_t nb,
                                                        uint32_t K, const uint32_t* __restrict__ meta, const affine_t* __restrict__ extra,
                                                        uint32_t main_count, xyzz_t* buckets, xyzz_t* partials) {
    __shared__ alignas(128) affine_t slots[2][128];
    __shared__ alignas(8) uint64_t bars[2][4];
    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t t = blockIdx.x * blockDim.x + tid;
    if (lane == 0) { mbar_init(smem_u32(&bars[0][warp]), 32); mbar_init(smem_u32(&bars[1][warp]), 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncwarp();
    const bool live = t < __ldg(meta + 1);
    uint32_t b = 0, sb = 1, i = 0, end = 0;
    if (live) {
        uint32_t lo = 0, hi = nb;
        while (hi - lo > 1) {
            uint32_t mid = (lo + hi) >> 1;
            if (__ldg(task_off + mid) <= t) lo = mid; else hi = mid;
        }
        b = lo;
        const uint32_t e0 = __ldg(offsets + b), nbk = __ldg(offsets + b + 1) - e0;
        sb = (nbk + K - 1) / K;
        const uint32_t sub = t - __ldg(task_off + b), base = nbk / sb, rem = nbk - base * sb;
        i = e0 + sub * base + min(sub, rem);
        end = i + base + (sub < rem ? 1u : 0u);
    }
    pdl_wait();                // the entries of k_scatter (the prologue above reads the plan only, see k_accumulate)
    const uint32_t steps = __reduce_max_sync(0xffffffffu, end - i);
    uint32_t sign[2] = {0, 0};
    auto issue = [&](uint32_t step) {
        const unsigned s = step & 1;
        const uint32_t bar = smem_u32(&bars[s][warp]);
        if (i + step < end) {
            const uint32_t e = __ldg(entries + i + step), idx = e & 0x7fffffffu;
            sign[s] = e >> 31;
            // the slot was read with ordinary loads two steps ago: order those (generic proxy) before the copy engine's write
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_arrive_expect_tx(bar, (uint32_t)sizeof(affine_t));
            bulk_copy_g2s(smem_u32(&slots[s][tid]), idx < main_count ? points + idx : extra + (idx - main_count), (uint32_t)sizeof(affine_t), bar);
        } else {
            mbar_arrive(bar);
        }
    };
    xyzz_t acc = xyzz_identity();
    if (steps) issue(0);
    for (uint32_t step = 0; step < steps; step++) {
        if (step + 1 < steps) issue(step + 1);
        mbar_wait(smem_u32(&bars[step & 1][warp]), (step >> 1) & 1);
        if (i + step < end) {
            const uint4* q4 = reinterpret_cast<const uint4*>(&slots[step & 1][tid]);
            affine_t q;
            uint4 v0 = q4[0], v1 = q4[1], v2 = q4[2], v3 = q4[3];
            q.x.v[0] = v0.x; q.x.v[1] = v0.y; q.x.v[2] = v0.z; q.x.v[3] = v0.w; q.x.v[4] = v1.x; q.x.v[5] = v1.y; q.x.v[6] = v1.z; q.x.v[7] = v1.w;
            q.y.v[0] = v2.x; q.y.v[1] = v2.y; q.y.v[2] = v2.z; q.y.v[3] = v2.w; q.y.v[4] = v3.x; q.y.v[5] = v3.y; q.y.v[6] = v3.z; q.y.v[7] = v3.w;
            if (sign[step & 1]) q.y = fe_neg<F>(q.y);
            acc = xyzz_madd<F>(acc, q);
        }
    }
    if (live) store_xyzz(sb == 1 ? buckets + b : partials + t, acc);
    pdl_trigger();
}

// Balanced first level of the per-bucket sums.  The task partials lie in bucket order; thread u sums the RUN of `run`
// consecutive partials [u*run, (u+1)*run) segment by segment (a segment = the part of one bucket inside the run) and writes each
// segment sum back at the segment's first index.  Every thread executes at most run-1 additions whatever the bucket sizes, so a
// warp never waits for its longest bucket.  k_bucket_finish_serial then adds, per bucket, the partial at the bucket's first index
// and those at the multiples of `run` inside it.  (Slots of single-task buckets hold no partial — k_accumulate wrote the bucket
// itself — and are segments of their own: read and written back, never mixed.)
template <class F>
__global__ void __launch_bounds__(128, 4) k_run_sum(const uint32_t* __restrict__ task_off, uint32_t nb, const uint32_t* __restrict__ meta, uint32_t run,
                                                 uint32_t smax, xyzz_t* partials) {
    // prologue: the plan's task_off and meta (three kernels back) are complete when this grid launches
    const uint32_t nt = meta[1];
    const uint64_t i0w = (uint64_t)(blockIdx.x * blockDim.x + threadIdx.x) * run;
    const uint32_t i0 = i0w < nt ? (uint32_t)i0w : nt, i1 = min(nt, i0 + run);
    // largest b with task_off[b] <= i0 (skips the empty buckets that share a start)
    uint32_t lo = 0, hi = nb;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(task_off + mid) <= i0) lo = mid; else hi = mid;
    }
    uint32_t b = lo, nxt = __ldg(task_off + b + 1), seg = i0;
    // giant buckets were summed by k_giant_finish: their slots are skipped (a thread wholly inside one does nothing)
    const bool giants_done = meta[2] <= MSM_MAX_GIANTS;
    bool skip = giants_done && nxt - __ldg(task_off + b) > smax;
    pdl_wait();                // the partials of k_accumulate, read after k_giant_finish has read them
    if (i0w >= nt || (skip && nxt >= i1)) return;
    xyzz_t acc = load_xyzz(partials + i0);
    bool dirty = false;
    for (uint32_t i = i0 + 1; i < i1; i++) {
        if (skip && i != nxt) continue;
        const xyzz_t v = load_xyzz(partials + i);
        if (i == nxt) {
            if (dirty) store_xyzz(partials + seg, acc);
            // the bucket that starts at i: usually the next one; behind a stretch of empty buckets, found by bisection
            b++; nxt = __ldg(task_off + b + 1);
            if (nxt <= i) {
                uint32_t l2 = b, h2 = nb;
                while (h2 - l2 > 1) {
                    const uint32_t mid = (l2 + h2) >> 1;
                    if (__ldg(task_off + mid) <= i) l2 = mid; else h2 = mid;
                }
                b = l2; nxt = __ldg(task_off + b + 1);
            }
            skip = giants_done && nxt - i > smax;
            seg = i; acc = v; dirty = false;
        } else {
            acc = xyzz_add<F, true>(acc, v);
            dirty = true;
        }
    }
    if (dirty) store_xyzz(partials + seg, acc);
    pdl_trigger();
}

// Thread-per-bucket finish pass, for MANY buckets with few partials each: with more buckets than resident quads the pass is
// throughput-bound and the quad-cooperative variant below only adds work.  run == 0: the bucket's partials are summed one by
// one; run > 0: k_run_sum ran first and the bucket's value is spread over its first slot and the multiples of `run` inside it.
template <class F>
__global__ void __launch_bounds__(128, 4) k_bucket_finish_serial(const uint32_t* __restrict__ offsets, const uint32_t* __restrict__ task_off, uint32_t nb,
                                                              uint32_t K, uint32_t smax, const uint32_t* __restrict__ meta, uint32_t run, xyzz_t* buckets,
                                                              const xyzz_t* __restrict__ partials) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    // prologue: the plan's offsets, task_off and meta (at least three kernels back) are complete when this grid launches
    uint32_t sb = 0, a = 0;
    if (b < nb) {
        const uint32_t nbk = __ldg(offsets + b + 1) - __ldg(offsets + b);
        sb = (nbk + K - 1) / K;
        if (sb > smax && meta[2] <= MSM_MAX_GIANTS) sb = 0;  // k_giant_finish
        a = __ldg(task_off + b);
    }
    pdl_wait();                                              // the partials of k_run_sum (or k_accumulate)
    if (sb < 2) return;                                      // 0: empty, 1: written by k_accumulate
    xyzz_t acc = load_xyzz(partials + a);
    if (run == 0) {
        for (uint32_t j = 1; j < sb; j++) acc = xyzz_add<F, true>(acc, load_xyzz(partials + a + j));
    } else {
        for (uint32_t k = (a / run + 1) * run; k < a + sb; k += run) acc = xyzz_add<F, true>(acc, load_xyzz(partials + k));
    }
    store_xyzz(buckets + b, acc);
    pdl_trigger();
}

// Buckets with 2 <= s_b <= smax tasks: a group of G = 2^log_g QUADS (quad.cuh) sums the bucket's partials — strided serial
// part, then a shuffle tree over the quads of the group.  One quad per bucket when buckets hold only a few partials.
template <class F>
__global__ void __launch_bounds__(128) k_bucket_finish(const uint32_t* __restrict__ offsets, const uint32_t* __restrict__ task_off, uint32_t nb,
                                                       uint32_t K, uint32_t smax, unsigned log_g, const uint32_t* __restrict__ meta,
                                                       xyzz_t* buckets, const xyzz_t* __restrict__ partials) {
    const uint32_t gq = (blockIdx.x * blockDim.x + threadIdx.x) >> 2;   // global quad
    const uint32_t G = 1u << log_g, b = gq >> log_g, gl = gq & (G - 1);
    uint32_t sb = 0, t0 = 0;
    if (b < nb) {
        const uint32_t nbk = __ldg(offsets + b + 1) - __ldg(offsets + b);
        sb = (nbk + K - 1) / K;
        t0 = __ldg(task_off + b);
        // giants are left to k_giant_finish — unless their list overflowed, then they are summed here (slow, correct)
        if (sb > smax && meta[2] <= MSM_MAX_GIANTS) sb = 0;
        if (sb < 2) sb = 0;
    }
    pdl_wait();                // the prologue above reads the plan only (at least two kernels back); the partials come from k_accumulate
    // warp-uniform trip count: every lane must take part in the quad additions' shuffles
    const unsigned my_trips = sb > gl ? (sb - gl + G - 1) / G : 0;
    const unsigned trips = __reduce_max_sync(0xffffffffu, my_trips);
    xyzz_t acc = xyzz_identity();
    for (unsigned k = 0; k < trips; k++) {
        const uint32_t j = gl + k * G;
        xyzz_t o = j < sb ? load_xyzz(partials + t0 + j) : xyzz_identity();
        acc = xyzz_add_quad<F>(acc, o);
    }
#pragma unroll 1
    for (unsigned d = G >> 1; d >= 1; d >>= 1) {
        xyzz_t o = shfl_down_xyzz(acc, 4 * d);
        if (gl >= d) o = xyzz_identity();
        acc = xyzz_add_quad<F>(acc, o);
    }
    if (gl == 0 && sb && (threadIdx.x & 3) == 0) store_xyzz(buckets + b, acc);
    pdl_trigger();
}

// ---------------------------------------------------------------------------------------------- bucket reduction
// sum_b (b+1) * B[b] = sum_t 2^t * T_t,  T_t = sum of B[b] over the b with bit t of (b+1) set.
// grid (blocks_per_bit, c, G); every CTA tree-sums its slice of one group's buckets for one bit.
constexpr unsigned TREE_THREADS = 256;              // 64 quads per CTA in the reduction kernels
constexpr unsigned TREE_QUADS = TREE_THREADS / 4;

// GIANT_SLICES CTAs per giant bucket: each sums a contiguous slice of the bucket's partial list (quads stride over it, then
// the block tree, quad.cuh); the last CTA to arrive (ticket counter) adds the slice sums and writes the bucket.
constexpr unsigned GIANT_SLICES = 16;
template <class F>
__global__ void __launch_bounds__(TREE_THREADS) k_giant_finish(const uint32_t* __restrict__ giants, const uint32_t* __restrict__ meta,
                                                               const uint32_t* __restrict__ offsets, const uint32_t* __restrict__ task_off, uint32_t K,
                                                               xyzz_t* buckets, const xyzz_t* __restrict__ partials, xyzz_t* slice_sums,
                                                               uint32_t* tickets) {
    extern __shared__ xyzz_t sm_tree[];
    __shared__ uint32_t ticket_s;
    pdl_wait();                // the partials of k_accumulate
    const uint32_t ng = meta[2];
    if (ng > MSM_MAX_GIANTS || blockIdx.x >= ng) return;  // overflow: k_bucket_finish took them
    const uint32_t b = giants[blockIdx.x];
    const uint32_t nbk = offsets[b + 1] - offsets[b], sb = (nbk + K - 1) / K, t0 = task_off[b];
    const uint32_t per = (sb + GIANT_SLICES - 1) / GIANT_SLICES;
    const uint32_t j_lo = blockIdx.y * per, j_hi = min(sb, j_lo + per);
    const unsigned qd = threadIdx.x >> 2, nq = blockDim.x >> 2;
    xyzz_t acc = xyzz_identity();
    for (uint32_t j0 = j_lo; j0 < j_hi; j0 += nq) {
        xyzz_t o = j0 + qd < j_hi ? load_xyzz(partials + t0 + j0 + qd) : xyzz_identity();
        acc = xyzz_add_quad<F>(acc, o);
    }
    acc = block_tree_sum_quad<F>(acc, sm_tree);
    xyzz_t* mine = slice_sums + (size_t)blockIdx.x * GIANT_SLICES;
    if (threadIdx.x == 0) {
        store_xyzz(mine + blockIdx.y, acc);
        __threadfence();
        ticket_s = atomicAdd(&tickets[blockIdx.x], 1u);
    }
    __syncthreads();
    if (ticket_s != GIANT_SLICES - 1) return;
    __threadfence();
    acc = qd < GIANT_SLICES ? load_xyzz(mine + qd) : xyzz_identity();
    acc = block_tree_sum_quad<F>(acc, sm_tree);
    if (threadIdx.x == 0) { store_xyzz(buckets + b, acc); tickets[blockIdx.x] = 0; }
    pdl_trigger();
}

// Two-level form of the same reduction (fewer additions, shorter dependency chains).  Split i = hi * W + lo, W = 2^w_lo:
//     sum_i i * B[i] = W * sum_hi hi * R[hi] + sum_lo lo * C[lo],   R[hi] = sum_lo B[hi W + lo],  C[lo] = sum_hi B[hi W + lo]
// k_gridsum: one CTA per row and per column of the (B/W + 1) x W bucket grid (row B/W holds the single bucket i = B);
// k_gridsum_final: one CTA per output bit: T_t = sum of C[lo] over bit t of lo (t < w_lo), of R[hi] over bit t - w_lo of hi
// (t >= w_lo).  Output layout and meaning are those of k_bitsum_final: c points per group, the MSM is sum_t 2^t T_t.
// About 2 B additions per group instead of (c - 1) B / 2.
template <class F>
__global__ void __launch_bounds__(128, 3) k_gridsum(const xyzz_t* __restrict__ buckets, uint32_t B, unsigned w_lo, xyzz_t* rc) {
    extern __shared__ xyzz_t sm_tree[];
    const uint32_t W = 1u << w_lo, nrows = (B >> w_lo) + 1;
    const unsigned g = blockIdx.z;
    const xyzz_t* bk = buckets + (size_t)g * B;
    const unsigned qd = threadIdx.x >> 2, nq = blockDim.x >> 2;
    const bool row = blockIdx.x < nrows;
    // a column holds B / W buckets — rows 0 .. B/W - 1, except column 0: rows 1 .. B/W (bucket 0 does not exist, bucket B closes
    // it) — so B / W trips cover every column: a power of two, no trip spent on the odd last row
    const uint32_t fixed = row ? blockIdx.x : blockIdx.x - nrows, count = row ? W : nrows - 1;
    const uint32_t shift = (!row && fixed == 0) ? 1u : 0u;
    xyzz_t acc = xyzz_identity();
    // The next trip's bucket is in flight while the current one is added (the additions are a dependent chain).  Each lane of the
    // quad fetches ONE coordinate (32 B) ahead — 8 registers instead of 32 — and the quad reassembles the point with shuffles.
    const unsigned lane = threadIdx.x & 31, base = lane & ~3u, coord = lane & 3;
    auto fetch = [&](uint32_t e) {
        fe part = fe_zero();
        if (e < count) {
            const uint32_t i = row ? fixed * W + e : (e + shift) * W + fixed;
            if (i >= 1 && i <= B) part = load_fe(reinterpret_cast<const fe*>(bk + (i - 1)) + coord);
        }
        return part;
    };
    pdl_wait();                // the buckets: k_plan, k_accumulate, k_giant_finish and the finish kernels all wrote some
    fe nxt = fetch(qd);
    for (uint32_t e0 = 0; e0 < count; e0 += nq) {
        xyzz_t o;
        o.X = shfl_fe(nxt, base); o.Y = shfl_fe(nxt, base + 1); o.ZZ = shfl_fe(nxt, base + 2); o.ZZZ = shfl_fe(nxt, base + 3);
        if (e0 + nq < count) nxt = fetch(e0 + nq + qd);
        acc = xyzz_add_quad<F>(acc, o);
    }
    acc = block_tree_sum_quad<F>(acc, sm_tree);
    if (threadIdx.x == 0) store_xyzz(rc + (size_t)g * (nrows + W) + blockIdx.x, acc);
    pdl_trigger();
}

template <class F>
__global__ void __launch_bounds__(TREE_THREADS) k_gridsum_final(const xyzz_t* __restrict__ rc, uint32_t B, unsigned w_lo, unsigned c, xyzz_t* out) {
    extern __shared__ xyzz_t sm_tree[];
    const uint32_t W = 1u << w_lo, nrows = (B >> w_lo) + 1;
    const unsigned t = blockIdx.x, g = blockIdx.y;
    const bool cols = t < w_lo;
    const xyzz_t* src = rc + (size_t)g * (nrows + W) + (cols ? nrows : 0);
    const uint32_t count = cols ? W : nrows;
    const unsigned bit = cols ? t : t - w_lo;
    const unsigned qd = threadIdx.x >> 2, nq = blockDim.x >> 2;
    xyzz_t acc = xyzz_identity();
    pdl_wait();                // the row / column sums of k_gridsum
    // the j-th index with `bit` set: e = (j >> bit) << (bit + 1) | 1 << bit | (j & (2^bit - 1))
    for (uint32_t j0 = 0;; j0 += nq) {
        const uint32_t first = ((j0 >> bit) << (bit + 1)) | (1u << bit) | (j0 & ((1u << bit) - 1));
        if (first >= count) break;     // uniform over the block
        const uint32_t j = j0 + qd, e = ((j >> bit) << (bit + 1)) | (1u << bit) | (j & ((1u << bit) - 1));
        xyzz_t o = e < count ? load_xyzz(src + e) : xyzz_identity();
        acc = xyzz_add_quad<F>(acc, o);
    }
    acc = block_tree_sum_quad<F>(acc, sm_tree);
    if (threadIdx.x == 0) store_xyzz(out + (size_t)g * c + t, acc);
}

// ---------------------------------------------------------------------------------------------- workspace
static void free_dev(void* p) { if (p) cudaFree(p); }

void msm_workspace_free(MsmWorkspace& ws) {
    free_dev(ws.d_digits); free_dev(ws.d_entries); free_dev(ws.d_partials);
    free_dev(ws.d_counts); free_dev(ws.d_offsets); free_dev(ws.d_task_off); free_dev(ws.d_buckets); free_dev(ws.d_chain); free_dev(ws.d_chain_flag);
    free_dev(ws.d_bitsums); free_dev(ws.d_meta); free_dev(ws.d_giants); free_dev(ws.d_giant_slices); free_dev(ws.d_giant_tickets);
    if (ws.h_bitsums) cudaFreeHost(ws.h_bitsums);
    for (auto& e : ws.ev) if (e) cudaEventDestroy(e);
    ws = MsmWorkspace();
}

// a kernel launch on `st`; pdl: programmatic stream serialization with the kernel before it (see "launch chain" above)
template <class... KArgs, class... Args>
static cudaError_t launch(bool pdl, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cfg.attrs = &attr; cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

static unsigned pow2_ceil_log(uint64_t x) {
    unsigned l = 0;
    while (((uint64_t)1 << l) < x) l++;
    return l;
}

template <class F, class FS>
int msm_run(const MsmBases& b, const size_t* offs, size_t n_main, const fe* const* d_scalars, unsigned k, bool scalars_mont, unsigned c,
            MsmWorkspace& ws, cudaStream_t st, MsmResultShape* shape, unsigned* launches, const affine_t* d_extra, size_t n_extra) {
    const size_t n = n_main + n_extra;                // scalars per MSM
    if (n_extra && !d_extra) { zk_set_error("msm: extra points missing"); return ZK_ERR_INVALID; }
    for (unsigned j = 0; j < k && j < MSM_MAX_BATCH; j++)
        if (offs[j] > b.n || n_main > b.n - offs[j]) { zk_set_error("msm: slice [%zu, %zu) outside the %zu resident bases", offs[j], offs[j] + n_main, b.n); return ZK_ERR_INVALID; }
    if (k == 0 || k > MSM_MAX_BATCH) { zk_set_error("msm: batch of %u outside [1, %u]", k, MSM_MAX_BATCH); return ZK_ERR_INVALID; }
    shape->c = 0; shape->groups = 0; shape->batch = k;
    if (n == 0) return ZK_OK;
    const bool use_table = b.c != 0;
    if (use_table) c = b.c;
    else if (c == 0) c = (unsigned)msm_default_window(n, false);
    if (c < 2 || c > MSM_MAX_WINDOW_BITS) { zk_set_error("msm: window bits %u outside [2, %u]", c, MSM_MAX_WINDOW_BITS); return ZK_ERR_INVALID; }
    const unsigned nwin = msm_num_windows(c);
    const unsigned gpm = use_table ? 1 : nwin;        // bucket groups per MSM
    const unsigned G = k * gpm;                       // bucket groups of the batch
    const uint32_t B = 1u << (c - 1);                 // buckets per group
    const size_t NB = (size_t)G * B;
    const size_t Mmax = n * nwin * (size_t)k;
    const size_t main_count = b.n * (size_t)std::max(1u, b.nwin);   // table entries; the extra points' rows are addressed behind them
    if (Mmax >= 0x7fffffffull || NB >= 0x7fffffffull || main_count + n_extra * nwin >= 0x7fffffffull) {
        zk_set_error("msm: %zu x %u x %u entries exceed the 31-bit index space", n, nwin, k);
        return ZK_ERR_INVALID;
    }
    // Entries per accumulation task: the accumulate kernel keeps `capacity` threads resident (4 CTAs of 128 per SM at
    // <= 128 registers); K is chosen so that the tasks fill a whole number of waves (a 1.02-wave grid costs two waves).
    // Short tasks keep the lanes of a warp balanced (a bucket of n_b entries is cut into ceil(n_b / K) equal parts: lengths lie
    // in (K s / (s + 1), K]) — measured on B200: one 28-entry wave is 1.5x slower than two 8-entry waves for the same additions.
    const size_t capacity = (size_t)ws.sm_count * (ws.wave_threads ? ws.wave_threads : 512);
    const size_t resident_quads = (size_t)ws.sm_count * TREE_QUADS;
    const bool many_buckets = NB > resident_quads;    // many small buckets: throughput regime (see k_bucket_finish_serial)
    const bool serial_finish = many_buckets;
    uint32_t K = ws.chunk;
    if (K == 0) {
        // (1) lane balance: a bucket of n_b entries is cut into ceil(n_b / K) equal tasks, so task lengths lie in (K s / (s + 1), K];
        //     with s >= 8 tasks per average bucket the lanes of a warp differ by ~10% (measured on B200, 2^16 points, window 15: tasks
        //     of 28 entries run the same additions 1.5x slower than tasks of 8), whatever the batch size;
        // (2) small inputs: never fewer tasks than threads the machine holds at once.
        const size_t n_avg = std::max<size_t>(1, Mmax / NB);
        // (measured at 2^16 points, windows 15 / 16, gpurun_out/msm_tune.json: K = 6..8 beats 4 by 1-3 %: fewer partials for the finish pass)
        size_t k_bal = many_buckets ? std::min<size_t>(64, std::max<size_t>(6, n_avg / 8)) : 64;
        const size_t slack = std::min<size_t>(NB / 2, capacity / 4);     // sum_b ceil(n_b/K) ~ M/K + (non-empty buckets)/2
        const size_t k_cap = std::max<size_t>(4, (Mmax + capacity - slack - 1) / (capacity - slack));
        K = (uint32_t)std::min(k_bal, k_cap);
    }
    const size_t NTmax = Mmax / K + NB + 1;           // sum_b ceil(n_b / K) <= M / K + (number of non-empty buckets)
    // lanes per bucket in the finish pass: ~a quarter of the expected partials per bucket
    const uint64_t s_avg = Mmax / ((uint64_t)K * NB) + 1;
    unsigned log_g = pow2_ceil_log((s_avg + 7) / 8);   // quads per bucket in the finish pass
    if (log_g > 3) log_g = 3;
    const uint32_t smax = 32u << log_g;               // more partials than this: the bucket is "giant"
    const uint32_t run = 4;                           // k_run_sum: consecutive partials summed per thread
    const unsigned w_lo = (c - 1) / 2;
    const uint32_t W = 1u << w_lo, nrows = (B >> w_lo) + 1;
    const size_t ntiles = (NB + PLAN_TILE - 1) / PLAN_TILE;

    static_assert(sizeof(xyzz_t) == 128 && sizeof(affine_t) == 64 && sizeof(fe) == 32, "layout");
    // scratch, grouped by what sizes it: the entry list (k * n * nwin), the bucket array (G * B), the slice sums (G * c)
    {
        const size_t need_entries = Mmax * sizeof(uint32_t), need_partials = NTmax * sizeof(xyzz_t);
        if (ws.cap_entries < need_entries) {
            free_dev(ws.d_digits); free_dev(ws.d_entries);
            ws.d_digits = nullptr; ws.d_entries = nullptr; ws.cap_entries = 0;
            ZK_CUDA(cudaMalloc(&ws.d_digits, Mmax * sizeof(int32_t)));
            ZK_CUDA(cudaMalloc(&ws.d_entries, need_entries));
            ws.cap_entries = need_entries;
        }
        if (ws.cap_partials < need_partials) {
            free_dev(ws.d_partials);
            ws.d_partials = nullptr; ws.cap_partials = 0;
            ZK_CUDA(cudaMalloc(&ws.d_partials, need_partials));
            ws.cap_partials = need_partials;
        }
        if (ws.cap_buckets < NB) {
            free_dev(ws.d_counts); free_dev(ws.d_offsets); free_dev(ws.d_task_off); free_dev(ws.d_buckets); free_dev(ws.d_chain); free_dev(ws.d_chain_flag);
            ws.d_counts = ws.d_offsets = ws.d_task_off = ws.d_chain_flag = nullptr; ws.d_chain = nullptr; ws.d_buckets = nullptr; ws.cap_buckets = 0;
            ZK_CUDA(cudaMalloc(&ws.d_counts, NB * sizeof(uint32_t)));
            ZK_CUDA(cudaMemsetAsync(ws.d_counts, 0, NB * sizeof(uint32_t), st));   // then kept zero by k_scatter
            ZK_CUDA(cudaMalloc(&ws.d_offsets, (NB + 1) * sizeof(uint32_t)));
            ZK_CUDA(cudaMalloc(&ws.d_task_off, (NB + 1) * sizeof(uint32_t)));
            ZK_CUDA(cudaMalloc(&ws.d_buckets, NB * sizeof(xyzz_t)));
            ZK_CUDA(cudaMalloc(&ws.d_chain, ntiles * sizeof(uint64_t)));
            ZK_CUDA(cudaMalloc(&ws.d_chain_flag, ntiles * sizeof(uint32_t)));
            ZK_CUDA(cudaMemsetAsync(ws.d_chain_flag, 0, ntiles * sizeof(uint32_t), st));
            ws.epoch = 0;
            ws.cap_buckets = NB;
        }
        const size_t need_bits = (size_t)G * (nrows + W) + (size_t)G * c;
        if (ws.cap_bits < need_bits) {
            free_dev(ws.d_bitsums);
            ws.d_bitsums = nullptr; ws.cap_bits = 0;
            ZK_CUDA(cudaMalloc(&ws.d_bitsums, need_bits * sizeof(xyzz_t)));
            ws.cap_bits = need_bits;
        }
        if (ws.cap_hbits < (size_t)G * c) {   // sized by G*c alone: few wide groups and many narrow ones differ
            if (ws.defer_sync) ZK_CUDA(cudaStreamSynchronize(st));   // an earlier deferred result may still be in flight
            if (ws.h_bitsums) cudaFreeHost(ws.h_bitsums);
            ws.h_bitsums = nullptr; ws.cap_hbits = 0;
            ZK_CUDA(cudaMallocHost(&ws.h_bitsums, 2 * (size_t)G * c * sizeof(xyzz_t)));
            ws.cap_hbits = (size_t)G * c;
        }
        if (!ws.d_meta) {
            ZK_CUDA(cudaMalloc(&ws.d_meta, 8 * sizeof(uint32_t)));
            ZK_CUDA(cudaMalloc(&ws.d_giants, MSM_MAX_GIANTS * sizeof(uint32_t)));
            ZK_CUDA(cudaMalloc(&ws.d_giant_slices, (size_t)MSM_MAX_GIANTS * GIANT_SLICES * sizeof(xyzz_t)));
            ZK_CUDA(cudaMalloc(&ws.d_giant_tickets, MSM_MAX_GIANTS * sizeof(uint32_t)));
            ZK_CUDA(cudaMemsetAsync(ws.d_giant_tickets, 0, MSM_MAX_GIANTS * sizeof(uint32_t), st));
        }
    }
    unsigned nl = 0;
    if (ws.profile && !ws.ev[0])
        for (int s = 0; s <= MSM_ST_COUNT; s++) ZK_CUDA(cudaEventCreate(&ws.ev[s]));
#define STAGE_MARK(s) do { if (ws.profile) ZK_CUDA(cudaEventRecord(ws.ev[s], st)); } while (0)

    MsmScalarSet sc{};
    for (unsigned j = 0; j < k; j++) { sc.p[j] = d_scalars[j]; sc.off[j] = (uint32_t)offs[j]; }
    const uint32_t epoch = ++ws.epoch;
    if (!ws.pdl) {
        // the launch shell this pipeline had before the PDL chain, kept for A/B (option msm_pdl = 0): both memsets are redundant
        ZK_CUDA(cudaMemsetAsync(ws.d_counts, 0, NB * sizeof(uint32_t), st));
        ZK_CUDA(cudaMemsetAsync(ws.d_buckets, 0, NB * sizeof(xyzz_t), st));
    }
    // kernels 2.. wait for their predecessor in-kernel; profile mode launches plainly so that the stage events bracket one kernel each
    const bool pdl = ws.pdl && !ws.profile;
    STAGE_MARK(0);
    // 1. digits + histogram (an ordinary launch: it follows everything before it on the stream, the previous call included)
    k_recode<FS><<<dim3((unsigned)((n + 127) / 128), k), 128, 0, st>>>(sc, scalars_mont ? 1 : 0, n, c, nwin, gpm, use_table ? 0 : 1, ws.d_digits,
                                                                        ws.d_counts, ws.d_meta);
    STAGE_MARK(1);
    // 2. plan: bucket offsets, task offsets, giant list, identity of the empty buckets
    ZK_CUDA(launch(pdl, k_plan, dim3((unsigned)ntiles), dim3(1024), 0, st, ws.d_counts, ws.d_offsets, ws.d_task_off, (uint32_t)NB, K, smax, ws.d_meta,
                   ws.d_giants, ws.d_chain, ws.d_chain_flag, epoch, ws.d_buckets));
    STAGE_MARK(2);
    // 3. scatter (counting sort by bucket)
    ZK_CUDA(launch(pdl, k_scatter, dim3((unsigned)((Mmax + 255) / 256)), dim3(256), 0, st, ws.d_digits, n, c, nwin, k, gpm, use_table ? 0 : 1, sc, b.n,
                   use_table ? 1 : 0, n_main, n_extra, (uint32_t)main_count, ws.d_offsets, ws.d_counts, ws.d_entries));
    STAGE_MARK(3);
    // 4. accumulation: one task per <= K sorted entries of one bucket
    ZK_CUDA(launch(pdl, ws.tma_gather ? k_accumulate_tma<F> : k_accumulate<F>, dim3((unsigned)((NTmax + 127) / 128)), dim3(128), 0, st, b.d_points,
                   ws.d_entries, ws.d_offsets, ws.d_task_off, (uint32_t)NB, K, ws.d_meta, d_extra, (uint32_t)main_count, ws.d_buckets, ws.d_partials));
    STAGE_MARK(4);
    // 5. per-bucket sums of the task partials (+ giants)
    // giants first: k_giant_finish reads the untouched partial lists, k_run_sum then rewrites partials in place
    ZK_CUDA(launch(pdl, k_giant_finish<F>, dim3(64, GIANT_SLICES), dim3(TREE_THREADS), TREE_QUADS * sizeof(xyzz_t), st, ws.d_giants, ws.d_meta,
                   ws.d_offsets, ws.d_task_off, K, ws.d_buckets, ws.d_partials, ws.d_giant_slices, ws.d_giant_tickets));
    if (serial_finish) {
        const size_t threads = (NTmax + run - 1) / run;
        ZK_CUDA(launch(pdl, k_run_sum<F>, dim3((unsigned)((threads + 127) / 128)), dim3(128), 0, st, ws.d_task_off, (uint32_t)NB, ws.d_meta, run, smax,
                       ws.d_partials));
        nl += 1;
        ZK_CUDA(launch(pdl, k_bucket_finish_serial<F>, dim3((unsigned)((NB + 127) / 128)), dim3(128), 0, st, ws.d_offsets, ws.d_task_off, (uint32_t)NB, K,
                       smax, ws.d_meta, run, ws.d_buckets, ws.d_partials));
    } else {
        ZK_CUDA(launch(pdl, k_bucket_finish<F>, dim3((unsigned)(((NB << (log_g + 2)) + 127) / 128)), dim3(128), 0, st, ws.d_offsets, ws.d_task_off,
                       (uint32_t)NB, K, smax, log_g, ws.d_meta, ws.d_buckets, ws.d_partials));
    }
    STAGE_MARK(5);
    // 6. two-level bucket reduction: row / column sums of the bucket grid, then their bit slices
    xyzz_t* d_rc = ws.d_bitsums;
    xyzz_t* d_T = ws.d_bitsums + (size_t)G * (nrows + W);
    {
        // a quad per 1-4 elements of a row / column, but never more CTAs x threads than are resident at once (384 threads per
        // SM at the kernel's register budget), so that the whole grid of a single MSM — 385 CTAs at window 16 — runs as one wave
        unsigned gt = 128;                          // k_gridsum is built for 3 CTAs of 128 threads per SM (<= 168 registers)
        while (gt > 32 && (gt / 4 >= 2 * std::max(W, nrows) || (size_t)G * (nrows + W) * gt > (size_t)ws.sm_count * 384)) gt /= 2;
        ZK_CUDA(launch(pdl, k_gridsum<F>, dim3(nrows + W, 1, G), dim3(gt), (gt / 4) * sizeof(xyzz_t), st, ws.d_buckets, B, w_lo, d_rc));
        unsigned ft = TREE_THREADS;                 // half of the elements carry a given bit
        while (ft > 32 && ft / 4 >= std::max(W, nrows)) ft /= 2;
        ZK_CUDA(launch(pdl, k_gridsum_final<F>, dim3(c, G), dim3(ft), (ft / 4) * sizeof(xyzz_t), st, d_rc, B, w_lo, c, d_T));
    }
    nl += 8;
    STAGE_MARK(6);
    ZK_CUDA(cudaGetLastError());
    shape->c = c; shape->groups = gpm;
    if (launches) *launches += nl;
    if (ws.d_T_out) {
        if ((size_t)G * c > ws.d_T_cap) { zk_set_error("msm: %u slice sums do not fit the caller's buffer of %zu points", G * c, ws.d_T_cap); return ZK_ERR_INVALID; }
        ZK_CUDA(cudaMemcpyAsync(ws.d_T_out, d_T, (size_t)G * c * sizeof(xyzz_t), cudaMemcpyDeviceToDevice, st));
        return ZK_OK;
    }
    ZK_CUDA(cudaMemcpyAsync(ws.h_bitsums + (size_t)(ws.h_slot & 1) * ws.cap_hbits, d_T, (size_t)G * c * sizeof(xyzz_t), cudaMemcpyDeviceToHost, st));
    if (ws.defer_sync) return ZK_OK;
    ZK_CUDA(cudaStreamSynchronize(st));
    if (ws.profile)
        for (int s = 0; s < MSM_ST_COUNT; s++) ZK_CUDA(cudaEventElapsedTime(&ws.stage_ms[s], ws.ev[s], ws.ev[s + 1]));
#undef STAGE_MARK
    // the O(c) serial tail (c doublings per group) is finished on the host from ws.h_bitsums (api.cu: msm_finish)
    return ZK_OK;
}

// one warp per output point: its 8 quads stride over the ranks, then a shuffle tree
template <class F> __global__ void __launch_bounds__(32) k_sum_partials(const xyzz_t* __restrict__ all, uint32_t world, uint32_t count, xyzz_t* out) {
    const unsigned i = blockIdx.x, qd = threadIdx.x >> 2;
    xyzz_t acc = xyzz_identity();
    for (uint32_t r0 = 0; r0 < world; r0 += 8) {
        const uint32_t r = r0 + qd;
        xyzz_t o = r < world ? load_xyzz(all + (size_t)r * count + i) : xyzz_identity();
        acc = xyzz_add_quad<F>(acc, o);
    }
#pragma unroll 1
    for (unsigned d = 4; d >= 1; d >>= 1) {
        xyzz_t o = shfl_down_xyzz(acc, 4 * d);
        if (qd >= d) o = xyzz_identity();
        acc = xyzz_add_quad<F>(acc, o);
    }
    if (threadIdx.x == 0) store_xyzz(out + i, acc);
}
template <class F> int msm_sum_partials(const xyzz_t* d_all, size_t world, size_t count, xyzz_t* d_out, cudaStream_t st) {
    if (count) k_sum_partials<F><<<(unsigned)count, 32, 0, st>>>(d_all, (uint32_t)world, (uint32_t)count, d_out);
    ZK_CUDA(cudaGetLastError());
    return ZK_OK;
}
template int msm_sum_partials<FpParams>(const xyzz_t*, size_t, size_t, xyzz_t*, cudaStream_t);
template int msm_sum_partials<FqParams>(const xyzz_t*, size_t, size_t, xyzz_t*, cudaStream_t);

#define INST(F, FS)                                                                                                             \
    template int msm_bases_create<F>(MsmBases&, const affine_t*, bool, size_t, unsigned, cudaStream_t);                          \
    template int msm_run<F, FS>(const MsmBases&, const size_t*, size_t, const fe* const*, unsigned, bool, unsigned, MsmWorkspace&, cudaStream_t, MsmResultShape*, unsigned*, \
                                const affine_t*, size_t);
INST(FpParams, FqParams)  // Pallas: coordinates Fp, scalars Fq
INST(FqParams, FpParams)  // Vesta:  coordinates Fq, scalars Fp
#undef INST

}  // namespace zkb
