// api.cu — the extern "C" boundary (include/zkb200.h): contexts, resident bases, MSM, NTT, diagnostics.
#include <cstdarg>
#include <cstring>
#include <map>
#include <mutex>
#include <vector>

#include "../../include/zkb200.h"
#include "ctx.hpp"
#include "host_field.hpp"
#include "msm.cuh"
#include "ntt.cuh"
#include "quad.cuh"

namespace zkb {

template <class F> int points_decompress(const uint8_t* d_in, affine_t* d_out, size_t n, unsigned* d_bad, cudaStream_t st);   // decompress.cu
template <class F> int points_from_uncompressed(const uint8_t* d_in, affine_t* d_out, size_t n, unsigned* d_bad, cudaStream_t st);
template <class F> int points_compress(const affine_t* d_in, uint8_t* d_out, size_t n, cudaStream_t st);
template <class F> int points_synthetic(affine_t* d_out, size_t n, uint64_t seed, cudaStream_t st);

static thread_local char g_err[512] = "";
void zk_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

// ---------------------------------------------------------------------------------------------- host tail of the MSM
template <class HP> static host::hxyzz msm_finish_t(const xyzz_t* T, unsigned c, unsigned G) {
    using namespace host;
    static_assert(sizeof(hxyzz) == sizeof(xyzz_t), "layout");
    hxyzz total = identity();
    for (int g = (int)G - 1; g >= 0; g--) {
        if (g != (int)G - 1)
            for (unsigned k = 0; k < c; k++) total = pdbl<HP>(total);
        hxyzz acc = identity();
        for (int t = (int)c - 1; t >= 0; t--) {
            hxyzz tt;
            memcpy(&tt, T + (size_t)g * c + t, sizeof tt);
            acc = padd<HP>(pdbl<HP>(acc), tt);
        }
        total = padd<HP>(total, acc);
    }
    return total;
}

static void xyzz_to_jac_out(int curve, const host::hxyzz& p, uint64_t out[12]) {
    host::hjac j = curve == ZK_PALLAS ? host::to_jacobian<host::HFp>(p) : host::to_jacobian<host::HFq>(p);
    memcpy(out, &j, sizeof j);
}

int ctx_msm_many(zk_ctx* ctx, const zk_bases* bases, size_t off, size_t n, const fe* const* d_scalars, size_t k, int mont, int window_bits,
                 uint64_t* out_xyz, const affine_t* d_extra, size_t n_extra) {
    std::vector<size_t> offs(k, off);
    return ctx_msm_many_offs(ctx, bases, offs.data(), n, d_scalars, k, mont, window_bits, out_xyz, d_extra, n_extra);
}

int ctx_msm_many_offs(zk_ctx* ctx, const zk_bases* bases, const size_t* offs, size_t n, const fe* const* d_scalars, size_t k, int mont, int window_bits,
                      uint64_t* out_xyz, const affine_t* d_extra, size_t n_extra) {
    if (window_bits < 0 || window_bits > (int)MSM_MAX_WINDOW_BITS) { zk_set_error("msm: window_bits %d outside [0, %u]", window_bits, MSM_MAX_WINDOW_BITS); return ZK_ERR_INVALID; }
    const bool pallas = bases->b.curve == ZK_PALLAS;
    // MSMs per pipeline: the context's limit, and no more than keeps the sorted entry list below 2^28 entries (1 GiB of scratch)
    const unsigned c_eff = bases->b.c ? bases->b.c : (window_bits ? (unsigned)window_bits : (unsigned)msm_default_window(n, false));
    const size_t per_msm = std::max<size_t>(1, (n + n_extra) * msm_num_windows(std::max(2u, c_eff)));
    size_t fuse = std::min<size_t>((size_t)std::max(1, ctx->batch), std::max<size_t>(1, ((size_t)1 << 28) / per_msm));
    if (ctx->profile) fuse = 1;   // stage times are those of ONE MSM (zk_ctx_last_stage_ms)
    for (size_t j0 = 0; j0 < k; j0 += fuse) {
        const unsigned cnt = (unsigned)std::min(fuse, k - j0);
        MsmResultShape shape;
        unsigned nl = 0;
        ctx->ws.h_slot = 0;
        int rc = pallas ? msm_run<FpParams, FqParams>(bases->b, offs + j0, n, d_scalars + j0, cnt, mont != 0, (unsigned)window_bits, ctx->ws, ctx->stream, &shape, &nl,
                                                      d_extra, n_extra)
                        : msm_run<FqParams, FpParams>(bases->b, offs + j0, n, d_scalars + j0, cnt, mont != 0, (unsigned)window_bits, ctx->ws, ctx->stream, &shape, &nl,
                                                      d_extra, n_extra);
        if (rc) return rc;
        ctx->launches += nl;
        for (unsigned j = 0; j < cnt; j++) {
            host::hxyzz r = host::identity();
            if (shape.groups) {
                const xyzz_t* h = ctx->ws.h_bitsums + (size_t)j * shape.groups * shape.c;
                r = pallas ? msm_finish_t<host::HFp>(h, shape.c, shape.groups) : msm_finish_t<host::HFq>(h, shape.c, shape.groups);
            }
            xyzz_to_jac_out(bases->b.curve, r, out_xyz + 12 * (j0 + j));
        }
    }
    return ZK_OK;
}

int ctx_msm_device(zk_ctx* ctx, const zk_bases* bases, size_t off, size_t n, const fe* d_scalars, int mont, int window_bits,
                   uint64_t out_xyz[12]) {
    return ctx_msm_many(ctx, bases, off, n, &d_scalars, 1, mont, window_bits, out_xyz);
}

static int ctx_side_streams_init(zk_ctx* ctx) {
    if (ctx->ev_fork) return ZK_OK;
    for (int l = 0; l < zk_ctx::SIDE_STREAMS; l++) ZK_CUDA(cudaStreamCreateWithFlags(&ctx->side[l], cudaStreamNonBlocking));
    ZK_CUDA(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    return ZK_OK;
}

int ctx_ensure(void** p, size_t* cap, size_t bytes) {
    if (*cap >= bytes) return ZK_OK;
    if (*p) cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    ZK_CUDA(cudaMalloc(p, bytes));
    *cap = bytes;
    return ZK_OK;
}

static int ctx_ntt_tables(zk_ctx* lane, int field, unsigned log_n, bool inverse, const fe** small, const NttTables** tabs) {
    zk_ctx* ctx = ctx_root(lane);                      // one cache per pool; entries are immutable once built
    std::lock_guard<std::mutex> tl(ctx->tab_mu);
    fe*& sm = ctx->ntt_small[field][inverse ? 1 : 0];
    if (!sm) {
        ZK_CUDA(cudaMalloc(&sm, 512 * sizeof(fe)));
        int rc = field == ZK_FP ? ntt_build_small_table<FpParams>(sm, inverse, lane->stream) : ntt_build_small_table<FqParams>(sm, inverse, lane->stream);
        if (rc) return rc;
        lane->launches += 2;
    }
    unsigned key = (unsigned)field | (inverse ? 2u : 0u) | (log_n << 2);
    auto it = ctx->ntt_tables.find(key);
    if (it == ctx->ntt_tables.end()) {
        NttTables t;
        int rc = field == ZK_FP ? ntt_build_tables<FpParams>(t, log_n, inverse, lane->stream) : ntt_build_tables<FqParams>(t, log_n, inverse, lane->stream);
        if (rc) return rc;
        lane->launches += t.full ? 8 : 7;
        it = ctx->ntt_tables.emplace(key, t).first;
    }
    *small = sm;
    *tabs = &it->second;
    return ZK_OK;
}

// the unscaled twiddle tables of a forward / inverse transform (pointwise evaluators take x_i = w^i from them)
int ctx_ntt_table_ptrs(zk_ctx* ctx, int field, unsigned log_n, bool inverse, const fe** ulo, const fe** mid, const fe** hi2) {
    const fe* small;
    const NttTables* tabs;
    int rc = ctx_ntt_tables(ctx, field, log_n, inverse, &small, &tabs);
    if (rc) return rc;
    *ulo = tabs->ulo; *mid = tabs->mid; *hi2 = tabs->hi2;
    return ZK_OK;
}

// Transform of `batch` polynomials: polynomial b is read from d_in + b * in_bs (its first in_len elements) and written to
// d_out + b * 2^log_n; d_in == d_out (in_bs = 2^log_n) is the in-place form.
int ctx_ntt_device_oop(zk_ctx* ctx, int field, const fe* d_in, size_t in_bs, fe* d_out, unsigned log_n, size_t batch, size_t in_len, int inverse, int coset) {
    if (field != ZK_FP && field != ZK_FQ) { zk_set_error("ntt: unknown field_id %d", field); return ZK_ERR_INVALID; }
    if (log_n > NTT_MAX_LOG_N) { zk_set_error("ntt: log_n %u > %u not supported", log_n, NTT_MAX_LOG_N); return ZK_ERR_INVALID; }
    const fe* small;
    const NttTables* tabs;
    const NttTables* inner = nullptr;
    int rc = ctx_ntt_tables(ctx, field, log_n, inverse != 0, &small, &tabs);
    if (rc) return rc;
    if (const unsigned log_inner = ntt_inner_log(log_n)) {
        const fe* small2;
        rc = ctx_ntt_tables(ctx, field, log_inner, inverse != 0, &small2, &inner);
        if (rc) return rc;
    }
    size_t bytes = ((size_t)batch << log_n) * sizeof(fe);
    fe* tmp = nullptr;
    if (log_n > NTT_MAX_LOG_SUB) {
        rc = ctx_ensure((void**)&ctx->d_ntt_tmp, &ctx->cap_ntt_tmp, bytes);
        if (rc) return rc;
        tmp = ctx->d_ntt_tmp;
    }
    unsigned nl = 0;
    if (ctx->profile) {
        if (!ctx->ev_ntt[0]) { ZK_CUDA(cudaEventCreate(&ctx->ev_ntt[0])); ZK_CUDA(cudaEventCreate(&ctx->ev_ntt[1])); }
        ZK_CUDA(cudaEventRecord(ctx->ev_ntt[0], ctx->stream));
    }
    rc = field == ZK_FP ? ntt_run<FpParams>(d_in, in_bs, d_out, tmp, small, *tabs, inner, log_n, batch, in_len, inverse != 0, coset != 0, ctx->stream, &nl)
                        : ntt_run<FqParams>(d_in, in_bs, d_out, tmp, small, *tabs, inner, log_n, batch, in_len, inverse != 0, coset != 0, ctx->stream, &nl);
    ctx->launches += nl;
    if (rc == ZK_OK && ctx->profile) {
        ZK_CUDA(cudaEventRecord(ctx->ev_ntt[1], ctx->stream));
        ZK_CUDA(cudaEventSynchronize(ctx->ev_ntt[1]));
        ZK_CUDA(cudaEventElapsedTime(&ctx->ntt_ms, ctx->ev_ntt[0], ctx->ev_ntt[1]));
    }
    return rc;
}

int ctx_ntt_device(zk_ctx* ctx, int field, fe* d_data, unsigned log_n, size_t batch, size_t in_len, int inverse, int coset) {
    return ctx_ntt_device_oop(ctx, field, d_data, (size_t)1 << (log_n > 62 ? 0 : log_n), d_data, log_n, batch, in_len, inverse, coset);
}

// ---------------------------------------------------------------------------------------------- lanes
static int ctx_init_lane(zk_ctx* c, int device_id) {
    c->device = device_id;
    cudaError_t se = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
    if (se != cudaSuccess) { zk_set_error("cudaStreamCreate: %s", cudaGetErrorString(se)); return ZK_ERR_CUDA; }
    c->stream = c->own_stream;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device_id) == cudaSuccess) c->ws.sm_count = prop.multiProcessorCount;
    return ZK_OK;
}

int ctx_acquire_lane(zk_ctx* ctx, LaneLock& out) {
    ctx = ctx_root(ctx);
    const bool pinned = ctx->stream != ctx->own_stream || ctx->profile || ctx->n_lanes <= 1;
    if (pinned) {
        out.lane = ctx;
        out.lk = std::unique_lock<std::mutex>(ctx->mu);
        return ZK_OK;
    }
    std::vector<zk_ctx*> lanes;
    unsigned start;
    {
        std::lock_guard<std::mutex> pl(ctx->pool_mu);
        while ((int)ctx->children.size() + 1 < ctx->n_lanes) {
            zk_ctx* c = new zk_ctx();
            c->parent = ctx;
            if (cudaSetDevice(ctx->device) != cudaSuccess || ctx_init_lane(c, ctx->device) != ZK_OK) { delete c; break; }
            c->batch = ctx->batch; c->ws.chunk = ctx->ws.chunk; c->ws.wave_threads = ctx->ws.wave_threads; c->ws.tma_gather = ctx->ws.tma_gather;
            c->ws.pdl = ctx->ws.pdl;
            ctx->children.push_back(c);
        }
        lanes.push_back(ctx);
        lanes.insert(lanes.end(), ctx->children.begin(), ctx->children.end());
        start = ctx->rr++;
    }
    // the primary lane first, then the children in order: a single-threaded caller always lands on the same (warm) lane, only
    // contention spills over; when every lane is busy the waiters spread round-robin
    for (size_t k = 0; k < lanes.size() && k < (size_t)ctx->n_lanes; k++) {
        zk_ctx* l = lanes[k];
        std::unique_lock<std::mutex> lk(l->mu, std::try_to_lock);
        if (lk.owns_lock()) { out.lane = l; out.lk = std::move(lk); return ZK_OK; }
    }
    zk_ctx* l = lanes[start % std::min<size_t>(lanes.size(), (size_t)ctx->n_lanes)];
    out.lane = l;
    out.lk = std::unique_lock<std::mutex>(l->mu);
    return ZK_OK;
}

// ---------------------------------------------------------------------------------------------- diagnostics kernels
template <class F> __global__ void k_field_op(int op, const fe* a, const fe* b, fe* out, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe x = load_fe(a + i), y = load_fe(b + i), r;
    if (op == 0) r = fe_mul<F>(x, y);
    else if (op == 1) r = fe_add<F>(x, y);
    else if (op == 2) r = fe_sub<F>(x, y);
    else r = fe_inv<F>(x);
    store_fe(out + i, r);
}
// ILP independent dependent-chains of fe_mul per thread (ILP = 1, 2, 4): latency vs throughput probe
template <class F, int ILP> __global__ void k_mul_chain(fe* out, unsigned iters) {
    fe x[ILP], y = fe_r2<F>();
    y.v[1] ^= blockIdx.x;
#pragma unroll
    for (int k = 0; k < ILP; k++) { x[k] = fe_one<F>(); x[k].v[0] ^= threadIdx.x + 977 * k; }
    for (unsigned i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < ILP; k++) x[k] = fe_mul<F>(x[k], y);
    }
    uint32_t acc = 0;
#pragma unroll
    for (int k = 0; k < ILP; k++) acc ^= x[k].v[0] ^ x[k].v[7];
    if (acc == 0x12345678u) store_fe(out, x[0]);  // keep the chains alive
}
// chain of XYZZ mixed additions (the MSM inner loop) on register-resident operands
template <class F> __global__ void k_madd_chain(xyzz_t* out, unsigned iters) {
    affine_t q;
    q.x = fe_one<F>(); q.y = fe_r2<F>();
    q.x.v[0] ^= threadIdx.x; q.y.v[1] ^= blockIdx.x;
    xyzz_t acc = xyzz_from_affine<F>(q);
    acc.X.v[2] ^= 0x55u;
    for (unsigned i = 0; i < iters; i++) {
        acc = xyzz_madd<F>(acc, q);
        q.x.v[3] ^= acc.X.v[0];   // data-dependent operand so nothing is hoisted
    }
    if (acc.X.v[0] == 0x12345678u && acc.ZZ.v[7] == 0x9abcdef0u) store_xyzz(out, acc);
}

// chains of full XYZZ additions: serial formula (kind 102) and the quad-cooperative one (kind 101)
template <class F, int QUAD> __global__ void k_add_chain(xyzz_t* out, unsigned iters) {
    affine_t q;
    q.x = fe_one<F>(); q.y = fe_r2<F>();
    q.x.v[0] ^= QUAD ? (threadIdx.x >> 2) : threadIdx.x; q.y.v[1] ^= blockIdx.x;
    xyzz_t acc = xyzz_from_affine<F>(q), b = acc;
    b.X.v[2] ^= 0x55u; b.ZZ.v[1] ^= 0x3u;
    for (unsigned i = 0; i < iters; i++) {
        acc = QUAD ? xyzz_add_quad<F>(acc, b) : xyzz_add<F>(acc, b);
        b.X.v[3] ^= acc.X.v[0];
    }
    if (acc.X.v[0] == 0x12345678u && acc.ZZ.v[7] == 0x9abcdef0u) store_xyzz(out, acc);
}

}  // namespace zkb

using namespace zkb;

// ============================================================================================== extern "C"
extern "C" {

const char* zk_last_error(void) { return g_err; }

int zk_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int zk_ctx_create(int device_id, zk_ctx** out) {
    if (!out) { zk_set_error("ctx_create: out is null"); return ZK_ERR_INVALID; }
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        zk_set_error("no CUDA device (%s): this library has no CPU fallback", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return ZK_ERR_NO_DEVICE;
    }
    if (device_id < 0 || device_id >= n) { zk_set_error("ctx_create: device %d outside [0, %d)", device_id, n); return ZK_ERR_INVALID; }
    ZK_CUDA(cudaSetDevice(device_id));
    zk_ctx* ctx = new zk_ctx();
    if (int rc = ctx_init_lane(ctx, device_id)) { delete ctx; return rc; }
    *out = ctx;
    return ZK_OK;
}

void zk_ctx_destroy(zk_ctx* ctx) {
    if (!ctx) return;
    for (zk_ctx* c : ctx->children) zk_ctx_destroy(c);
    ctx->children.clear();
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    msm_workspace_free(ctx->ws);
    for (int l = 0; l < zk_ctx::SIDE_STREAMS; l++)
        if (ctx->side[l]) { cudaStreamSynchronize(ctx->side[l]); cudaStreamDestroy(ctx->side[l]); }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->h_scratch) cudaFreeHost(ctx->h_scratch);
    if (ctx->h_gather) cudaFreeHost(ctx->h_gather);
    if (ctx->d_gather_sum) cudaFree(ctx->d_gather_sum);
    if (ctx->d_scalars) cudaFree(ctx->d_scalars);
    if (ctx->d_open) cudaFree(ctx->d_open);
    if (ctx->d_ipa) cudaFree(ctx->d_ipa);
    if (ctx->d_expr) cudaFree(ctx->d_expr);
    if (ctx->d_flag) cudaFree(ctx->d_flag);
    if (ctx->d_ntt) cudaFree(ctx->d_ntt);
    if (ctx->d_ntt_tmp) cudaFree(ctx->d_ntt_tmp);
    for (int f = 0; f < 2; f++) for (int d = 0; d < 2; d++) if (ctx->ntt_small[f][d]) cudaFree(ctx->ntt_small[f][d]);
    for (auto& kv : ctx->ntt_tables) ntt_free_tables(kv.second);
    for (auto& e : ctx->ev_ntt) if (e) cudaEventDestroy(e);
    cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

int zk_ctx_set_stream(zk_ctx* ctx, void* cuda_stream) {
    if (!ctx) { zk_set_error("set_stream: ctx is null"); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return ZK_OK;
}

uint64_t zk_ctx_launch_count(const zk_ctx* ctx) {
    if (!ctx) return 0;
    uint64_t n = ctx->launches;
    for (const zk_ctx* c : ctx->children) n += c->launches;
    return n;
}

int zk_ctx_set_profile(zk_ctx* ctx, int enabled) {
    if (!ctx) { zk_set_error("set_profile: ctx is null"); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->ws.profile = enabled != 0;
    ctx->profile = enabled != 0;
    return ZK_OK;
}

int zk_ctx_set_option(zk_ctx* ctx, const char* name, long value) {
    if (!ctx || !name) { zk_set_error("set_option: null argument"); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!strcmp(name, "msm_chunk")) {
        if (value < 0 || value > 4096) { zk_set_error("set_option: msm_chunk %ld outside [0, 4096]", value); return ZK_ERR_INVALID; }
        ctx->ws.chunk = (uint32_t)value;
        for (zk_ctx* c : ctx->children) c->ws.chunk = (uint32_t)value;
        return ZK_OK;
    }
    if (!strcmp(name, "ctx_lanes")) {
        if (value < 1 || value > 16) { zk_set_error("set_option: ctx_lanes %ld outside [1, 16]", value); return ZK_ERR_INVALID; }
        ctx->n_lanes = (int)value;       // lanes already created stay allocated; fewer are used from now on
        return ZK_OK;
    }
    if (!strcmp(name, "msm_batch")) {
        if (value < 1 || value > (long)MSM_MAX_BATCH) { zk_set_error("set_option: msm_batch %ld outside [1, %u]", value, MSM_MAX_BATCH); return ZK_ERR_INVALID; }
        ctx->batch = (int)value;
        for (zk_ctx* c : ctx->children) c->batch = (int)value;
        return ZK_OK;
    }
    if (!strcmp(name, "msm_tma")) {
        if (value < 0 || value > 1) { zk_set_error("set_option: msm_tma %ld outside [0, 1]", value); return ZK_ERR_INVALID; }
        ctx->ws.tma_gather = value != 0;
        for (zk_ctx* c : ctx->children) c->ws.tma_gather = value != 0;
        return ZK_OK;
    }
    if (!strcmp(name, "msm_pdl")) {
        if (value < 0 || value > 1) { zk_set_error("set_option: msm_pdl %ld outside [0, 1]", value); return ZK_ERR_INVALID; }
        ctx->ws.pdl = value != 0;
        for (zk_ctx* c : ctx->children) c->ws.pdl = value != 0;
        return ZK_OK;
    }
    if (!strcmp(name, "msm_wave_threads")) {
        if (value < 0 || value > 2048) { zk_set_error("set_option: msm_wave_threads %ld outside [0, 2048]", value); return ZK_ERR_INVALID; }
        ctx->ws.wave_threads = (uint32_t)value;
        for (zk_ctx* c : ctx->children) c->ws.wave_threads = (uint32_t)value;
        return ZK_OK;
    }
    zk_set_error("set_option: unknown option '%s'", name);
    return ZK_ERR_INVALID;
}

int zk_ctx_last_stage_ms(const zk_ctx* ctx, float* out, size_t capacity) {
    if (!ctx || !out || capacity < 8) { zk_set_error("last_stage_ms: need room for 8 floats"); return ZK_ERR_INVALID; }
    for (int k = 0; k < 6; k++) out[k] = ctx->ws.stage_ms[k];
    out[6] = ctx->ntt_ms;
    out[7] = 0;
    return ZK_OK;
}

// ---------------------------------------------------------------------------------------------- bases
int zk_bases_upload(zk_ctx* ctx, int curve_id, const uint64_t* xy_mont, size_t n, int window_bits, int points_on_device, zk_bases** out) {
    if (!ctx || !out || (!xy_mont && n)) { zk_set_error("bases_upload: null argument"); return ZK_ERR_INVALID; }
    if (curve_id != ZK_PALLAS && curve_id != ZK_VESTA) { zk_set_error("bases_upload: unknown curve_id %d", curve_id); return ZK_ERR_INVALID; }
    if (window_bits < -1 || window_bits == 1 || window_bits > (int)MSM_MAX_WINDOW_BITS) { zk_set_error("bases_upload: window_bits %d not in {-1, 0, 2..%u}", window_bits, MSM_MAX_WINDOW_BITS); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    unsigned c = window_bits < 0 ? (unsigned)msm_default_window(n, true) : (unsigned)window_bits;
    zk_bases* bs = new zk_bases();
    bs->ctx = ctx;
    bs->b.curve = curve_id;
    int rc = curve_id == ZK_PALLAS ? msm_bases_create<FpParams>(bs->b, (const affine_t*)xy_mont, points_on_device != 0, n, c, ctx->stream)
                                   : msm_bases_create<FqParams>(bs->b, (const affine_t*)xy_mont, points_on_device != 0, n, c, ctx->stream);
    if (rc) { msm_bases_free(bs->b); delete bs; return rc; }
    if (c) ctx->launches += 1;
    *out = bs;
    return ZK_OK;
}

void zk_bases_free(zk_bases* bases) {
    if (!bases) return;
    std::lock_guard<std::mutex> lk(bases->ctx->mu);
    cudaSetDevice(bases->ctx->device);
    msm_bases_free(bases->b);
    delete bases;
}

size_t zk_bases_len(const zk_bases* bases) { return bases ? bases->b.n : 0; }
int zk_bases_window_bits(const zk_bases* bases) { return bases ? (int)bases->b.c : 0; }

// Point codecs between the reference's serialised forms and affine Montgomery points; host pointers.
//   mode 0: 33-byte compressed   -> affine   (decompression: one square root per point)
//   mode 1: 65-byte uncompressed -> affine   (unchecked, as SerdeAsUnchecked)
//   mode 2: affine -> 33-byte compressed
static int points_codec(zk_ctx* ctx, int curve_id, int mode, const void* in, size_t n, void* out, const char* what) {
    if (!ctx || (!in && n) || (!out && n)) { zk_set_error("%s: null argument", what); return ZK_ERR_INVALID; }
    if (curve_id != ZK_PALLAS && curve_id != ZK_VESTA) { zk_set_error("%s: unknown curve_id %d", what, curve_id); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    if (n == 0) return ZK_OK;
    const size_t in_bytes = (mode == 0 ? 33 : mode == 1 ? 65 : sizeof(affine_t)) * n, out_bytes = (mode == 2 ? 33 : sizeof(affine_t)) * n;
    void *d_in = nullptr, *d_out = nullptr;
    unsigned* d_bad = nullptr;
    unsigned bad = 0;
    cudaError_t e = cudaMalloc(&d_in, in_bytes);
    if (e == cudaSuccess) e = cudaMalloc(&d_out, out_bytes);
    if (e == cudaSuccess) e = cudaMalloc(&d_bad, sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMemsetAsync(d_bad, 0, sizeof(unsigned), ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_in, in, in_bytes, cudaMemcpyHostToDevice, ctx->stream);
    int rc = ZK_OK;
    if (e == cudaSuccess) {
        const bool pallas = curve_id == ZK_PALLAS;
        if (mode == 0)
            rc = pallas ? points_decompress<FpParams>((const uint8_t*)d_in, (affine_t*)d_out, n, d_bad, ctx->stream)
                        : points_decompress<FqParams>((const uint8_t*)d_in, (affine_t*)d_out, n, d_bad, ctx->stream);
        else if (mode == 1)
            rc = pallas ? points_from_uncompressed<FpParams>((const uint8_t*)d_in, (affine_t*)d_out, n, d_bad, ctx->stream)
                        : points_from_uncompressed<FqParams>((const uint8_t*)d_in, (affine_t*)d_out, n, d_bad, ctx->stream);
        else
            rc = pallas ? points_compress<FpParams>((const affine_t*)d_in, (uint8_t*)d_out, n, ctx->stream)
                        : points_compress<FqParams>((const affine_t*)d_in, (uint8_t*)d_out, n, ctx->stream);
        if (rc == ZK_OK) {
            ctx->launches += 1;
            e = cudaMemcpyAsync(out, d_out, out_bytes, cudaMemcpyDeviceToHost, ctx->stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(&bad, d_bad, sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        }
    }
    cudaFree(d_in); cudaFree(d_out); cudaFree(d_bad);
    if (e != cudaSuccess) { zk_set_error("%s: %s", what, cudaGetErrorString(e)); return ZK_ERR_CUDA; }
    if (rc == ZK_OK && bad) {
        zk_set_error(mode == 0 ? "%s: %u of %zu encodings are invalid (x off the curve, x >= modulus, or unknown flag bits)" : "%s: %u of %zu points have a non-canonical coordinate", what, bad, n);
        return ZK_ERR_INVALID;
    }
    return rc;
}

int zk_points_decompress(zk_ctx* ctx, int curve_id, const uint8_t* in33, size_t n, uint64_t* out_xy) {
    return points_codec(ctx, curve_id, 0, in33, n, out_xy, "points_decompress");
}
int zk_points_from_uncompressed(zk_ctx* ctx, int curve_id, const uint8_t* in65, size_t n, uint64_t* out_xy) {
    return points_codec(ctx, curve_id, 1, in65, n, out_xy, "points_from_uncompressed");
}
int zk_points_compress(zk_ctx* ctx, int curve_id, const uint64_t* xy_mont, size_t n, uint8_t* out33) {
    return points_codec(ctx, curve_id, 2, xy_mont, n, out33, "points_compress");
}

int zk_points_synthetic(zk_ctx* ctx, int curve_id, uint64_t seed, size_t n, uint64_t* out_xy) {
    if (!ctx || (!out_xy && n)) { zk_set_error("points_synthetic: null argument"); return ZK_ERR_INVALID; }
    if (curve_id != ZK_PALLAS && curve_id != ZK_VESTA) { zk_set_error("points_synthetic: unknown curve_id %d", curve_id); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    if (n == 0) return ZK_OK;
    affine_t* d = nullptr;
    ZK_CUDA(cudaMalloc(&d, n * sizeof(affine_t)));
    int rc = curve_id == ZK_PALLAS ? points_synthetic<FpParams>(d, n, seed, ctx->stream) : points_synthetic<FqParams>(d, n, seed, ctx->stream);
    cudaError_t e = cudaSuccess;
    if (rc == ZK_OK) {
        ctx->launches += 1;
        e = cudaMemcpyAsync(out_xy, d, n * sizeof(affine_t), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    }
    cudaFree(d);
    if (e != cudaSuccess) { zk_set_error("points_synthetic: %s", cudaGetErrorString(e)); return ZK_ERR_CUDA; }
    return rc;
}

// ---------------------------------------------------------------------------------------------- MSM
int zk_msm_dev(zk_ctx* ctx, const zk_bases* bases, size_t off, size_t n, const void* d_scalars, int scalars_are_mont, int window_bits, uint64_t out_xyz[12]) {
    if (!ctx || !bases || !out_xyz || (!d_scalars && n)) { zk_set_error("msm: null argument"); return ZK_ERR_INVALID; }
    if (ctx_root(bases->ctx) != ctx_root(ctx)) { zk_set_error("msm: bases belong to another context"); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    return ctx_msm_device(ctx, bases, off, n, (const fe*)d_scalars, scalars_are_mont, window_bits, out_xyz);
}

int zk_msm_batch(zk_ctx* root, const zk_bases* bases, size_t off, size_t n, const uint64_t* scalars, size_t k, int scalars_are_mont, int window_bits, uint64_t* out_xyz) {
    if (!root || !bases || (!out_xyz && k) || (!scalars && n && k)) { zk_set_error("msm: null argument"); return ZK_ERR_INVALID; }
    if (ctx_root(bases->ctx) != ctx_root(root)) { zk_set_error("msm: bases belong to another context"); return ZK_ERR_INVALID; }
    LaneLock ll;                             // host pointers in, host result out: any free lane of the pool
    if (int rc = ctx_acquire_lane(root, ll)) return rc;
    zk_ctx* ctx = ll.lane;
    ZK_CUDA(cudaSetDevice(ctx->device));
    if (k == 0) return ZK_OK;
    // Scalars in page-locked (cudaHostAlloc / cudaHostRegister) memory are read by the recode kernel straight over PCIe
    // (unified addressing): no staging copy, the transfer is fused into the first kernel.  Pageable memory is staged.
    const fe* d_sc = nullptr;
    int rc = ZK_OK;
    cudaPointerAttributes attr;
    if (n && cudaPointerGetAttributes(&attr, scalars) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer) {
        d_sc = (const fe*)attr.devicePointer;
    } else {
        cudaGetLastError();  // clear the "invalid value" some drivers report for pageable pointers
        rc = ctx_ensure((void**)&ctx->d_scalars, &ctx->cap_scalars, std::max<size_t>(k * n, 1) * sizeof(fe));
        if (rc) return rc;
        if (n) ZK_CUDA(cudaMemcpyAsync(ctx->d_scalars, scalars, k * n * sizeof(fe), cudaMemcpyHostToDevice, ctx->stream));
        d_sc = ctx->d_scalars;
    }
    std::vector<const fe*> scs(k);
    for (size_t j = 0; j < k; j++) scs[j] = d_sc + j * n;
    return ctx_msm_many(ctx, bases, off, n, scs.data(), k, scalars_are_mont, window_bits, out_xyz);
}

// Multi-GPU sharding (SURVEY.md §8e): this rank's MSM is left on the device as its slice sums and nothing is synchronised, so
// the caller can enqueue the all-gather on the same stream while the kernels still run.
static int msm_partial_impl(zk_ctx* ctx, const zk_bases* bases, size_t off, size_t n, const void* scalars, int scalars_are_mont, int window_bits,
                   void* d_out, size_t capacity_points, unsigned* out_c, unsigned* out_groups) {
    if (!ctx || !bases || !d_out || !out_c || !out_groups || (!scalars && n)) { zk_set_error("msm_partial: null argument"); return ZK_ERR_INVALID; }
    if (ctx_root(bases->ctx) != ctx_root(ctx)) { zk_set_error("msm: bases belong to another context"); return ZK_ERR_INVALID; }
    if (window_bits < 0 || window_bits > (int)MSM_MAX_WINDOW_BITS) { zk_set_error("msm: window_bits %d outside [0, %u]", window_bits, MSM_MAX_WINDOW_BITS); return ZK_ERR_INVALID; }
    if (n == 0) { zk_set_error("msm_partial: empty slice"); return ZK_ERR_INVALID; }
    const fe* d_sc = nullptr;
    cudaPointerAttributes attr;
    const bool known = cudaPointerGetAttributes(&attr, scalars) == cudaSuccess;
    if (!known) cudaGetLastError();   // some drivers report "invalid value" for pageable pointers
    if (known && (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged)) {
        d_sc = (const fe*)scalars;
    } else if (known && attr.type == cudaMemoryTypeHost && attr.devicePointer) {
        d_sc = (const fe*)attr.devicePointer;          // page-locked: read over PCIe by the recode kernel
    } else {
        int rc = ctx_ensure((void**)&ctx->d_scalars, &ctx->cap_scalars, n * sizeof(fe));
        if (rc) return rc;
        ZK_CUDA(cudaMemcpyAsync(ctx->d_scalars, scalars, n * sizeof(fe), cudaMemcpyHostToDevice, ctx->stream));
        d_sc = ctx->d_scalars;
    }
    MsmResultShape shape;
    unsigned nl = 0;
    ctx->ws.d_T_out = (xyzz_t*)d_out;
    ctx->ws.d_T_cap = capacity_points;
    int rc = bases->b.curve == ZK_PALLAS
                 ? msm_run<FpParams, FqParams>(bases->b, &off, n, &d_sc, 1, scalars_are_mont != 0, (unsigned)window_bits, ctx->ws, ctx->stream, &shape, &nl)
                 : msm_run<FqParams, FpParams>(bases->b, &off, n, &d_sc, 1, scalars_are_mont != 0, (unsigned)window_bits, ctx->ws, ctx->stream, &shape, &nl);
    ctx->ws.d_T_out = nullptr;
    ctx->ws.d_T_cap = 0;
    ctx->launches += nl;
    if (rc) return rc;
    *out_c = shape.c;
    *out_groups = shape.groups;
    return ZK_OK;
}

// d_all: `world` gathered partials of zk_msm_partial (device, world x groups*c points, same shape on every rank).  Sums them
// per slice on the device, copies groups*c points to the host and finishes the O(c) tail there.
static int msm_finish_gathered_impl(zk_ctx* ctx, int curve_id, const void* d_all, size_t world, unsigned c, unsigned groups, uint64_t out_xyz[12]) {
    if (!ctx || !d_all || !out_xyz || world == 0) { zk_set_error("msm_finish_gathered: null argument"); return ZK_ERR_INVALID; }
    if (curve_id != ZK_PALLAS && curve_id != ZK_VESTA) { zk_set_error("msm_finish_gathered: unknown curve_id %d", curve_id); return ZK_ERR_INVALID; }
    const size_t count = (size_t)c * groups;
    if (count == 0 || count > 4096) { zk_set_error("msm_finish_gathered: bad shape c = %u, groups = %u", c, groups); return ZK_ERR_INVALID; }
    int rc = ctx_ensure((void**)&ctx->d_gather_sum, &ctx->cap_gather_sum, count * sizeof(xyzz_t));
    if (rc) return rc;
    if (ctx->cap_h_gather < count) {
        if (ctx->h_gather) cudaFreeHost(ctx->h_gather);
        ctx->h_gather = nullptr; ctx->cap_h_gather = 0;
        ZK_CUDA(cudaMallocHost(&ctx->h_gather, count * sizeof(xyzz_t)));
        ctx->cap_h_gather = count;
    }
    rc = curve_id == ZK_PALLAS ? msm_sum_partials<FpParams>((const xyzz_t*)d_all, world, count, ctx->d_gather_sum, ctx->stream)
                               : msm_sum_partials<FqParams>((const xyzz_t*)d_all, world, count, ctx->d_gather_sum, ctx->stream);
    if (rc) return rc;
    ctx->launches += 1;
    ZK_CUDA(cudaMemcpyAsync(ctx->h_gather, ctx->d_gather_sum, count * sizeof(xyzz_t), cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(cudaStreamSynchronize(ctx->stream));
    host::hxyzz r = curve_id == ZK_PALLAS ? msm_finish_t<host::HFp>(ctx->h_gather, c, groups) : msm_finish_t<host::HFq>(ctx->h_gather, c, groups);
    xyzz_to_jac_out(curve_id, r, out_xyz);
    return ZK_OK;
}

int zk_msm_partial(zk_ctx* ctx, const zk_bases* bases, size_t off, size_t n, const void* scalars, int scalars_are_mont, int window_bits,
                   void* d_out, size_t capacity_points, unsigned* out_c, unsigned* out_groups) {
    if (!ctx) { zk_set_error("msm_partial: null argument"); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    return msm_partial_impl(ctx, bases, off, n, scalars, scalars_are_mont, window_bits, d_out, capacity_points, out_c, out_groups);
}
int zk_msm_finish_gathered(zk_ctx* ctx, int curve_id, const void* d_all, size_t world, unsigned c, unsigned groups, uint64_t out_xyz[12]) {
    if (!ctx) { zk_set_error("msm_finish_gathered: null argument"); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    return msm_finish_gathered_impl(ctx, curve_id, d_all, world, c, groups, out_xyz);
}

int zk_msm(zk_ctx* ctx, const zk_bases* bases, size_t off, size_t n, const uint64_t* scalars, int scalars_are_mont, int window_bits, uint64_t out_xyz[12]) {
    return zk_msm_batch(ctx, bases, off, n, scalars, 1, scalars_are_mont, window_bits, out_xyz);
}

static int check_curve(int curve_id) {
    if (curve_id != ZK_PALLAS && curve_id != ZK_VESTA) { zk_set_error("unknown curve_id %d", curve_id); return ZK_ERR_INVALID; }
    return ZK_OK;
}

int zk_jacobian_to_affine(int curve_id, const uint64_t xyz[12], uint64_t out_xy[8]) {
    if (!xyz || !out_xy) { zk_set_error("null argument"); return ZK_ERR_INVALID; }
    if (int rc = check_curve(curve_id)) return rc;
    host::hjac j;
    memcpy(&j, xyz, sizeof j);
    host::haffine a = curve_id == ZK_PALLAS ? host::to_affine<host::HFp>(host::from_jacobian<host::HFp>(j))
                                            : host::to_affine<host::HFq>(host::from_jacobian<host::HFq>(j));
    memcpy(out_xy, &a, sizeof a);
    return ZK_OK;
}

int zk_jacobian_sum(int curve_id, const uint64_t* xyz, size_t count, uint64_t out_xyz[12]) {
    if ((!xyz && count) || !out_xyz) { zk_set_error("null argument"); return ZK_ERR_INVALID; }
    if (int rc = check_curve(curve_id)) return rc;
    host::hxyzz acc = host::identity();
    for (size_t i = 0; i < count; i++) {
        host::hjac j;
        memcpy(&j, xyz + 12 * i, sizeof j);
        acc = curve_id == ZK_PALLAS ? host::padd<host::HFp>(acc, host::from_jacobian<host::HFp>(j))
                                    : host::padd<host::HFq>(acc, host::from_jacobian<host::HFq>(j));
    }
    xyzz_to_jac_out(curve_id, acc, out_xyz);
    return ZK_OK;
}

int zk_jacobian_add(int curve_id, const uint64_t a_xyz[12], const uint64_t b_xyz[12], uint64_t out_xyz[12]) {
    if (!a_xyz || !b_xyz || !out_xyz) { zk_set_error("null argument"); return ZK_ERR_INVALID; }
    uint64_t both[24];
    memcpy(both, a_xyz, 96);
    memcpy(both + 12, b_xyz, 96);
    return zk_jacobian_sum(curve_id, both, 2, out_xyz);
}

// ---------------------------------------------------------------------------------------------- NTT
int zk_ntt_dev(zk_ctx* ctx, int field_id, void* d_data, unsigned log_n, size_t batch, size_t in_len, int inverse, int coset) {
    if (!ctx || (!d_data && batch)) { zk_set_error("ntt: null argument"); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    return ctx_ntt_device(ctx, field_id, (fe*)d_data, log_n, batch, in_len, inverse, coset);
}

int zk_ntt_dev_oop(zk_ctx* ctx, int field_id, const void* d_in, size_t in_stride, size_t in_len, void* d_out, unsigned log_n, size_t batch, int inverse,
                   int coset) {
    if (!ctx || ((!d_in || !d_out) && batch)) { zk_set_error("ntt: null argument"); return ZK_ERR_INVALID; }
    if (log_n > NTT_MAX_LOG_N) { zk_set_error("ntt: log_n %u > %u not supported", log_n, NTT_MAX_LOG_N); return ZK_ERR_INVALID; }
    const size_t n = (size_t)1 << log_n;
    if (in_len == 0 || in_len > n) in_len = n;
    if (in_stride < in_len && batch > 1) { zk_set_error("ntt: input stride %zu shorter than the %zu elements read per polynomial", in_stride, in_len); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    return ctx_ntt_device_oop(ctx, field_id, (const fe*)d_in, in_stride, (fe*)d_out, log_n, batch, in_len, inverse, coset);
}

// ---------------------------------------------------------------------------------------------- device memory for the *_dev entry points
int zk_dev_alloc(zk_ctx* ctx, size_t bytes, void** out) {
    if (!ctx || !out) { zk_set_error("dev_alloc: null argument"); return ZK_ERR_INVALID; }
    *out = nullptr;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    ZK_CUDA(cudaMalloc(out, bytes ? bytes : 1));
    return ZK_OK;
}
int zk_dev_free(zk_ctx* ctx, void* d_ptr) {
    if (!ctx) { zk_set_error("dev_free: null argument"); return ZK_ERR_INVALID; }
    if (!d_ptr) return ZK_OK;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    ZK_CUDA(cudaStreamSynchronize(ctx->stream));
    ZK_CUDA(cudaFree(d_ptr));
    return ZK_OK;
}
int zk_dev_upload(zk_ctx* ctx, void* d_dst, const void* src, size_t bytes) {
    if (!ctx || ((!d_dst || !src) && bytes)) { zk_set_error("dev_upload: null argument"); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    ZK_CUDA(cudaMemcpyAsync(d_dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    ZK_CUDA(cudaStreamSynchronize(ctx->stream));   // the source may be pageable and reused by the caller
    return ZK_OK;
}
int zk_dev_download(zk_ctx* ctx, void* dst, const void* d_src, size_t bytes) {
    if (!ctx || ((!dst || !d_src) && bytes)) { zk_set_error("dev_download: null argument"); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    ZK_CUDA(cudaMemcpyAsync(dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(cudaStreamSynchronize(ctx->stream));
    return ZK_OK;
}

int zk_ntt_batch(zk_ctx* root, int field_id, uint64_t* data, unsigned log_n, size_t batch, size_t in_len, int inverse, int coset) {
    if (!root || (!data && batch)) { zk_set_error("ntt: null argument"); return ZK_ERR_INVALID; }
    if (log_n > NTT_MAX_LOG_N) { zk_set_error("ntt: log_n %u > %u not supported", log_n, NTT_MAX_LOG_N); return ZK_ERR_INVALID; }
    LaneLock ll;                             // host pointers in and out: any free lane of the pool
    if (int rc0 = ctx_acquire_lane(root, ll)) return rc0;
    zk_ctx* ctx = ll.lane;
    ZK_CUDA(cudaSetDevice(ctx->device));
    if (batch == 0) return ZK_OK;
    const size_t n = (size_t)1 << log_n, poly_bytes = n * sizeof(fe), bytes = batch * poly_bytes;
    if (in_len == 0 || in_len > n || inverse) in_len = n;
    // (Transforming page-locked memory in place over PCIe was measured and is slower than two staged copies: the tile loads
    //  are 64-128 B requests.  MSM scalars, read once in full lines, do take the zero-copy route — zk_msm_batch.)
    int rc = ctx_ensure((void**)&ctx->d_ntt, &ctx->cap_ntt, bytes);
    if (rc) return rc;
    // Only the first in_len coefficients of every polynomial cross PCIe (the kernels zero-pad by position), and for batches in
    // page-locked memory the three stages are pipelined over chunks of polynomials: copy-in of chunk k+1, the transform of
    // chunk k and the copy-out of chunk k-1 run on three streams.  16 x FFT(8n) of kimchi's quotient step (in_len = n) moves
    // 32 MiB in and 256 MiB out: the call is bound by the copy-out alone instead of the sum of all three.
    cudaPointerAttributes attr;
    bool pinned = cudaPointerGetAttributes(&attr, data) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    size_t per = batch;                                  // polynomials per chunk
    if (pinned && !ctx->profile && batch >= 2 && bytes >= ((size_t)8 << 20)) {
        per = std::max<size_t>(1, ((size_t)16 << 20) / poly_bytes);
        if (per * 2 > batch) per = (batch + 1) / 2;
    }
    if (per == batch) {
        ZK_CUDA(cudaMemcpy2DAsync(ctx->d_ntt, poly_bytes, data, poly_bytes, in_len * sizeof(fe), batch, cudaMemcpyHostToDevice, ctx->stream));
        rc = ctx_ntt_device(ctx, field_id, ctx->d_ntt, log_n, batch, in_len, inverse, coset);
        if (rc) return rc;
        ZK_CUDA(cudaMemcpyAsync(data, ctx->d_ntt, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        ZK_CUDA(cudaStreamSynchronize(ctx->stream));
        return ZK_OK;
    }
    rc = ctx_side_streams_init(ctx);
    if (rc) return rc;
    cudaStream_t s_in = ctx->side[0], s_out = ctx->side[1];
    const size_t chunks = (batch + per - 1) / per;
    std::vector<cudaEvent_t> ev(2 * chunks, nullptr);
    cudaError_t e = cudaEventRecord(ctx->ev_fork, ctx->stream);      // work already queued on the caller's stream comes first
    if (e == cudaSuccess) e = cudaStreamWaitEvent(s_in, ctx->ev_fork, 0);
    for (size_t k = 0; k < chunks && e == cudaSuccess && rc == ZK_OK; k++) {
        const size_t j0 = k * per, cnt = std::min(per, batch - j0);
        fe* d = ctx->d_ntt + j0 * n;
        const uint64_t* h = data + 4 * j0 * n;
        e = cudaEventCreateWithFlags(&ev[2 * k], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev[2 * k + 1], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaMemcpy2DAsync(d, poly_bytes, h, poly_bytes, in_len * sizeof(fe), cnt, cudaMemcpyHostToDevice, s_in);
        if (e == cudaSuccess) e = cudaEventRecord(ev[2 * k], s_in);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ev[2 * k], 0);
        if (e != cudaSuccess) break;
        rc = ctx_ntt_device(ctx, field_id, d, log_n, cnt, in_len, inverse, coset);
        if (rc) break;
        e = cudaEventRecord(ev[2 * k + 1], ctx->stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(s_out, ev[2 * k + 1], 0);
        if (e == cudaSuccess) e = cudaMemcpyAsync((void*)h, d, cnt * poly_bytes, cudaMemcpyDeviceToHost, s_out);
    }
    cudaStreamSynchronize(s_in);
    cudaStreamSynchronize(ctx->stream);
    cudaError_t e2 = cudaStreamSynchronize(s_out);
    for (auto& x : ev) if (x) cudaEventDestroy(x);
    if (rc) return rc;
    if (e != cudaSuccess || e2 != cudaSuccess) { zk_set_error("ntt: %s", cudaGetErrorString(e != cudaSuccess ? e : e2)); return ZK_ERR_CUDA; }
    return ZK_OK;
}

int zk_ntt(zk_ctx* ctx, int field_id, uint64_t* data, unsigned log_n, int inverse, int coset) {
    return zk_ntt_batch(ctx, field_id, data, log_n, 1, 0, inverse, coset);
}

// ---------------------------------------------------------------------------------------------- diagnostics
int zk_debug_field_op(zk_ctx* ctx, int field_id, int op, const uint64_t* a, const uint64_t* b, uint64_t* out, size_t n) {
    if (!ctx || !a || !b || !out) { zk_set_error("null argument"); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    fe *da, *db, *dout;
    ZK_CUDA(cudaMalloc(&da, n * sizeof(fe)));
    ZK_CUDA(cudaMalloc(&db, n * sizeof(fe)));
    ZK_CUDA(cudaMalloc(&dout, n * sizeof(fe)));
    ZK_CUDA(cudaMemcpyAsync(da, a, n * sizeof(fe), cudaMemcpyHostToDevice, ctx->stream));
    ZK_CUDA(cudaMemcpyAsync(db, b, n * sizeof(fe), cudaMemcpyHostToDevice, ctx->stream));
    unsigned blocks = (unsigned)((n + 127) / 128);
    if (field_id == ZK_FP) k_field_op<FpParams><<<blocks, 128, 0, ctx->stream>>>(op, da, db, dout, n);
    else k_field_op<FqParams><<<blocks, 128, 0, ctx->stream>>>(op, da, db, dout, n);
    ZK_CUDA(cudaGetLastError());
    ctx->launches += 1;
    ZK_CUDA(cudaMemcpyAsync(out, dout, n * sizeof(fe), cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(cudaStreamSynchronize(ctx->stream));
    cudaFree(da); cudaFree(db); cudaFree(dout);
    return ZK_OK;
}

// kind: 1, 2, 4 = fe_mul chains with that many independent chains per thread; 100 = xyzz_madd chain.
// blocks == 0: 4 per SM.  Reports operations per second (fe_mul, or madd for kind 100).
int zk_debug_op_throughput(zk_ctx* ctx, int field_id, int kind, unsigned blocks, unsigned threads, unsigned iters, double* out_ops_per_s) {
    if (!ctx || !out_ops_per_s || threads == 0 || threads > 1024) { zk_set_error("op_throughput: bad argument"); return ZK_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    ZK_CUDA(cudaSetDevice(ctx->device));
    cudaDeviceProp prop;
    ZK_CUDA(cudaGetDeviceProperties(&prop, ctx->device));
    if (blocks == 0) blocks = prop.multiProcessorCount * 4;
    xyzz_t* dout;
    ZK_CUDA(cudaMalloc(&dout, sizeof(xyzz_t)));
    cudaEvent_t e0, e1;
    ZK_CUDA(cudaEventCreate(&e0));
    ZK_CUDA(cudaEventCreate(&e1));
    for (int rep = 0; rep < 2; rep++) {  // first launch warms up
        ZK_CUDA(cudaEventRecord(e0, ctx->stream));
#define LAUNCH(F)                                                                                        \
        if (kind == 1) k_mul_chain<F, 1><<<blocks, threads, 0, ctx->stream>>>((fe*)dout, iters);         \
        else if (kind == 2) k_mul_chain<F, 2><<<blocks, threads, 0, ctx->stream>>>((fe*)dout, iters);    \
        else if (kind == 4) k_mul_chain<F, 4><<<blocks, threads, 0, ctx->stream>>>((fe*)dout, iters);    \
        else if (kind == 101) k_add_chain<F, 1><<<blocks, threads, 0, ctx->stream>>>(dout, iters);                \
        else if (kind == 102) k_add_chain<F, 0><<<blocks, threads, 0, ctx->stream>>>(dout, iters);                \
        else k_madd_chain<F><<<blocks, threads, 0, ctx->stream>>>(dout, iters);
        if (field_id == ZK_FP) { LAUNCH(FpParams) } else { LAUNCH(FqParams) }
#undef LAUNCH
        ZK_CUDA(cudaGetLastError());
        ZK_CUDA(cudaEventRecord(e1, ctx->stream));
        ZK_CUDA(cudaEventSynchronize(e1));
    }
    ctx->launches += 2;
    float ms = 0;
    ZK_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    double per_thread = kind == 101 ? 0.25 : kind >= 100 ? 1.0 : (double)kind;
    *out_ops_per_s = per_thread * iters * (double)blocks * threads / (ms * 1e-3);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(dout);
    return ZK_OK;
}

int zk_debug_mul_throughput(zk_ctx* ctx, int field_id, unsigned iters, double* out_mul_per_s) {
    return zk_debug_op_throughput(ctx, field_id, 2, 0, 256, iters, out_mul_per_s);
}

}  // extern "C"

namespace zkb {
int ctx_msm_partial_nolock(zk_ctx* ctx, const zk_bases* bases, size_t off, size_t n, const void* scalars, int scalars_are_mont, int window_bits,
                           void* d_out, size_t capacity_points, unsigned* out_c, unsigned* out_groups) {
    return msm_partial_impl(ctx, bases, off, n, scalars, scalars_are_mont, window_bits, d_out, capacity_points, out_c, out_groups);
}
int ctx_msm_finish_gathered_nolock(zk_ctx* ctx, int curve_id, const void* d_all, size_t world, unsigned c, unsigned groups, uint64_t out_xyz[12]) {
    return msm_finish_gathered_impl(ctx, curve_id, d_all, world, c, groups, out_xyz);
}
}  // namespace zkb
