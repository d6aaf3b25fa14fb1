/*
 * zkb200.h — C ABI of the B200-native MSM + NTT hot path of o1-labs/proof-systems (Kimchi).
 *
 * The reference has NO C ABI or plugin loader on this path: its seam is two Rust traits and one arkworks trait
 * (SURVEY.md §8b).  These entry points are what a Rust `extern "C"` block behind those traits binds
 * (INTEGRATION.md shows the shim); each one names the reference interface it replaces.
 *
 * Conventions (identical to the reference's in-memory representation, so no re-encoding at the boundary):
 *   field element   4 x uint64_t little-endian limbs, MONTGOMERY form (R = 2^256) unless a parameter says canonical
 *                   == ark_ff::Fp256<MontBackend<_,4>>.0.0   (curves/src/pasta/fields/fp.rs:8-12, fq.rs:8-12;
 *                   the reference itself treats Fp as raw limbs in kimchi/src/cached_prover_index.rs:486-530)
 *   affine point    x || y, 8 x uint64_t; the identity (Affine{infinity: true},
 *                   poly-commitment/src/commitment.rs:563-569) is encoded as all zeros — (0,0) is not on y^2 = x^3 + 5
 *   Jacobian point  X || Y || Z, 12 x uint64_t, x = X/Z^2, y = Y/Z^3, identity Z = 0  (ark_ec Projective)
 *   field_id        ZK_FP = Pallas base / Vesta scalar field, ZK_FQ = Vesta base / Pallas scalar field
 *   curve_id        ZK_PALLAS (coordinates Fp, scalars Fq), ZK_VESTA (coordinates Fq, scalars Fp)
 *
 * Every function returns 0 on success or a negative ZK_ERR_* code; zk_last_error() describes the last failure of
 * the calling thread.  Nothing unwinds across the boundary.  A context is a pool of lanes (stream + workspace each; option
 * "ctx_lanes", default 4): calls that take HOST pointers from different threads — the 15 concurrent rayon callers of
 * kimchi/src/prover.rs:329-351 — each take a free lane and overlap on the GPU; calls on an external stream, calls that take
 * device pointers and zk_srs_open (which holds the context across its callbacks) are serialised on the primary lane.
 * There is NO CPU fallback: without a CUDA device zk_ctx_create fails with ZK_ERR_NO_DEVICE.
 */
#ifndef ZKB200_H
#define ZKB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

#define ZK_FP 0
#define ZK_FQ 1
#define ZK_PALLAS 0
#define ZK_VESTA 1

#define ZK_OK 0
#define ZK_ERR_INVALID (-1)
#define ZK_ERR_CUDA (-2)
#define ZK_ERR_NO_DEVICE (-3)
#define ZK_ERR_LENGTH (-4)

typedef struct zk_ctx zk_ctx;       /* one CUDA device + stream + scratch; one per process/rank in multi-GPU runs */
typedef struct zk_bases zk_bases;   /* a resident set of MSM bases (an SRS `g`, or one Lagrange basis) */
typedef struct zk_srs zk_srs;       /* host-side mirror of poly_commitment::ipa::SRS<G> on top of the above */

/* ------------------------------------------------------------------ library / context */
const char* zk_last_error(void);
int zk_device_count(void);
int zk_ctx_create(int device_id, zk_ctx** out);
void zk_ctx_destroy(zk_ctx* ctx);
/* Run on the caller's CUDA stream (a cudaStream_t, e.g. torch.cuda.current_stream().cuda_stream); NULL = own stream. */
int zk_ctx_set_stream(zk_ctx* ctx, void* cuda_stream);
/* Kernels launched by this context so far (bench.py's gpu_launches). */
uint64_t zk_ctx_launch_count(const zk_ctx* ctx);
/* Per-stage device timing with CUDA events on the launching stream (bench.py's roofline line).  After a profiled call
 * zk_ctx_last_stage_ms fills out[0..5] = MSM stages {recode, plan, scatter, accumulate, finish, bitsum} of the last
 * MSM and out[6] = all kernels of the last NTT call, in milliseconds.  capacity >= 8. */
int zk_ctx_set_profile(zk_ctx* ctx, int enabled);
/* Tuning knobs.  "msm_chunk": sorted entries per accumulation task (0 = built-in default: the tasks fill the machine once).
 *                "msm_batch": 1..16 MSMs of one call fused into ONE pipeline with one bucket group per MSM (zk_msm_batch,
 *                zk_srs_commit_non_hiding with several chunks, zk_srs_commit_evaluations_batch, the L/R pair of
 *                zk_ipa_round_lr): every latency-bound stage is paid once per batch; default 16.
 *                "msm_wave_threads": accumulation threads per SM the task count is sized for (0 = built-in default).
 *                "msm_pdl": 1 (default) launches the MSM pipeline's kernels after the first with programmatic dependent launch
 *                and no per-call memsets; 0 uses plain launches behind two memsets (same results, for A/B timing). */
int zk_ctx_set_option(zk_ctx* ctx, const char* name, long value);
int zk_ctx_last_stage_ms(const zk_ctx* ctx, float* out, size_t capacity);

/* ------------------------------------------------------------------ resident bases
 * Replaces holding `SRS::g: Vec<G>` / a cached Lagrange basis in host memory (poly-commitment/src/ipa.rs:56-75,780-795).
 * window_bits: 0 = keep only the points (per-window buckets, host combines windows);
 *              2..16 = also precompute T[w][i] = 2^(w*window_bits) * P_i so every MSM on these bases uses ONE bucket set;
 *              -1 = pick the table window from n.
 * points_on_device != 0: xy_mont is a device pointer. */
int zk_bases_upload(zk_ctx* ctx, int curve_id, const uint64_t* xy_mont, size_t n, int window_bits, int points_on_device,
                    zk_bases** out);
void zk_bases_free(zk_bases* bases);
size_t zk_bases_len(const zk_bases* bases);
int zk_bases_window_bits(const zk_bases* bases);

/* Point decompression on the device: n points in ark-serialize's compressed short-Weierstrass form — the format of
 * srs/pallas.srs / srs/vesta.srs through SerdeAs (utils/src/serialization.rs:65-106): 32-byte LE canonical x, then a flag
 * byte (bit 7: y is the larger root, bit 6: infinity) — to affine Montgomery points.  ZK_ERR_INVALID if some x is off-curve. */
int zk_points_decompress(zk_ctx* ctx, int curve_id, const uint8_t* in33, size_t n, uint64_t* out_xy);
/* The other two codecs of utils/src/serialization.rs: the 65-byte uncompressed, unchecked form of srs/test_*.srs
 * (SerdeAsUnchecked, :108-146: x || y || flag byte, bit 6 = infinity; no curve check — ZK_ERR_INVALID only for a coordinate
 * >= the modulus), and the inverse of zk_points_decompress (the form PolyComm / OpeningProof serialise to, :65-84). */
int zk_points_from_uncompressed(zk_ctx* ctx, int curve_id, const uint8_t* in65, size_t n, uint64_t* out_xy);
int zk_points_compress(zk_ctx* ctx, int curve_id, const uint64_t* xy_mont, size_t n, uint8_t* out33);

/* Synthetic on-curve points for workloads larger than the 2^16 generators the reference ships (BASELINE config 4): point i is
 * a deterministic function of (curve_id, seed, i) — try-and-increment on x until x^3 + 5 is a square (csrc/decompress.cu).
 * Benchmark / test input only: the points have no known relation to the SRS generators. */
int zk_points_synthetic(zk_ctx* ctx, int curve_id, uint64_t seed, size_t n, uint64_t* out_xy);

/* ------------------------------------------------------------------ MSM
 * zk_msm == <G::Group as VariableBaseMSM>::msm_bigint(&bases[off..off+n], scalars)   (scalars_are_mont = 0: canonical
 *           integers, poly-commitment/src/ipa.rs:672,943,953; commitment.rs:382,387)
 *        == VariableBaseMSM::msm(...).unwrap()                                        (scalars_are_mont = 1: the
 *           into_bigint conversion runs on the device, ipa.rs:649,658,659)
 * window_bits: 0 = default; ignored when the bases carry a table.  out_xyz: Jacobian.
 * The *_dev variant takes scalars already resident in device memory (n x 4 u64). */
int zk_msm(zk_ctx* ctx, const zk_bases* bases, size_t off, size_t n, const uint64_t* scalars, int scalars_are_mont,
           int window_bits, uint64_t out_xyz[12]);
int zk_msm_dev(zk_ctx* ctx, const zk_bases* bases, size_t off, size_t n, const void* d_scalars, int scalars_are_mont,
               int window_bits, uint64_t out_xyz[12]);
/* k MSMs sharing the same bases slice (the chunks of t, the 15 witness columns): scalars k x n x 4, out k x 12. */
int zk_msm_batch(zk_ctx* ctx, const zk_bases* bases, size_t off, size_t n, const uint64_t* scalars, size_t k,
                 int scalars_are_mont, int window_bits, uint64_t* out_xyz);

/* Multi-GPU sharding by points (SURVEY.md §8e; the reference's own split is poly-commitment/src/ipa.rs:652-662 and
 * benches/msm.rs:92-140).  zk_msm_partial runs this rank's slice and leaves its result on the DEVICE as groups*c "slice sums"
 * (XYZZ points, 128 bytes each; the MSM is sum_g 2^(c g) sum_t 2^t T[g][t]) in d_out — nothing is copied to the host and
 * nothing is synchronised, so the caller enqueues the all-gather of d_out (ncclAllGather, world x groups*c x 128 bytes) on the
 * context's stream while the kernels still run.  zk_msm_finish_gathered adds the gathered partials slice by slice on the
 * device, reads groups*c points back and finishes the O(c) tail on the host; every rank gets identical bits.  `scalars` may
 * be device memory, page-locked host memory (read over PCIe) or pageable host memory (staged).  All ranks must use bases with
 * the same window (same c and groups). */
int zk_msm_partial(zk_ctx* ctx, const zk_bases* bases, size_t off, size_t n, const void* scalars, int scalars_are_mont,
                   int window_bits, void* d_out, size_t capacity_points, unsigned* out_c, unsigned* out_groups);
int zk_msm_finish_gathered(zk_ctx* ctx, int curve_id, const void* d_all, size_t world, unsigned c, unsigned groups,
                           uint64_t out_xyz[12]);
/* The same exchange with the communicator owned by the library: one NCCL communicator per context (one per process / GPU), the
 * all-gather enqueued from C on the context's stream right behind the MSM kernels, the cross-rank sum and the tail as above.
 *   zk_comm_unique_id   ncclGetUniqueId on one rank; the caller distributes the 128 bytes (MPI, a torch store, a file)
 *   zk_comm_init_rank   ncclCommInitRank — collective over the `world` ranks
 *   zk_msm_sharded      one MSM over world x n points: this rank's slice of ITS resident bases with its n scalars (device,
 *                       page-locked or pageable host memory); collective; every rank receives the identical result.  The reference's
 *                       1/2/4/8-way split: poly-commitment/benches/msm.rs:92-140.
 * NCCL is bound at run time (libnccl.so.2 of the host process, else the system's); without it these calls return ZK_ERR_INVALID. */
typedef struct zk_comm zk_comm;
int zk_comm_unique_id(uint8_t out_id[128]);
int zk_comm_init_rank(zk_ctx* ctx, const uint8_t id[128], int world, int rank, zk_comm** out);
void zk_comm_destroy(zk_comm* comm);
int zk_comm_world(const zk_comm* comm);
int zk_comm_rank(const zk_comm* comm);
int zk_msm_sharded(zk_comm* comm, const zk_bases* bases, size_t off, size_t n, const void* scalars, int scalars_are_mont,
                   int window_bits, uint64_t out_xyz[12]);
/* Projective::into_affine / `+` on the host (result handling; multi-GPU partial sums after the all-gather). */
int zk_jacobian_to_affine(int curve_id, const uint64_t xyz[12], uint64_t out_xy[8]);
int zk_jacobian_add(int curve_id, const uint64_t a_xyz[12], const uint64_t b_xyz[12], uint64_t out_xyz[12]);
int zk_jacobian_sum(int curve_id, const uint64_t* xyz, size_t count, uint64_t out_xyz[12]);

/* ------------------------------------------------------------------ NTT
 * == Radix2EvaluationDomain::<F>::new(1 << log_n).{fft_in_place, ifft_in_place}(data)
 *    (coset != 0: the domain is get_coset(F::GENERATOR), i.e. coset_fft / coset_ifft)
 * reached from Evaluations::interpolate / DensePolynomial::evaluate_over_domain at kimchi/src/prover.rs:289,377,907,1163,
 * kimchi/src/circuits/constraints.rs:494, poly-commitment/src/utils.rs:195-198.
 * data: batch polynomials of 2^log_n elements, back to back, transformed in place, natural order in and out.
 * in_len: forward input length per polynomial (elements >= in_len are taken as zero, like ark's resize); 0 = full. */
int zk_ntt(zk_ctx* ctx, int field_id, uint64_t* data, unsigned log_n, int inverse, int coset);
int zk_ntt_batch(zk_ctx* ctx, int field_id, uint64_t* data, unsigned log_n, size_t batch, size_t in_len, int inverse,
                 int coset);
int zk_ntt_dev(zk_ctx* ctx, int field_id, void* d_data, unsigned log_n, size_t batch, size_t in_len, int inverse,
               int coset);
/* Out of place, device to device: polynomial b is read from d_in + b * in_stride elements (its first in_len elements, the rest
 * of the domain is taken as zero) and its transform written to d_out + b * 2^log_n — DensePolynomial::evaluate_over_domain_by_ref
 * of n coefficients over d8 (kimchi/src/circuits/constraints.rs:488-507) without materialising the zero padding, and the
 * building block of a device-resident iFFT(n) -> FFT(8n) -> pointwise -> iFFT(8n) pipeline (SURVEY.md §8f row 3).
 * log_n up to 30 (three passes beyond 2^20). */
int zk_ntt_dev_oop(zk_ctx* ctx, int field_id, const void* d_in, size_t in_stride, size_t in_len, void* d_out, unsigned log_n,
                   size_t batch, int inverse, int coset);

/* Device memory for callers without a CUDA binding of their own (the Rust shim keeps witness / quotient polynomials resident
 * between calls of the *_dev entry points).  Synchronous copies; pointers are plain device pointers. */
int zk_dev_alloc(zk_ctx* ctx, size_t bytes, void** out);
int zk_dev_free(zk_ctx* ctx, void* d_ptr);
int zk_dev_upload(zk_ctx* ctx, void* d_dst, const void* src, size_t bytes);
int zk_dev_download(zk_ctx* ctx, void* dst, const void* d_src, size_t bytes);

/* ------------------------------------------------------------------ SRS mirror (poly-commitment/src/lib.rs:61-241, ipa.rs)
 * zk_srs_create            SRS{g, h} with g resident on the device            (ipa.rs:56-75)
 * zk_srs_max_poly_size     SRS::max_poly_size / size                           (ipa.rs:596-599, :798)
 * zk_srs_add_lagrange_basis register the basis of a domain (cache entry of get_lagrange_basis, ipa.rs:780-795)
 * zk_srs_commit_non_hiding SRS::commit_non_hiding(plnm, num_chunks)            (ipa.rs:638-683): coefficients in
 *                          Montgomery form; writes max(ceil(len/|g|), num_chunks, 1) affine chunks, returns the count
 * zk_srs_commit_evaluations_non_hiding  SRS::commit_evaluations_non_hiding     (ipa.rs:706-728): evals on a domain of
 *                          evals_domain_size >= domain_size are sub-sampled; fails (ZK_ERR_INVALID) where the reference panics
 * zk_srs_mask_custom       SRS::mask_custom: chunk_i + blinder_i * h           (ipa.rs:605-622); ZK_ERR_LENGTH ==
 *                          CommitmentError::BlindersDontMatch (poly-commitment/src/error.rs:3-9) */
int zk_srs_create(zk_ctx* ctx, int curve_id, const uint64_t* g_xy, size_t n, const uint64_t h_xy[8], int window_bits,
                  zk_srs** out);
void zk_srs_destroy(zk_srs* srs);
size_t zk_srs_max_poly_size(const zk_srs* srs);
int zk_srs_add_lagrange_basis(zk_srs* srs, size_t domain_size, const uint64_t* basis_xy, int window_bits);
/* SRS::get_lagrange_basis_from_domain_size -> SRS::lagrange_basis (ipa.rs:780-788, 1065-1172) computed ON THE DEVICE from the
 * resident generators: inverse FFT over group elements + normalisation, registered for commit_evaluations_non_hiding.
 * domain_size: a power of two.  A domain larger than |g| gives CHUNKED bases (ipa.rs:1145-1171): ceil(domain / |g|) partial
 * commitments per element (zk_srs_lagrange_basis_chunks), stored chunk-major — chunk c's domain_size points come first for c = 0,
 * and PolyComm i of the reference is (chunk_c[i])_c.  zk_srs_get_lagrange_basis copies all chunks to the host (chunks x n x 8 u64);
 * zk_srs_add_lagrange_basis takes the same layout; zk_srs_commit_evaluations_non_hiding then writes `chunks` points. */
int zk_srs_lagrange_basis(zk_srs* srs, size_t domain_size, int window_bits);
size_t zk_srs_lagrange_basis_chunks(const zk_srs* srs, size_t domain_size);
int zk_srs_get_lagrange_basis(zk_srs* srs, size_t domain_size, uint64_t* out_xy, size_t capacity_points);
int zk_srs_commit_non_hiding(zk_srs* srs, const uint64_t* coeffs_mont, size_t len, size_t num_chunks, uint64_t* out_xy,
                             size_t out_capacity, size_t* out_chunks);
int zk_srs_commit_evaluations_non_hiding(zk_srs* srs, size_t domain_size, const uint64_t* evals_mont,
                                         size_t evals_domain_size, uint64_t out_xy[8]);
/* k commit_evaluations_non_hiding calls on one domain in a single call (the reference issues the 15 witness columns
 * concurrently from rayon workers, kimchi/src/prover.rs:329-351): evals_mont = k x domain_size, out_xy = k x 8.  The
 * independent MSMs run as one fused pipeline (zk_ctx_set_option "msm_batch"). */
int zk_srs_commit_evaluations_batch(zk_srs* srs, size_t domain_size, const uint64_t* evals_mont, size_t k, uint64_t* out_xy);
int zk_srs_mask_custom(zk_srs* srs, const uint64_t* chunks_xy, size_t n_chunks, const uint64_t* blinders_mont,
                       size_t n_blinders, uint64_t* out_xy);

/* ------------------------------------------------------------------ IPA opening rounds, device resident (SRS::open, ipa.rs:929-1007)
 * The coefficients a and the evaluation vector b are uploaded once and folded in HBM; the bases are the resident SRS table
 * (`bases`, zk_bases_upload of srs.g) and are never folded: round j's commitments are MSMs over the original points with
 * scalars a[.] * b_poly_coefficients(u_1..u_j)[.] (commitment.rs:565-581).  The host keeps the Fiat-Shamir sponge and the
 * blinders.  Per round:
 *   zk_ipa_round_lr    out_l = <a_hi, g_lo>, out_r = <a_lo, g_hi> (Jacobian; the host adds rand*h + ip*u_base, ipa.rs:943-961),
 *                      out_ip_l = <a_hi, b_lo>, out_ip_r = <a_lo, b_hi> (Montgomery field elements)
 *   zk_ipa_round_fold  a <- a_lo + u_inv a_hi,  b <- b_lo + u b_hi,  g <- g_lo + [u] g_hi (implicitly)  (ipa.rs:980-1006,
 *                      u = u_pre.to_field(endo_r), Montgomery)
 * n = the SRS size rounded up to a power of two (the reference pads g with the identity, a and b with zero, ipa.rs:848-862).
 * zk_ipa_read copies the leading min(len, capacity) elements of the current a and b; after the last fold (len == 1) those are
 * a0 and b0, and out_g_xyz (optional, Jacobian) receives g0, the proof's `sg`.  `bases` must outlive the handle. */
typedef struct zk_ipa zk_ipa;
int zk_ipa_begin(zk_ctx* ctx, const zk_bases* bases, const uint64_t* a_mont, const uint64_t* b_mont, size_t n, zk_ipa** out);
void zk_ipa_free(zk_ipa* ipa);
size_t zk_ipa_len(const zk_ipa* ipa);
int zk_ipa_round_lr(zk_ipa* ipa, uint64_t out_l_xyz[12], uint64_t out_r_xyz[12], uint64_t out_ip_l[4], uint64_t out_ip_r[4]);
int zk_ipa_round_fold(zk_ipa* ipa, const uint64_t u_mont[4], const uint64_t u_inv_mont[4]);
int zk_ipa_read(zk_ipa* ipa, uint64_t* out_a, uint64_t* out_b, size_t capacity, uint64_t out_g_xyz[12]);
/* zk_points_fold_dev: the reference's per-round base fold g'[i] = g[i] + [u] g[h + i], i < h (G::combine_one_endo,
 * poly-commitment/src/ipa.rs:1002-1006, combine.rs:292-342) on device-resident affine points: d_g holds 2h points, d_out
 * receives h (may not alias d_g), u in Montgomery form of the scalar field.  Not used by zk_srs_open / zk_ipa_* (those never
 * fold the bases); kept as a parity-tested building block and as the measured alternative (DESIGN.md 4.4). */
int zk_points_fold_dev(zk_ctx* ctx, int curve_id, const void* d_g, size_t h, const uint64_t u_mont[4], void* d_out);

/* ------------------------------------------------------------------ SRS::open as one call (poly-commitment/src/ipa.rs:823-1061)
 * == <OpeningProof<G> as OpenProof<G>>::open(srs, group_map, plnms, elm, polyscale, evalscale, sponge, rng)  (ipa.rs:1193-1218).
 * Everything with arithmetic in it runs in the library: combine_polys (utils.rs:103-202: scaled accumulation of the batch, the
 * iFFT of the evaluation-form part, chunk linearisation), b_init (ipa.rs:876-888), the combined inner product (:891-896), the
 * log2 |g| folding rounds (:929-1007; h and U ride as two extra bases of every round's MSM pair exactly like the reference's
 * `[g_lo, &[self.h, u_base]].concat()`), r_prime, delta, z1, z2 (:1022-1052).  What stays with the caller is what the reference
 * keeps generic: the Fiat-Shamir sponge and the group map behind three callbacks, and the random scalars, passed in the order
 * the reference draws them (rand_l, rand_r per round, then d, r_delta).
 *
 * zk_open_poly: one entry of `plnms` — DensePolynomialOrEvaluations + the PolyComm of blinders (utils.rs:18-23, 84-94).
 *   data         Montgomery field elements: coefficients, or evaluations; host (pageable or page-locked) or DEVICE memory
 *   len          element count
 *   domain_size  0 = DensePolynomial; otherwise Evaluations over the domain of that size, len a multiple of it (stride = len /
 *                domain_size, utils.rs:151-158); every evaluation-form entry must use the same domain (the reference asserts)
 *   blinders     the chunks of the blinder commitment `p_i_comm` (Montgomery scalars), n_blinders of them
 * Callbacks return 0 on success; any other value aborts the call with ZK_ERR_INVALID. */
typedef struct zk_open_poly {
    const uint64_t* data;
    size_t len;
    size_t domain_size;
    const uint64_t* blinders;
    size_t n_blinders;
} zk_open_poly;
typedef struct zk_open_transcript {
    void* user;
    /* ipa.rs:898-910: sponge.absorb_fr(shift_scalar(combined_inner_product)); t = sponge.challenge_fq();
     * U = group_map.to_group(t).  in: combined_inner_product (Montgomery scalar); out: U, affine Montgomery */
    int (*u_base)(void* user, const uint64_t combined_inner_product[4], uint64_t out_u_xy[8]);
    /* ipa.rs:962-970: absorb_g(l), absorb_g(r); u = squeeze_prechallenge(sponge).to_field(endo_r).  out: u (Montgomery scalar) */
    int (*round)(void* user, unsigned round, const uint64_t l_xy[8], const uint64_t r_xy[8], uint64_t out_u[4]);
    /* ipa.rs:1040-1041: absorb_g(delta); c = ScalarChallenge(sponge.challenge()).to_field(endo_r).  out: c (Montgomery scalar) */
    int (*final_challenge)(void* user, const uint64_t delta_xy[8], uint64_t out_c[4]);
} zk_open_transcript;
/* rounds = ceil(log2 |g|).  rng_scalars: 2 * rounds + 2 Montgomery scalars (n_rng_scalars must say so).
 * out_lr_xy: rounds x 2 affine points (l_0, r_0, l_1, ...), capacity lr_capacity_rounds rounds; out_rounds receives rounds. */
int zk_srs_open(zk_srs* srs, const zk_open_poly* polys, size_t n_polys, const uint64_t* elm_mont, size_t n_elm,
                const uint64_t polyscale[4], const uint64_t evalscale[4], const uint64_t* rng_scalars, size_t n_rng_scalars,
                const zk_open_transcript* transcript, uint64_t* out_lr_xy, size_t lr_capacity_rounds, size_t* out_rounds,
                uint64_t out_delta_xy[8], uint64_t out_z1[4], uint64_t out_z2[4], uint64_t out_sg_xy[8]);

/* ------------------------------------------------------------------ d8 pipeline, first pointwise evaluator (SURVEY.md §8f row 3)
 * The permutation part of the quotient polynomial in evaluation form over d8 (m = 2^log_m points), all operands resident on the
 * device — kimchi/src/circuits/polynomials/permutation.rs:223-357, `perm`:
 *   out[i] = alpha0 * zkpm[i] * ( z[i] * prod_{k<7} (w_k[i] + gamma + beta * shift_k * x_i)
 *                               - z[(i + next_shift) mod m] * prod_{k<7} (w_k[i] + gamma + beta * sigma_k[i]) ),     x_i = omega_m^i
 * d_w[k]: the 7 permuted witness columns over d8 (the output of zk_ntt_dev_oop on the interpolated columns); d_sigma[k]:
 * permutation_coefficients8 (e.g. the sections of a cached prover index, zk_index_cache_section); d_z: z over d8; d_zkpm:
 * permutation_vanishing_polynomial_l
 * over d8; next_shift = m / n = 8 (z(x omega) is z shifted by eight positions of d8, constraints.rs:497-505); beta, gamma, alpha0
 * and the 7 shifts (cs.shift) are Montgomery scalars passed by value. */
int zk_perm_quotient_dev(zk_ctx* ctx, int field_id, unsigned log_m, const void* const d_w[7], const void* d_z,
                         const void* const d_sigma[7], const void* d_zkpm, const uint64_t beta[4], const uint64_t gamma[4],
                         const uint64_t alpha0[4], const uint64_t shifts[28], unsigned next_shift, void* d_out);

/* ------------------------------------------------------------------ constraint evaluator (kimchi's expression framework)
 * zk_expr_eval_dev replaces Expr::evaluations(&env) (kimchi/src/circuits/expr.rs:1938-2190; call sites kimchi/src/prover.rs:794-892:
 * every gate's combined constraint and the lookup constraints, evaluated over d4 or d8 and added into t4 / t8).  The expression is
 * passed in the reference's flat form, the RPN program of PolishToken (expr.rs:819-836, Expr::to_polish), and evaluated at every
 * point of the output domain by one kernel with the semantics of PolishToken::evaluate (expr.rs:856-940):
 *   ZK_EXPR_CONST k    push constants[k] — Literal, EndoCoefficient, Mds{row,col} and Challenge terms resolved by the caller
 *   ZK_EXPR_CELL c     push column (c & 0x7fffffff) at the current row, or the next row when bit 31 is set:
 *                      evals[(len / out_len * i + domain_mult * shift) % len]   (SubEvals indexing, expr.rs:1976-1982);
 *                      VanishesOnZeroKnowledgeAndPreviousRows and UnnormalizedLagrangeBasis are columns the caller supplies
 *   ZK_EXPR_DUP, ZK_EXPR_POW n, ZK_EXPR_ADD, ZK_EXPR_MUL, ZK_EXPR_SUB, ZK_EXPR_STORE, ZK_EXPR_LOAD k   as in the reference
 *   (SkipIf / SkipIfNot are resolved by the caller: the feature flags are known when the program is built)
 * Columns are device-resident arrays of Montgomery field elements over a domain `domain_mult` times d1 (len = domain_mult * |d1|,
 * at least as fine as the output domain); out_len = out_domain_mult * |d1|.  accumulate != 0 adds the result into d_out (t4 += / t8 +=,
 * prover.rs:876-882).  A program that would underflow the stack, leave more than one value, or index outside its tables is refused
 * with ZK_ERR_INVALID (ExprError::EmptyStack / the reference's assert) before anything runs; limits: stack 24, cache 96, 64 columns. */
enum { ZK_EXPR_CONST = 0, ZK_EXPR_CELL = 1, ZK_EXPR_DUP = 2, ZK_EXPR_POW = 3, ZK_EXPR_ADD = 4, ZK_EXPR_MUL = 5, ZK_EXPR_SUB = 6,
       ZK_EXPR_STORE = 7, ZK_EXPR_LOAD = 8 };
typedef struct zk_expr_token { uint32_t op; uint32_t arg; } zk_expr_token;
typedef struct zk_expr_column { const void* d_evals; uint64_t len; uint32_t domain_mult; uint32_t reserved; } zk_expr_column;
int zk_expr_eval_dev(zk_ctx* ctx, int field_id, const zk_expr_token* tokens, size_t n_tokens, const uint64_t* constants_mont,
                     size_t n_constants, const zk_expr_column* cols, size_t n_cols, uint64_t out_len, unsigned out_domain_mult,
                     int accumulate, void* d_out);

/* ------------------------------------------------------------------ the quotient's polynomial tail (kimchi/src/prover.rs:905-918)
 * zk_poly_add_dev                   dst[i] += src[i], i < len — `t4.interpolate() + t8.interpolate()`, `f += &public_poly`,
 *                                   `quotient += &bnd` on device-resident coefficient vectors (the shorter operand is `src`)
 * zk_poly_divide_by_vanishing_dev   DensePolynomial::divide_by_vanishing_poly(d1): f (len coefficients) = q (x^n - 1) + r, n = 2^log_n;
 *                                   writes the len - n coefficients of q to d_quot (nothing when len <= n: q = 0, r = f) and reports
 *                                   whether r == 0 — the prover's "rest of division by vanishing polynomial" check (prover.rs:910-914).
 *                                   d_quot may not alias d_f.  The quotient's chunks then go to zk_msm_dev as they lie. */
int zk_poly_add_dev(zk_ctx* ctx, int field_id, void* d_dst, const void* d_src, size_t len);
int zk_poly_divide_by_vanishing_dev(zk_ctx* ctx, int field_id, const void* d_f, size_t len, unsigned log_n, void* d_quot, int* remainder_is_zero);

/* ------------------------------------------------------------------ cached prover index (SURVEY.md §8f row 4)
 * Device-side ingestion of kimchi's mmap-backed proving-key cache, kimchi/src/cached_prover_index.rs:26-56 ("MINAPK01", format 3):
 * the file stores the index's big arrays — coefficients8 (15 columns), permutation_coefficients8 (7), the gate selectors over d4 / d8,
 * sid, the lookup tables — as raw Montgomery limbs, which is the device format, so the payload is copied to the device AS IT LIES in
 * the mapping (one copy, no per-element decoding) and then serves as resident operands (zk_perm_quotient_dev, zk_msm_dev ...).
 * image: the file's bytes (e.g. the mmap); expect_identifier: NULL or the identifier the file must carry (IdentifierMismatch).
 * Section tags are the reference's SectionTag values: 0x01 sid, 0x10 + i coefficients8[i], 0x20..0x25 selectors,
 * 0x30 + i permutation_coefficients8[i], 0x40..0x45 optional selectors, 0x50..0x56 lookup arrays. */
typedef struct zk_index_cache zk_index_cache;
typedef struct zk_index_header {      /* ScalarHeader + preamble fields, cached_prover_index.rs:173-225 */
    uint32_t public_inputs, prev_challenges;
    uint64_t zk_rows, max_poly_size, domain_d1_size;
    uint32_t feature_flags, optional_selectors_present, lookup_selectors_present, num_sections;
    int disable_gates_checks, has_verifier_index_digest;
    uint64_t endo[4], shift[7][4], verifier_index_digest[4];   /* Montgomery limbs */
    char identifier[512];
} zk_index_header;
int zk_index_cache_load(zk_ctx* ctx, const void* image, size_t image_len, const char* expect_identifier, zk_index_cache** out);
void zk_index_cache_free(zk_index_cache* cache);
int zk_index_cache_header(const zk_index_cache* cache, zk_index_header* out);
int zk_index_cache_section(const zk_index_cache* cache, uint32_t tag, const void** d_ptr, size_t* n_elems, uint32_t* elem_domain_size);

/* ------------------------------------------------------------------ diagnostics (tests/test_gpu_field.py, DESIGN.md compute model)
 * Element-wise device field ops on n elements (op: 0 mul, 1 add, 2 sub, 3 inverse of a), host pointers. */
int zk_debug_field_op(zk_ctx* ctx, int field_id, int op, const uint64_t* a, const uint64_t* b, uint64_t* out, size_t n);
/* Sustained Montgomery multiplications per second of the device (iters dependent fe_mul per thread, full grid). */
int zk_debug_mul_throughput(zk_ctx* ctx, int field_id, unsigned iters, double* out_mul_per_s);
/* Latency/throughput probe: kind 1, 2, 4 = that many independent dependent-chains of fe_mul per thread, 100 = a chain
 * of XYZZ mixed additions; blocks x threads grid (blocks 0 = 4 per SM); reports operations per second. */
int zk_debug_op_throughput(zk_ctx* ctx, int field_id, int kind, unsigned blocks, unsigned threads, unsigned iters,
                           double* out_ops_per_s);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* ZKB200_H */
