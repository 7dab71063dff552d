/* dot_ring_b200 -- C ABI of the B200-native ring-proof engine.
 *
 * This is the drop-in boundary for the hot path of Chainscore/dot-ring (SURVEY.md section 8b).  The
 * reference has no FFI of its own for this path: it crosses from Python into Cython
 * (dot_ring/ring_proof/polynomial/ntt.pyx, dot_ring/curve/native_field/bandersnatch_te.pyx) and into
 * the SWIG bindings of blst (dot_ring/ring_proof/pcs/kzg.py).  Each entry point below names the
 * reference interface it replaces (file:line in the reference tree).  INTEGRATION.md shows the ctypes
 * stubs a dot-ring maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; caller owns every byte buffer; handles own device memory.
 *   - encodings are the reference's wire encodings: Fr 32-byte little-endian canonical; G1 96-byte
 *     uncompressed / 48-byte compressed zcash big-endian; Bandersnatch points 32 bytes
 *     (y little-endian, x-sign in bit 7 of the last byte).
 *   - return value 0 on success, negative error code otherwise; dr_last_error() gives the message
 *     (thread-local).  DR_EINVAL corresponds to the reference raising ValueError.  A cryptographically
 *     invalid proof is a verdict (0/1 in an output array), never an error.
 *   - one dr_ctx per GPU; calls on one ctx are serialised by the caller; calls are synchronous at the
 *     ABI and asynchronous inside (one CUDA stream per ctx).
 */
#ifndef DOT_RING_B200_H
#define DOT_RING_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DR_OK 0
#define DR_EINVAL (-1) /* malformed encoding / bad argument (reference: ValueError) */
#define DR_ECUDA (-2)  /* CUDA runtime failure */
#define DR_ENOMEM (-3)
#define DR_ESTATE (-4) /* handle used in the wrong state */

typedef struct dr_ctx dr_ctx;
typedef struct dr_srs dr_srs;
typedef struct dr_ring dr_ring;

const char* dr_last_error(void);
const char* dr_version(void);
/* 1 when built for the GPU (nvcc, sm_100a); 0 for the CPU emulation build used only by tests/host. */
int dr_is_cuda_build(void);

/* CUDA devices visible to this process (one dr_ctx per device; dot_ring_b200.engine.EnginePool shards batches over them). */
int dr_device_count(void);

/* ---- context ------------------------------------------------------------------------------- */
int dr_ctx_create(int device, dr_ctx** out);
void dr_ctx_destroy(dr_ctx* ctx);
int dr_ctx_sync(dr_ctx* ctx);
/* Device scratch freed by earlier calls is kept for reuse (up to 24 GB per process); this returns it to the driver. */
int dr_ctx_trim(dr_ctx* ctx);
/* Device-side timing with CUDA events on the ctx stream (bench.py): start, then stop -> ms. */
int dr_ctx_timer_start(dr_ctx* ctx);
int dr_ctx_timer_stop(dr_ctx* ctx, float* ms_out);
/* Number of kernels this library has launched in this process (bench.py "gpu_launches"). */
uint64_t dr_launch_count(void);
/* Device properties for reports: name into buf, returns SM count (0 in emulation). */
int dr_ctx_device_info(dr_ctx* ctx, char* name_buf, size_t name_len, int* sm_count, int* sm_clock_khz, size_t* free_bytes, size_t* total_bytes);

/* ---- SRS + KZG commit ------------------------------------------------------------------------
 * Replaces dot_ring/ring_proof/pcs/srs.py:98-148 (SRS, `blst.P1_Affines.as_memory`) and
 * dot_ring/ring_proof/pcs/kzg.py:152-175 (`KZG.commit` -> `blst.P1_Affines.mult_pippenger`).
 * g1_be96: n_g1 uncompressed points [tau^i]_1; g2_be192: [1]_2 and [tau]_2 (srs.py:57-88 layout).
 * window_bits selects the fixed-base table: bits 0..7 = c, the window width (2..15; c + 1 <= 16); bits 8..15 = k, how many of the low windows
 * take c + 1 bits instead (0 = uniform).  W = ceil((256 - k) / c) table additions per coefficient, table bytes =
 * n_g1 * (W + k) * 2^(c-1) * 96.  Bit 16 = GLV: every scalar is split as k1 + k2 * lambda (128-bit halves, lambda the eigenvalue of
 * the G1 endomorphism), the table covers 128 bits (W = ceil((128 - k) / c), c up to 16, a slightly longer last window) and a
 * coefficient costs 2W additions: c = 16 gives 16 additions in 161 GB for 6145 points.  0 = auto: that GLV table when it leaves 14 GB of the
 * free device memory (a 180 GB B200 with the bundled 6145-point SRS), else c = 14, k = 4 (18 additions, 106 GB) when that leaves max(24 GB, a
 * quarter of its size), else the widest uniform windows that do (uniform 14 bits = 19 additions, 92 GB).
 */
int dr_srs_load(dr_ctx* ctx, const uint8_t* g1_be96, size_t n_g1, const uint8_t* g2_be192, int window_bits, dr_srs** out);
void dr_srs_destroy(dr_srs* srs);
size_t dr_srs_size(const dr_srs* srs);
size_t dr_srs_table_bytes(const dr_srs* srs);
/* The table geometry in use: window width c, number of (c + 1)-bit windows, GLV split (0 / 1), table additions per coefficient. */
void dr_srs_geometry(const dr_srs* srs, uint32_t* window_bits, uint32_t* wide_windows, uint32_t* glv, uint32_t* additions);
/* `batch` polynomials of n coefficients each (coefficient j of polynomial b at coeffs_le32 + 32*(b*n+j));
 * values >= r are reduced (kzg.py passes unreduced quotient coefficients, ops.py:215-220); all-zero ->
 * infinity (kzg.py:167-168).  Output: batch x 96-byte uncompressed commitments. */
int dr_kzg_commit(dr_ctx* ctx, dr_srs* srs, const uint8_t* coeffs_le32, size_t n, size_t batch, uint8_t* out_be96);
/* `KZG.open` (dot_ring/ring_proof/pcs/kzg.py:178-191 over `synthetic_div_with_eval`, pcs/utils.py:27-35) for `batch` polynomials of n >= 1
 * coefficients: values_le32[b] = f_b(x_b) and proofs_be96[b] = commit((f_b - f_b(x_b)) / (X - x_b)), the quotient committed like dr_kzg_commit. */
int dr_kzg_open(dr_ctx* ctx, dr_srs* srs, const uint8_t* coeffs_le32, size_t n, size_t batch, const uint8_t* points_le32, uint8_t* proofs_be96, uint8_t* values_le32);
/* The pairing equation every KZG verifier of the reference ends in (pcs/kzg.py:194-338: `verify`, `batch_verify`,
 * `batch_verify_linear_preconverted` after their random linear combination):
 *   *ok = ( e(sum_i lhs_scalars[i] * lhs_points[i], [1]_2) == e(sum_j rhs_scalars[j] * rhs_points[j], [tau]_2) )
 * with [1]_2, [tau]_2 the G2 points of `srs`.  Points 96-byte uncompressed, scalars 32-byte little-endian (reduced mod r here).
 * Replaces the two `mult_pippenger` calls + `blst_miller_loop` x 2 + `blst_final_verify` (pcs/pairing.py:24-31). */
int dr_kzg_pairing_check(dr_ctx* ctx, dr_srs* srs, const uint8_t* lhs_points_be96, const uint8_t* lhs_scalars_le32, size_t n_lhs, const uint8_t* rhs_points_be96,
                         const uint8_t* rhs_scalars_le32, size_t n_rhs, int* ok);
/* How the table entries of a commitment are summed: 0 = XYZZ mixed additions (10 multiplications each), 1 = batched-affine
 * pairing rounds (one inversion per round of independent additions, ~6.3 multiplications each) for polynomials long enough to
 * fill a round.  Same group element either way; tests cross-check the two. */
int dr_ctx_set_commit_mode(dr_ctx* ctx, int mode);
/* Same with operands already resident on the device (Montgomery limbs); used for roofline timing. */
int dr_kzg_commit_bench(dr_ctx* ctx, dr_srs* srs, size_t n, size_t batch, int iters, uint64_t seed, float* ms_per_iter, uint8_t* out_first_be96);

/* ---- variable-base G1 MSM ---------------------------------------------------------------------------------
 * Replaces `KZG.msm_g1` = `blst.P1_Affines.mult_pippenger(points, scalars)` (dot_ring/ring_proof/pcs/kzg.py:147-149) for point sets
 * that are not the fixed SRS: sum_i (k_i mod r) * P_i by the bucket method (signed windows, counting sort by bucket, work units
 * bounded per thread, segmented bucket reduction).  points: n x 96-byte uncompressed; scalars: n x 32-byte little-endian.
 * dr_g1_msm_bench times the same pipeline with operands resident on the device over the synthetic SRS P_i = tau^i * G
 * (distribution 0: uniform scalars from splitmix64(seed), 1: all ones, 2: random bits), so the result is checkable as
 * (sum_i k_i tau^i) * G at any size. */
int dr_g1_msm(dr_ctx* ctx, const uint8_t* points_be96, const uint8_t* scalars_le32, size_t n, uint8_t out_be96[96]);
/* n points tau^(offset + i) * G, i < n, as 96-byte uncompressed encodings (synthetic SRS slices for sizes the bundled 6145-point
 * SRS does not cover: the 2^11 .. 2^20 sweep and MSMs split by point range across GPUs). */
int dr_g1_synthetic_srs(dr_ctx* ctx, const uint8_t tau_le32[32], size_t offset, size_t n, uint8_t* out_be96);
int dr_g1_msm_bench(dr_ctx* ctx, size_t n, int iters, uint64_t seed, int distribution, const uint8_t tau_le32[32], float* ms_per_iter, uint32_t* window_bits,
                    uint8_t out_be96[96]);

/* ---- G1 codecs -------------------------------------------------------------------------------
 * Replaces kzg.py:121-144 (`compress_g1`, `serialize_g1_uncompressed`, `decompress_g1`).
 * ok[i] = 0 marks a malformed encoding (reference: ValueError("invalid BLS12-381 G1 encoding")). */
int dr_g1_compress(dr_ctx* ctx, const uint8_t* in_be96, size_t count, uint8_t* out_be48);
int dr_g1_decompress(dr_ctx* ctx, const uint8_t* in_be48, size_t count, uint8_t* out_be96, uint8_t* ok);

/* ---- Fr NTT ------------------------------------------------------------------------------------
 * Replaces `BlsScalarNTTPlan.transform/transform_scaled` (ring_proof/polynomial/ntt.pyx:104-163) behind
 * `inverse_fft` / `evaluate_poly_fft` (ring_proof/polynomial/fft.py:87-144): natural order in and out,
 * out[k] = scale * sum_j in[j] * omega^(j*k).  inverse != 0 uses omega^-1 and scale 1/n.
 * data_le32: batch x n elements, transformed in place.  n is a power of two, 2 <= n <= 2^22 (the reference's plans stop at 4096). */
int dr_fr_ntt(dr_ctx* ctx, uint8_t* data_le32, size_t n, size_t batch, int inverse, const uint8_t omega_le32[32]);
/* Same transform with operands resident on the device (`batch` pseudo-random vectors, `iters` forward transforms): ms per
 * iteration for the HBM / integer roofline of the NTT passes.  n <= 4096: one CTA per transform in shared memory; larger n
 * (up to 2^22, e.g. the 2^16 / 2^18 domains of a 65k-key ring): two passes n = n1 * n2 through HBM. */
int dr_fr_ntt_bench(dr_ctx* ctx, size_t n, size_t batch, int iters, const uint8_t omega_le32[32], float* ms_per_iter, uint8_t first_le32[32]);

/* ---- ring: key ingestion, fixed columns, ring root ---------------------------------------------------
 * Replaces `Ring.__init__` (dot_ring/vrf/ring/members.py:22-55: per-key decode + subgroup check, padding,
 * blinding-base powers) and `RingRoot.from_ring` (dot_ring/vrf/ring/root.py:21-44,133-173: three
 * iNTT(N) + three KZG commits) plus the per-ring constants the prover re-derives on every call in the
 * reference (constraints.py:43-62: 4x LDE of px, py, s, L_0, L_{N-4}).
 * All field elements are 32-byte little-endian canonical; points are affine (x | y). */
typedef struct dr_ring_params {
    uint32_t domain_size;      /* N (params.py:119); a power of two in [512, 65536] */
    uint32_t max_ring_size;    /* params.py:120 */
    uint32_t padding_rows;     /* must be 4 (params.py:196-197) */
    uint32_t suite_id_len;
    uint32_t h2c_dst_len;
    uint32_t hash_id;          /* suite hash: 0 = SHA-512 (Bandersnatch-SHA512-ELL2-v1), 1 = SHAKE128 (Bandersnatch-SHAKE128-ELL2-v1) */
    uint8_t omega[32];         /* params.omega: primitive N-th root of unity */
    uint8_t radix_omega[32];   /* params.radix_omega: primitive 4N-th root (sqrt-extended for 4N > 2048) */
    uint8_t seed[64];          /* accumulator_base */
    uint8_t blinding_base[64];
    uint8_t padding_point[64];
    uint8_t generator[64];
    uint8_t suite_id[32];      /* e.g. "Bandersnatch-SHA512-ELL2-v1" */
    uint8_t h2c_dst[64];       /* hash-to-curve DST, e.g. suite_id | 0x60 */
} dr_ring_params;

int dr_ring_create(dr_ctx* ctx, dr_srs* srs, const dr_ring_params* params, const uint8_t* keys32, size_t n_keys, dr_ring** out);
void dr_ring_destroy(dr_ring* ring);
/* 144-byte ring root = compress(C_px) | compress(C_py) | compress(C_s)  (root.py:74-87). */
int dr_ring_root(dr_ring* ring, uint8_t root144[144]);
/* Uncompressed fixed commitments (3 x 96 bytes) as absorbed by the verifier key (root.py:54-71). */
int dr_ring_fixed_commitments(dr_ring* ring, uint8_t out288[288]);
/* `Ring.nm_points` (members.py:55): N affine points, x | y little-endian (64 bytes each). */
int dr_ring_points(dr_ring* ring, uint8_t* out_xy64, size_t n_points);

/* ---- Ring VRF prove, batched -----------------------------------------------------------------------
 * Replaces `RingVRF[Bandersnatch].prove` (dot_ring/vrf/ring/vrf.py:185-209) = `PedersenVRF.prove`
 * (vrf/pedersen/vrf.py:86-126) + `RingProofBuilder.build` (ring_proof/proof_builder.py:38-142) for n
 * independent (alpha, ad, secret key, producer index) items against one ring.
 *   blob / offsets: item i has alpha = blob[alpha_off[i] .. +alpha_len[i]) and ad likewise;
 *   secret_keys32: n x 32-byte little-endian scalars; producer_index[i]: row of pk(sk_i) in the ring;
 *   zk_rows: n x 12 x 32 bytes replacing the reference's `secrets.randbelow` draws in column order
 *            b, acc_x, acc_y, acc_ip (columns.py:43-53,153-161), or NULL for test_vectors=True (zeros);
 *   proofs784: n x 784 bytes (192-byte Pedersen part | 592-byte ring payload);
 *   status[i]: 0 ok, non-zero when sk_i does not own ring row producer_index[i] (reference: ValueError). */
int dr_ring_prove_batch(dr_ctx* ctx, dr_ring* ring, size_t n, const uint8_t* blob, const uint32_t* alpha_off, const uint32_t* alpha_len,
                        const uint32_t* ad_off, const uint32_t* ad_len, const uint8_t* secret_keys32, const uint32_t* producer_index,
                        const uint8_t* zk_rows, uint8_t* proofs784, uint32_t* status);
/* ---- Ring VRF prove, one batch over several rings ------------------------------------------------------------
 * Batches `RingVRF[Bandersnatch].prove` (dot_ring/vrf/ring/vrf.py:185-209) over items that belong to different rings: item i is
 * proved against rings[ring_index[i]], and producer_index[i] is a row of that ring.  blob / offsets, secret_keys32, zk_rows (NULL:
 * zeros), proofs784 and status[i] (non-zero when sk_i does not own that row of that ring) are as in dr_ring_prove_batch, and each
 * proof equals dr_ring_prove_batch of its own ring on the same item.  Domain sizes may differ: items are grouped by domain size,
 * every group runs its own equal-width passes, and the results land in the caller's order.  The rings share one pass, so a batch
 * spread over K rings costs one call's fixed latency instead of K.  n == 0 returns DR_OK.  DR_EINVAL when a ring belongs to another
 * context, when the rings use different dr_srs handles, differ in suite (id, DST, hash, generator, blinding base, accumulator seed,
 * padding point) or, at one domain size, in omega / radix_omega, when an index is out of range, or when n > 0 and n_rings == 0. */
int dr_ring_prove_multi(dr_ctx* ctx, dr_ring* const* rings, size_t n_rings, const uint32_t* ring_index, size_t n, const uint8_t* blob,
                        const uint32_t* alpha_off, const uint32_t* alpha_len, const uint32_t* ad_off, const uint32_t* ad_len, const uint8_t* secret_keys32,
                        const uint32_t* producer_index, const uint8_t* zk_rows, uint8_t* proofs784, uint32_t* status);
/* ---- bare ring proofs from a caller's blinding factor ---------------------------------------------------------------
 * Replaces `RingProofBuilder(...).build()` (dot_ring/ring_proof/proof_builder.py:38-142) alone, without `PedersenVRF.prove`: item i proves
 * that relation_i = PK_k + t_i * B for row k = producer_index[i] of rings[ring_index[i]], with the caller's blinding factor
 * t_i = blinding_le32[i] (e.g. what dr_pedersen_prove_batch_ex returns, or a fresh one for a plain anonymous-membership proof).
 *   relations_xy64[i]: PK_k + t_i * B, affine x | y, 32-byte little-endian each (the layout dr_ring_proof_verify_batch reads);
 *   payloads592[i]: the 592-byte ring-proof payload (proof_payload.py:68-91);
 *   zk_rows: 12 x 32 bytes per item as in dr_ring_prove_batch, NULL for zeros;
 *   label: the transcript label; NULL or label_len == 0 means the rings' suite id (what dr_ring_prove_batch absorbs), otherwise the
 *          transcript starts as RingRoot.verifier_transcript_prefix(label) does: label, "vk", [1]_1, [1]_2 | [tau]_2 and the three fixed
 *          commitments (e.g. "w3f-ring-proof-test" for w3f ring-proof verifiers).  label_len <= 32, as in dr_verifier_key.
 * The ring, SRS and suite rules of dr_ring_prove_multi apply unchanged, and results land in the caller's order.  Any row below
 * max_ring_size is proved against the point that row holds (there is no secret key to check it against, so no status word).
 * n == 0 returns DR_OK.  DR_EINVAL when a blinding factor is not below the Bandersnatch subgroup order, producer_index[i] >=
 * max_ring_size of its ring, label_len > 32, or a check of dr_ring_prove_multi fails.  dr_ring_prove_phase_ms and
 * dr_ring_prove_commit_kernel_ms report this call as they report dr_ring_prove_multi. */
int dr_ring_proof_prove_multi(dr_ctx* ctx, dr_ring* const* rings, size_t n_rings, const uint32_t* ring_index, size_t n, const uint32_t* producer_index,
                              const uint8_t* blinding_le32, const uint8_t* zk_rows, const uint8_t* label, size_t label_len, uint8_t* relations_xy64,
                              uint8_t* payloads592);
/* Per-phase device time of the last dr_ring_prove_batch / dr_ring_prove_multi on this ctx (ms, the whole call, summed over its
 * domain groups): [0] pedersen+witness, [1] interpolate, [2] commits (all MSMs), [3] LDE+constraints+quotient, [4] evaluations+openings
 * polys, [5] transcripts+assembly. */
int dr_ring_prove_phase_ms(dr_ctx* ctx, float out[6]);
/* Device time (CUDA events on the ctx stream, around the launches only) and launch count of the dominant kernel, the dense fixed-base
 * commit `CommitBodyT`, within the last dr_ring_prove_batch / dr_ring_prove_multi on this ctx (summed over its domain groups): 3
 * launches per pass (quotient + two openings). */
int dr_ring_prove_commit_kernel_ms(dr_ctx* ctx, float* ms, uint32_t* launches);
/* Window width of the table the sparse witness commitments of this ring read (built at the first proof; 0 before that). */
uint32_t dr_ring_witness_table_bits(const dr_ring* ring);
/* Proofs processed per internal pass (bounds device scratch: about 1 KiB * domain_size per proof). 0 = default 1024. */
int dr_ctx_set_prove_chunk(dr_ctx* ctx, size_t chunk);
/* Witness-column commitments (columns.py:29-60,153-161) are computed from the evaluation form over Lagrange prefix-sum bases
 * (~130 non-zero terms per column instead of N); enabled != 0 switches to the reference's route, KZG.commit of the interpolated
 * coefficients.  Both give the same group element, hence identical proofs (tests cross-check the two). */
int dr_ctx_set_dense_witness_commit(dr_ctx* ctx, int enabled);
/* Domains above 4096 (the reference stops there, params.py:172-173; dr_ring_create accepts up to 2^16 when the SRS has 3N+1 points)
 * cannot use the single-CTA transforms: evaluations are materialised, cosets twisted element-wise and the two-pass NTT runs in
 * between.  enabled != 0 forces that route at any domain size so that tests can compare it with the fused kernels. */
int dr_ctx_set_generic_ntt_path(dr_ctx* ctx, int enabled);

/* ---- batched Bandersnatch point operations -------------------------------------------------------------
 * dr_te_decode_batch replaces `dec_point` (dot_ring/vrf/codec.py:39-45) / `CurvePoint.string_to_point`
 * (dot_ring/curve/point.py:178-214): ok[i] = 0 <=> the reference raises ValueError; checked != 0 adds the
 * non-identity prime-subgroup test of `Curve.valid_point` (dot_ring/curve/curve.py:56-67).
 * dr_te_mul_batch replaces `BandersnatchPoint.__mul__` (dot_ring/curve/specs/bandersnatch.py:177-191):
 * out[i] = (scalars[i] mod order) * points[i] (or points[0] when n_points == 1). */
int dr_te_decode_batch(dr_ctx* ctx, const uint8_t* in32, size_t n, int checked, uint8_t* out_xy64, uint8_t* ok);
int dr_te_mul_batch(dr_ctx* ctx, const uint8_t* points32, size_t n_points, const uint8_t* scalars32, size_t n, uint8_t* out32, uint8_t* ok);
/* dr_te_msm replaces `BandersnatchPoint.msm` (dot_ring/curve/specs/bandersnatch.py:194-286; native signed Pippenger at
 * native_field/bandersnatch_te.pyx:257-418): out = sum_i (scalars[i] mod order) * points[i], 32-byte encodings. */
int dr_te_msm(dr_ctx* ctx, const uint8_t* points32, const uint8_t* scalars32, size_t n, uint8_t out32[32]);

/* ---- VRF verification, batched -------------------------------------------------------------------------------
 * Item i: input = blob[in_off[i] .. +in_len[i]) (salt | alpha), ad = blob[ad_off[i] .. +ad_len[i]).
 * verdict[i]: 1 valid, 0 invalid, 2 malformed (the reference raises ValueError while decoding: bad length is the
 * caller's business, bad point / non-canonical scalar is reported here).
 * dr_pedersen_verify_batch replaces `PedersenVRF.decode` + `.verify` (dot_ring/vrf/pedersen/vrf.py:48-73,128-143) per item and, as
 * the conjunction of the verdicts, `PedersenVRF.batch_verify` (:171-242).  proofs192: O | Ybar | R | Ok | s | sb.
 * dr_tiny_verify_batch replaces `TinyVRF.decode` + `.verify` (dot_ring/vrf/ietf/tiny.py:46-83).  proofs80: O | c (16) | s. */
typedef struct dr_vrf_suite {
    uint32_t suite_id_len;
    uint32_t h2c_dst_len;
    uint32_t hash_id;          /* 0 = SHA-512 suite, 1 = SHAKE128 suite (specs/bandersnatch.py:48-144) */
    uint32_t pad;
    uint8_t suite_id[32];
    uint8_t h2c_dst[64];
    uint8_t generator[64];     /* affine x | y, 32-byte little-endian each */
    uint8_t blinding_base[64];
} dr_vrf_suite;
int dr_pedersen_verify_batch(dr_ctx* ctx, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                             const uint32_t* ad_len, const uint8_t* proofs192, uint8_t* verdict);
int dr_tiny_verify_batch(dr_ctx* ctx, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                         const uint32_t* ad_len, const uint8_t* public_keys32, const uint8_t* proofs80, uint8_t* verdict);

/* Thin VRF (dot_ring/vrf/ietf/thin.py:38-152): proofs96 = O | R | s.  dr_thin_verify_batch replaces `ThinVRF.decode` + `.verify` per item and,
 * as the conjunction of the verdicts, `ThinVRF.batch_verify`; dr_thin_prove_batch replaces `ThinVRF.prove`. */
int dr_thin_verify_batch(dr_ctx* ctx, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                         const uint32_t* ad_len, const uint8_t* public_keys32, const uint8_t* proofs96, uint8_t* verdict);
int dr_thin_prove_batch(dr_ctx* ctx, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                        const uint32_t* ad_len, const uint8_t* secret_keys32, uint8_t* proofs96);

/* Batched provers for the two plain schemes: `PedersenVRF.prove` (dot_ring/vrf/pedersen/vrf.py:86-126) and `TinyVRF.prove`
 * (dot_ring/vrf/ietf/tiny.py:35-70); nonces are the reference's deterministic transcript nonces (primitives.py:66-82). */
int dr_pedersen_prove_batch(dr_ctx* ctx, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                            const uint32_t* ad_len, const uint8_t* secret_keys32, uint8_t* proofs192);
/* Same, also returning the blinding factor of every proof (`PedersenVRF._blinding_factor`, vrf/pedersen/vrf.py:111-126,144-162) as
 * n x 32 little-endian bytes when blinding32 != NULL (what `verify_unblinding` is later given). */
int dr_pedersen_prove_batch_ex(dr_ctx* ctx, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len,
                               const uint32_t* ad_off, const uint32_t* ad_len, const uint8_t* secret_keys32, uint8_t* proofs192, uint8_t* blinding32);
int dr_tiny_prove_batch(dr_ctx* ctx, const dr_vrf_suite* suite, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                        const uint32_t* ad_len, const uint8_t* secret_keys32, uint8_t* proofs80);

/* ---- ring-proof verification ------------------------------------------------------------------------------------
 * dr_ring_proof_verify_batch replaces `Verify(...).is_valid()` (dot_ring/ring_proof/verify.py:213-324: payload decode,
 * `derive_challenges_after_vk`, `_compute_quotient_and_linearization_terms`, `linear_pcs_verifications`) followed by
 * `KZG.batch_verify_linear_preconverted` (pcs/kzg.py:56-108,304-338) for n (relation point, 592-byte payload) pairs under
 * one verifier key.  coeffs_le32: 2n canonical non-zero Fr values, the random batching coefficients the reference draws in
 * `_random_nonzero_coefficients` (the caller owns the randomness; (1, r) per proof for independent checks).
 * aggregate == 0: one pairing check per proof, verdict[i] as above.  aggregate != 0: all proofs folded into one check
 * (`RingVRF.batch_verify`, vrf/ring/vrf.py:239-283); verdict[i] then only reports decode / Pedersen status, *all_ok the result.
 * dr_ring_verify_batch = `RingVRF.decode` + `RingVRF.verify` / `batch_verify` (vrf/ring/vrf.py:60-93,226-283): Pedersen part +
 * ring proof with the relation Ybar against the verifier key of `ring` (the caller compares ring roots, root.py:111-112). */
typedef struct dr_verifier_key {
    uint32_t domain_size;
    uint32_t label_len;
    uint8_t label[32];         /* transcript label, e.g. the suite id or "w3f-ring-proof-test" */
    uint8_t omega[32];
    uint8_t seed[64];          /* accumulator base, affine x | y */
    uint8_t g1_0_be96[96];     /* [1]_1 */
    uint8_t g2_be192[384];     /* [1]_2, [tau]_2 uncompressed */
    uint8_t fixed_be96[288];   /* C_px, C_py, C_s uncompressed */
} dr_verifier_key;
int dr_ring_proof_verify_batch(dr_ctx* ctx, const dr_verifier_key* key, size_t n, const uint8_t* relations_xy64, const uint8_t* payloads592, const uint8_t* coeffs_le32,
                               int aggregate, uint8_t* verdict, int* all_ok);
int dr_ring_verify_batch(dr_ctx* ctx, dr_ring* ring, size_t n, const uint8_t* blob, const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off,
                         const uint32_t* ad_len, const uint8_t* proofs784, const uint8_t* coeffs_le32, int aggregate, uint8_t* verdict, int* all_ok);

/* ---- ring verification from ring roots -------------------------------------------------------------------------
 * A verifier needs nothing of a ring but its root (the fixed commitments): `Verify(...)` runs on them alone (verify.py:213-324), and
 * RingRoot.matches_ring (root.py:111-112) is the only use the reference makes of the keys.  A dr_ring_verifier is the verifier key of
 * one ring, built from its 144-byte root = compress(C_px) | compress(C_py) | compress(C_s) (root.py:74-87): no keys, no SRS handle,
 * no window table.  params: domain_size, omega, seed, generator, blinding_base, suite_id, h2c_dst, hash_id are read (the rest of
 * dr_ring_params is ignored); g1_0_be96 = [1]_1, g2_be192 = [1]_2 | [tau]_2 as in dr_srs_load.  DR_EINVAL where RingRoot.decode raises
 * (any of the three encodings rejected as by dr_g1_decompress) or on bad params; domain_size as in dr_ring_create.  Decoding checks no
 * subgroup (blst); a commitment on the curve but outside G1 is tested once here and then multiplied exactly.
 * dr_ring_verify_multi is dr_ring_verify_batch for a batch whose item i is checked against verifiers[verifier_index[i]], with the same
 * blob / offsets / proofs / coefficients / verdict / all_ok conventions; domain sizes may differ between the verifiers.
 * aggregate != 0 folds ALL items, whatever their ring, into one pairing check (rings over one SRS share [1]_2 and [tau]_2).
 * DR_EINVAL when a verifier belongs to another context, when the verifiers differ in suite (id, DST, hash, generator, blinding base),
 * in [1]_1 or in the G2 points, or when an index is out of range. */
typedef struct dr_ring_verifier dr_ring_verifier;
int dr_ring_verifier_create(dr_ctx* ctx, const dr_ring_params* params, const uint8_t* g1_0_be96, const uint8_t* g2_be192, const uint8_t root144[144],
                            dr_ring_verifier** out);
void dr_ring_verifier_destroy(dr_ring_verifier* v);
int dr_ring_verify_multi(dr_ctx* ctx, dr_ring_verifier* const* verifiers, size_t n_verifiers, const uint32_t* verifier_index, size_t n, const uint8_t* blob,
                         const uint32_t* in_off, const uint32_t* in_len, const uint32_t* ad_off, const uint32_t* ad_len, const uint8_t* proofs784,
                         const uint8_t* coeffs_le32, int aggregate, uint8_t* verdict, int* all_ok);

/* ---- ring roots from keys, and their updates -------------------------------------------------------------------------
 * The 144-byte ring root of a key vector without a dr_ring: `RingRoot.from_ring(Ring(keys))` (dot_ring/vrf/ring/members.py:22-55,
 * root.py:21-44,133-173) = compress(C_px) | compress(C_py) | compress(C_s) of the public vector PK || padding || 2^i B || 4 zero rows,
 * keys mapped as dr_ring_create maps them (undecodable / identity / out-of-subgroup -> padding point).  Equal to dr_ring_root of
 * dr_ring_create on the same keys, params and SRS G1 points, but `srs` needs only N points (not 3N + 1), may have any window geometry,
 * and its G2 points are not used; nothing of the prover's ring (LDEs, verifier key, transcript) is built.
 * params: domain_size, max_ring_size, padding_rows, omega, blinding_base, padding_point are read; the rest is ignored.
 * dr_ring_roots_from_keys: ring k's keys are the next key_counts[k] 32-byte keys of keys32 after those of the rings before it; all rings
 * share `params`; roots144 receives n_rings roots.  One call decodes every key, transforms and commits every ring's columns in batches.
 * dr_ring_root_update: the root of the key vector in which row rows[j] held old_keys32[j] (NULL: every listed row held padding, an
 * append) and now holds new_keys32[j], from root144 alone.  Old and new keys are mapped by the same rule (a new key that does not
 * decode nulls the row); C_s does not change.  n == 0 copies the input root after the checks.  out_root144 may alias root144.
 * DR_EINVAL: a check of dr_ring_create on N, padding_rows, max_ring_size or omega fails; key_counts[k] > max_ring_size; the SRS has
 * fewer than N points or belongs to another context; a row >= max_ring_size or a row listed twice; root144 does not decode (as
 * RingRoot.decode); the root's C_s is not the C_s of these params and this SRS (a root built for other params or another SRS).
 * A commitment that sums to infinity is encoded as dr_g1_compress encodes infinity. */
int dr_ring_roots_from_keys(dr_ctx* ctx, dr_srs* srs, const dr_ring_params* params, size_t n_rings, const uint8_t* keys32, const uint32_t* key_counts,
                            uint8_t* roots144);
int dr_ring_root_update(dr_ctx* ctx, dr_srs* srs, const dr_ring_params* params, const uint8_t root144[144], size_t n, const uint32_t* rows,
                        const uint8_t* old_keys32, const uint8_t* new_keys32, uint8_t out_root144[144]);

/* Aggregated batches of at least `n` proofs fold the two sides with two variable-base MSMs instead of 13 scalar multiplications
 * per proof (default 8192; same verdicts, tests lower it to exercise the path on small batches). */
int dr_ring_verify_set_msm_threshold(size_t n);

/* Tiny / Thin / Pedersen batches below `n` items (default 8192) run the eight-lane cooperative kernels (3 - 4x lower latency per item),
 * larger ones the one-thread-per-item kernels (higher throughput); same verdicts, tests drive both through this knob. */
int dr_vrf_verify_set_coop_threshold(size_t n);

/* ---- pairing check ------------------------------------------------------------------------------------------
 * Replaces `blst_miller_loop` + `blst_final_verify` (dot_ring/ring_proof/pcs/pairing.py:24-31) for a batch:
 * equal[i] = ( e(a1_i, b1_i) == e(a2_i, b2_i) ), G1 as 96-byte and G2 as 192-byte zcash uncompressed encodings
 * (x.c1 | x.c0 | y.c1 | y.c0, srs.py:80-88).  DR_EINVAL on a malformed point. */
int dr_pairing_check_batch(dr_ctx* ctx, const uint8_t* a1_be96, const uint8_t* b1_be192, const uint8_t* a2_be96, const uint8_t* b2_be192, size_t n, uint8_t* equal);

/* ---- arithmetic-layer self test + integer-pipe ceilings ----------------------------------------
 * dr_field_op: element-wise Montgomery arithmetic on the device (reference equivalent:
 * dot_ring/curve/native_field/scalar.pyx:12-165 `Scalar`, tested by tests/test_curve_ops/test_native_field.py).
 * field: 0 = BLS12-381 Fq (48-byte big-endian), 1 = Fr, 2 = Bandersnatch scalar field (32-byte
 * little-endian).  op: 0 mul, 1 add, 2 sub, 3 inv(a), 4 sqr(a), 5 neg(a).
 * dr_microbench: whole-chip ops/s of kind 0 IMAD, 1 IMAD.WIDE, 2 Fq mul, 3 Fr mul, 4 G1 mixed add, 5 DFMA, 6 IMAD + DFMA interleaved 2 : 1 (is the
 * FP64 pipe free next to the integer pipe?); 7 / 8: one dependent Fr / Fq squaring chain per warp with one warp per SM (the latency the
 * one-thread-per-item kernels pay), 9 / 10: the same for inversions; 11 / 12: Fq / Fr squaring throughput.  ops/s / (32 x SM count) is then the rate of ONE chain. */
int dr_field_op(dr_ctx* ctx, int field, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t count);
int dr_microbench(dr_ctx* ctx, int kind, int iters, double* ops_per_s, float* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* DOT_RING_B200_H */
