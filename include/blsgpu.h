/*
 * blsgpu.h — C ABI of libblsgpu.so: B200 (sm_100a) batch BLS12-381 signature verification.
 *
 * This is the drop-in boundary for nim-blscurve's batch-verification path: the Nim module
 * blscurve/cuda/blsgpu_abi.nim (see INTEGRATION.md) binds exactly these symbols and the bodies of
 * batchVerifySerial / batchVerifyParallel / batchVerify / aggregateAll / combine call them instead
 * of BLST.  File:line references are into /root/reference.
 *
 * Data formats are the reference's in-memory formats, byte for byte:
 *   SignatureSet = (PublicKey, array[32,byte], Signature)      blscurve/bls_batch_verifier.nim:34
 *     = blst_p1_affine (2 x 48 B) | 32 B message | blst_p2_affine (4 x 48 B) = 320 bytes, no padding;
 *     every Fp is 6 x u64 little-endian limbs in Montgomery form    vendor/blst/bindings/blst.h:63,:170,:197
 *   affine infinity = all-zero bytes.
 *   GT output = 576 bytes as blst_bendian_from_fp12 writes them     vendor/blst/src/fp12_tower.c:773-786
 *
 * Return convention for verification calls: 1 = valid, 0 = invalid (same booleans as the reference,
 * including false on empty input — bls_batch_verifier.nim:137, :312 — and on an infinite public key —
 * vendor/blst/src/aggregate.c:296), negative = runtime failure (CUDA error, bad argument); the text is
 * available from blsgpu_last_error().  There is no CPU fallback: without a CUDA device every call fails.
 *
 * Threading: one in-flight call per blsgpu_ctx (like one BatchedBLSVerifierCache per caller,
 * bls_batch_verifier.nim:389-391); different contexts may be used from different host threads.
 * Host pointers are borrowed for the duration of the call only.
 */
#ifndef BLSGPU_H
#define BLSGPU_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct blsgpu_ctx blsgpu_ctx;

#define BLSGPU_SET_BYTES 320
#define BLSGPU_GT_BYTES 576
#define BLSGPU_ERR_CUDA (-1)
#define BLSGPU_ERR_ARG (-2)
#define BLSGPU_ERR_CAPACITY (-3)

/* Number of CUDA devices visible (0 when none: the library cannot work). */
int blsgpu_device_count(void);

/* Replaces BatchedBLSVerifierCache.init (bls_batch_verifier.nim:108-119): device scratch for batches of up
 * to max_sets signature sets on CUDA device `device`.  NULL on failure (see blsgpu_last_error(NULL)). */
blsgpu_ctx *blsgpu_create(int device, size_t max_sets);
void blsgpu_destroy(blsgpu_ctx *ctx);
const char *blsgpu_last_error(const blsgpu_ctx *ctx);
size_t blsgpu_capacity(const blsgpu_ctx *ctx);

/* Multi-GPU context (SURVEY.md section 8b: `blsgpu_create(const int* devices, int ndev, size_t max_sets)`): replaces the
 * Taskpools fan-out INSIDE the call (bls_batch_verifier.nim:316-369).  blsgpu_batch_verify on such a context cuts the
 * batch into ndev balanced contiguous shares (the rule of parallel_chunks.nim:42-55), runs share k on devices[k]
 * (scalars from the global derivation, so verdict and GT do not depend on ndev), pulls the ndev 576-byte Fp12
 * partials + flags to devices[0] over NVLink peer copies and runs ONE final exponentiation.  blsgpu_msm_g1 /
 * blsgpu_msm_g2 on such a context shard the points the same way (one affine partial sum per device, summed on
 * devices[0]).  Every other entry point runs on devices[0].  A device may be listed more than once. */
blsgpu_ctx *blsgpu_create_multi(const int *devices, int ndev, size_t max_sets);
/* Number of shares (devices) a context spans: 1 for blsgpu_create. */
int blsgpu_device_span(const blsgpu_ctx *ctx);

/* Run on an existing CUDA stream (cudaStream_t passed as void*; NULL = the context's own stream). */
int blsgpu_set_stream(blsgpu_ctx *ctx, void *cuda_stream);

/* Random-linear-combination scalars exactly as the reference derives them
 * (blst_min_pubkey_sig_core.nim:476-505, :545-556; chunking parallel_chunks.nim:42-55):
 *   chunks == 0: serial derivation (batchVerifySerial): seed = SHA256(srb)
 *   chunks  > 0: batchVerifyParallel with numThreads = chunks: numBatches = min(n, chunks),
 *                seed_c = SHA256(srb || LE64(c)); per set seed <- SHA256(seed) until LE64(seed[0..8]) != 0.
 * Computed on the device; out receives n little-endian 64-bit scalars. */
int blsgpu_rlc_scalars(blsgpu_ctx *ctx, const uint8_t srb[32], size_t n, uint32_t chunks, uint64_t *out);

/* Replaces the body of batchVerifySerial (:121-160) / batchVerifyParallel (:296-371):
 * ctx.init + update* + commit + merge + finalVerify on BLST become one device pipeline.
 *   sets     n x 320 bytes, host memory
 *   chunks   scalar derivation mode as above (ignored when scalars != NULL)
 *   scalars  optional n explicit 64-bit blinding scalars (all must be non-zero)
 *   gt_out   optional 576 bytes: the GT value after final exponentiation, FE(conj(ML(S,G1)) * prod ML(...))
 */
int blsgpu_batch_verify(blsgpu_ctx *ctx, const void *sets, size_t n, const uint8_t srb[32], uint32_t chunks,
                        const uint64_t *scalars, uint8_t gt_out[576]);

/* Same with the sets already resident in device memory (d_sets: device pointer, n x 320 bytes). */
int blsgpu_batch_verify_dev(blsgpu_ctx *ctx, const void *d_sets, size_t n, const uint8_t srb[32],
                            uint32_t chunks, const uint64_t *scalars, uint8_t gt_out[576]);

/* Multi-GPU: one rank's share of a batch of total_n sets.  The rank owns the global index range
 * [first, first + n) (the balanced split of parallel_chunks.nim over ranks) and derives the scalars of
 * exactly those indices from the global (total_n, chunks) derivation, so the result does not depend on
 * the number of ranks.  Output: the 576-byte Fp12 partial  conj(ML(S_k, G1)) * prod_{i in k} ML([r_i]pk_i, H(m_i))
 * in the reference's in-memory Fp12 layout (what blst_pairing_merge multiplies, aggregate.c:410-458), and
 * *flags != 0 if a set of this share must fail the batch (infinite public key).  Such a share's partial is SEALED:
 * it is the zero element of Fp12 (576 zero bytes), which absorbs the product of the gathered partials and which the
 * final exponentiation maps to zero != one — so the partial alone carries the verdict and ranks need to exchange
 * nothing else (one 576-byte collective); blsgpu_finalize* then return 0 with an all-zero GT.
 * sets_on_device != 0: `sets` is a device pointer. */
int blsgpu_partial(blsgpu_ctx *ctx, const void *sets, int sets_on_device, size_t n, size_t first, size_t total_n,
                   const uint8_t srb[32], uint32_t chunks, const uint64_t *scalars, uint8_t partial_out[576],
                   int *flags);

/* Stream-ordered forms for the multi-GPU pipeline (no host synchronisation, results stay on the device so a
 * collective can follow on the same stream): d_partial_out = 576 bytes of device memory, d_flag_out = one
 * device int (non-zero when a set of the share has an infinite public key). */
int blsgpu_partial_dev(blsgpu_ctx *ctx, const void *d_sets, size_t n, size_t first, size_t total_n,
                       const uint8_t srb[32], uint32_t chunks, void *d_partial_out, int *d_flag_out);
/* d_partials: count x 576 bytes on the device (e.g. the all-gather output), d_flags: count ints or NULL. */
int blsgpu_finalize_dev(blsgpu_ctx *ctx, const void *d_partials, size_t count, const int *d_flags,
                        uint8_t gt_out[576]);

/* Product of `count` gathered partials, ONE final exponentiation, comparison with 1 (aggregate.c:494-500).
 * The per-share flags are not an input: a flagged share's partial is sealed (all zero, see blsgpu_partial), so the
 * product is zero and the result is 0 / all-zero GT, the reference's `false` for an infinite public key
 * (bls_batch_verifier.nim:153, :259).  blsgpu_finalize_dev additionally accepts gathered flags (d_flags, NULL = none). */
int blsgpu_finalize(blsgpu_ctx *ctx, const uint8_t *partials, size_t count, uint8_t gt_out[576]);

/* hash_to_G2 for n messages of msg_len bytes each (replaces blst_hash_to_g2 + blst_p2_to_affine,
 * vendor/blst/src/map_to_g2.c:388-396): out_compressed (nullable) n x 96 bytes Zcash compressed form,
 * out_affine (nullable) n x 192 bytes blst_p2_affine.  dst_len <= 255. */
int blsgpu_hash_to_g2(blsgpu_ctx *ctx, const uint8_t *msgs, size_t n, size_t msg_len, const uint8_t *dst,
                      size_t dst_len, uint8_t *out_compressed, uint8_t *out_affine);

/* aggregateAll (blst_min_pubkey_sig_core.nim:179-195): sum of n affine points; 0 on empty input. */
int blsgpu_aggregate_g1(blsgpu_ctx *ctx, const void *points96, size_t n, uint8_t out96[96]);
int blsgpu_aggregate_g2(blsgpu_ctx *ctx, const void *points192, size_t n, uint8_t out192[192]);

/* subtractAll (blst_min_pubkey_sig_core.nim:197-209; replaces its blst_p{1,2}_from_affine / _add_or_double_affine /
 * _cneg / _to_affine calls): dst <- dst - sum of the n affine points, in place.  n == 0 leaves dst untouched (:199-200).
 * Returns 1, or a negative error code. */
int blsgpu_subtract_g1(blsgpu_ctx *ctx, uint8_t dst96[96], const void *elems96, size_t n);
int blsgpu_subtract_g2(blsgpu_ctx *ctx, uint8_t dst192[192], const void *elems192, size_t n);

/* Segmented aggregateAll: segment k sums points[offsets[k] .. offsets[k+1]) (an empty segment yields infinity, the case
 * aggregateAll reports as false, blst_min_pubkey_sig_core.nim:183-184); out96 receives nseg affine points.  One launch for
 * all committees of a block (SURVEY.md §8d config 2: 128 x 128 + 512 public keys). */
int blsgpu_aggregate_g1_segments(blsgpu_ctx *ctx, const void *points96, const uint32_t *offsets, size_t nseg,
                                 uint8_t *out96);

/* aggregateVerify (blscurve/bls_sig_min_pubkey.nim:155-204 over ContextCoreAggregateVerify,
 * blst_min_pubkey_sig_core.nim:310-398: update per pair, finish(signature), commit, finalverify): n (public key, message)
 * pairs and ONE signature, no blinding: FE( prod ML(pk_i, H(m_i)) * ML(sig, -G1) ) == 1.  Message i is
 * msgs[msg_offsets[i] .. msg_offsets[i+1]); dst as in blsgpu_hash_to_g2.  n == 0 -> 0; an infinite public key -> 0
 * (aggregate.c:296); an infinite signature contributes nothing (aggregate.c:486-492).  With n == 1 this is `verify` /
 * coreVerifyNoGroupCheck (blst_min_pubkey_sig_core.nim:264-297).  gt_out (nullable): the 576 GT bytes. */
int blsgpu_aggregate_verify(blsgpu_ctx *ctx, const void *pubkeys96, size_t n, const uint8_t *msgs,
                            const uint32_t *msg_offsets, const uint8_t *dst, size_t dst_len, const void *sig192,
                            uint8_t gt_out[576]);

/* fastAggregateVerify (bls_sig_min_pubkey.nim:238-258): aggregateAll of the n public keys on the device, then the
 * single-pair check above on one message.  n == 0 -> 0. */
int blsgpu_fast_aggregate_verify(blsgpu_ctx *ctx, const void *pubkeys96, size_t n, const uint8_t *msg, size_t msg_len,
                                 const uint8_t *dst, size_t dst_len, const void *sig192, uint8_t gt_out[576]);

/* Batched PublicKey.fromBytes / Signature.fromBytes (blscurve/blst/bls_sig_io.nim:42-122): n encodings of in_len bytes
 * each (public keys: 48 compressed -> blst_p1_uncompress e1.c:261, or 96 -> blst_p1_deserialize e1.c:328; signatures: 96
 * -> blst_p2_uncompress e2.c:312, or 192 -> blst_p2_deserialize e2.c:391), then "infinity public keys are not allowed"
 * and, when group_check != 0, the subgroup check (blst_p1_affine_in_g1 / blst_p2_affine_in_g2); group_check == 0 is
 * fromBytesKnownOnCurve.  out receives n affine points in the in-memory Montgomery layout (all-zero on failure),
 * status[i] (nullable) the BLST_ERROR of element i (bindings/blst.h:47-56: 0 success, 1 bad encoding, 2 not on curve,
 * 3 not in group, 6 public key is infinity).  Returns 1 when every element decoded, 0 otherwise, < 0 on runtime error. */
int blsgpu_pubkeys_from_bytes(blsgpu_ctx *ctx, const uint8_t *in, size_t n, size_t in_len, int group_check,
                              uint8_t *out96, uint8_t *status);
int blsgpu_signatures_from_bytes(blsgpu_ctx *ctx, const uint8_t *in, size_t n, size_t in_len, int group_check,
                                 uint8_t *out192, uint8_t *status);
/* The inverse (blst_p1_affine_compress / blst_p2_affine_compress, bls_sig_io.nim:20-36): n x 48 / n x 96 bytes. */
int blsgpu_pubkeys_to_bytes(blsgpu_ctx *ctx, const void *points96, size_t n, uint8_t *out48);
int blsgpu_signatures_to_bytes(blsgpu_ctx *ctx, const void *points192, size_t n, uint8_t *out96);

/* G1 multi-scalar multiplication (replaces blst_p1s_mult_pippenger + blst_p1_to_affine,
 * vendor/blst/src/multi_scalar.c:415-434; call shape of benchmarks/bls12381_msm_g1.nim:57-59):
 * points n x 96 bytes affine, scalars n x ceil(nbits/8) bytes little-endian, out = affine sum. */
int blsgpu_msm_g1(blsgpu_ctx *ctx, const void *points96, const void *scalars, size_t n, size_t nbits,
                  uint8_t out96[96]);
int blsgpu_msm_g1_dev(blsgpu_ctx *ctx, const void *d_points96, const void *d_scalars, size_t n, size_t nbits,
                      uint8_t out96[96]);

/* G2 multi-scalar multiplication (replaces blst_p2s_mult_pippenger + blst_p2_to_affine,
 * vendor/blst/src/multi_scalar.c:442-446; with nbits = 64 this is the signature half of
 * MultiSignatureSet.combine, blst_min_pubkey_sig_core.nim:637-644): points n x 192 bytes affine. */
int blsgpu_msm_g2(blsgpu_ctx *ctx, const void *points192, const void *scalars, size_t n, size_t nbits,
                  uint8_t out192[192]);
int blsgpu_msm_g2_dev(blsgpu_ctx *ctx, const void *d_points192, const void *d_scalars, size_t n, size_t nbits,
                      uint8_t out192[192]);

/* MultiSignatureSet.combine (blscurve/bls_batch_verifier.nim:100-106 -> blst_min_pubkey_sig_core.nim:570-647): the
 * random linear combination of n (public key, signature) pairs on ONE message, with the reference's scalar order
 * (SHA-256 chain on secureRandomBytes, four 64-bit scalars per digest taken last-first, zeros skipped) and its two
 * Pippenger calls (nbits = 64).  n == 1 copies the pair; n == 0 is an error (raiseAssert in the reference).
 * Returns 1 and the affine pair (96 + 192 bytes). */
int blsgpu_combine(blsgpu_ctx *ctx, const uint8_t srb[32], const void *pubkeys96, const void *sigs192, size_t n,
                   uint8_t pk_out[96], uint8_t sig_out[192]);

/* Per-stage device times (ms) of the last batch_verify/partial call on this context, measured with CUDA
 * events on the call's stream.  Returns the number of stages written (<= max); names via blsgpu_stage_name. */
int blsgpu_last_stage_ms(const blsgpu_ctx *ctx, float *ms, int max);
const char *blsgpu_stage_name(int stage);
/* Kernel launches issued by the last call. */
int blsgpu_last_launches(const blsgpu_ctx *ctx);

/* Test/diagnostic entry points */
/* Fp unit ops on the device: op 0=mul 1=add 2=sub 3=sqr 4=inverse (Fermat) 6=inverse (binary Euclid); a,b,out: n x 48
 * bytes (Montgomery). */
int blsgpu_test_fp(blsgpu_ctx *ctx, int op, const void *a, const void *b, size_t n, void *out);
/* One device field primitive on n records, through the functions the pipelines call.  A record is field elements
 * (48 B each, Montgomery, little-endian) followed by an op-specific tail of u32 words padded to 16 B; in_rec_bytes and
 * out_rec_bytes must be the op's sizes, else (or for an unknown op) BLSGPU_ERR_ARG.  Per op, inputs -> outputs:
 *   Fp, one thread per record:    FP_MUL, FP_MUL_NI (a, b -> a b/R);  FP_SQR, FP_SQR_NI (a -> a^2/R);  FP_ADD, FP_SUB
 *                                 (a, b -> a +- b);  FP_NEG, FP_INV, FP_INV_VARTIME, FP_POW_P34, FP_FROM_MONT (a -> r);
 *                                 FP_PARITY, FP_IS_LEXICALLY_LARGEST_CANON (a -> word)
 *   Fp2, one thread per record:   FP2_MUL (a, b -> r);  FP2_SQR, FP2_MUL_XI, FP2_INV, FP2_INV_VARTIME (a -> r);
 *                                 FP2_MUL_FP (a, Fp k -> r);  FP2_RSQRT_OR_Z (a -> r, word is_square);
 *                                 FP2_SGN0, FP2_IS_LEXICALLY_LARGEST (a -> word)
 *   Fp2 on a lane pair (fp2h):    H_MUL (a, b -> r);  H_SQR, H_MUL_XI, H_CONJ, H_INV (a -> r);  H_MUL_FP (a, Fp k -> r)
 *   one lane of a six-lane team:  TEAM_DOT3 (a0..a2, b0..b2 -> sum a_t b_t / R);  TEAM_DOT4 (a0..a3, b0..b3, words
 *                                 dbl_mask, zero_mask -> the same with a_t doubled / zeroed per mask bit)
 *   one six-lane team:            TEAM_MUL_LINE (Fp12 f in tower order, line l0 l1 l2 -> f * line);
 *                                 TEAM_SQUARE (f -> f^2)
 *   Fp, one thread per record:    LIN_FINISH (x0..x6 positive, x7..x13 negative, words m0..m13 in 0..15 ->
 *                                 sum m_j x_j over the positive terms minus the negative ones, mod p) */
enum {
    BLSGPU_TF_FP_MUL, BLSGPU_TF_FP_MUL_NI, BLSGPU_TF_FP_SQR, BLSGPU_TF_FP_SQR_NI, BLSGPU_TF_FP_ADD, BLSGPU_TF_FP_SUB,
    BLSGPU_TF_FP_NEG, BLSGPU_TF_FP_INV, BLSGPU_TF_FP_INV_VARTIME, BLSGPU_TF_FP_POW_P34, BLSGPU_TF_FP_FROM_MONT,
    BLSGPU_TF_FP_PARITY, BLSGPU_TF_FP_IS_LEXICALLY_LARGEST_CANON,
    BLSGPU_TF_FP2_MUL, BLSGPU_TF_FP2_SQR, BLSGPU_TF_FP2_MUL_XI, BLSGPU_TF_FP2_MUL_FP, BLSGPU_TF_FP2_INV,
    BLSGPU_TF_FP2_INV_VARTIME, BLSGPU_TF_FP2_RSQRT_OR_Z, BLSGPU_TF_FP2_SGN0, BLSGPU_TF_FP2_IS_LEXICALLY_LARGEST,
    BLSGPU_TF_H_MUL, BLSGPU_TF_H_SQR, BLSGPU_TF_H_MUL_XI, BLSGPU_TF_H_MUL_FP, BLSGPU_TF_H_CONJ, BLSGPU_TF_H_INV,
    BLSGPU_TF_TEAM_DOT3, BLSGPU_TF_TEAM_DOT4, BLSGPU_TF_TEAM_MUL_LINE, BLSGPU_TF_TEAM_SQUARE,
    BLSGPU_TF_LIN_FINISH,
    BLSGPU_TF_COUNT
};
int blsgpu_test_field(blsgpu_ctx *ctx, int op, const void *in, size_t in_rec_bytes, size_t n, void *out,
                      size_t out_rec_bytes);
/* The message hash of the small-batch route (the pipeline's map kernel, then the cofactor-clearing dataflow program):
 * n <= 4096 sets in (host, 320 B each); out_in / out_out (nullable): n x 6 field elements (48 B each, Montgomery) =
 * the homogeneous E2 point (X : Y : Z) before / after the program.  H(m_i) = (X/Z, Y/Z) of out_out. */
int blsgpu_test_small_hash(blsgpu_ctx *ctx, const void *sets320, size_t n, uint8_t *out_in, uint8_t *out_out);
/* Integer-multiply pipe microbenchmark: returns measured 32x32->64 multiply-accumulates per second. */
double blsgpu_imad_peak(blsgpu_ctx *ctx, int wide);
/* Register-resident Montgomery multiplications per second of this library's fp_mul (no memory traffic). */
double blsgpu_fpmul_peak(blsgpu_ctx *ctx, int threads_per_block, int blocks_per_sm);
/* Generate n valid signature sets on the device (synthetic workload for benchmarks):
 * sk_i = 1 + (SHA256(seed || LE64(first+i)) mod 2^250), pk = [sk]G1, msg = SHA256("blsgpu" || LE64(first+i)),
 * sig = [sk]H(msg).  out: device pointer if out_on_device, else host. */
int blsgpu_make_sets(blsgpu_ctx *ctx, uint64_t seed, size_t first, size_t n, void *out, int out_on_device);

/* Synthetic MSM inputs on the device (benchmark only): P_i = [k_i]G1 (96-bit k_i), 255-bit coefficients. */
int blsgpu_msm_make_inputs(blsgpu_ctx *ctx, uint64_t seed, size_t n, void *d_points96, void *d_scalars32);

#ifdef __cplusplus
}
#endif
#endif
