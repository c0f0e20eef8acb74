/*
 * multilinear_b200 — C ABI of the B200 (sm_100a) CUDA backend for the polynomial-commitment hot path
 * of fr34za/multilinear (reference sources cited as path:line relative to /root/reference/).
 *
 * The reference has no FFI of its own (SURVEY.md §8b): the boundary is the crate's public generic
 * functions, monomorphised for Field128.  Every entry point below is the function a Rust maintainer
 * binds with `extern "C"` to replace the body of the cited reference function (see INTEGRATION.md).
 *
 * Conventions
 *   - Field element: 16 bytes, little-endian canonical u128 in [0, M), M = 2^128 - 45*2^40 + 1
 *     (src/field.rs:33-38, src/ntt/mod.rs:35).  `&[Field128]` <-> (const uint8_t*, size_t count).
 *     Element buffers must be 16-byte aligned (Rust's u128 alignment).
 *   - ReedSolomonPair: 32 bytes {value, minus_value} (#[repr(C)], src/fri/mod.rs:30-35).
 *   - HashDigest: 32 bytes (src/merkle_tree/mod.rs:5).  Direction: u8, 0 = Left, 1 = Right (:13-18).
 *   - Every function returns an int status (ML_OK = 0).  The reference's assert!/panic! sites map to
 *     ML_ERR_NOT_POW2 / ML_ERR_SIZE / ML_ERR_NOT_RS_CODE; `None` maps to ML_ERR_OUT_OF_RANGE.
 *     ml_last_error() returns a thread-local message.  Nothing unwinds across the boundary.
 *   - Functions without a `_dev` suffix take HOST pointers, copy to the GPU, run the CUDA kernels and
 *     copy the result back; `_dev` variants take DEVICE pointers (same layout) and a stream and leave
 *     results in HBM.  There is no CPU fallback: without a usable CUDA device every compute entry
 *     point fails with ML_ERR_CUDA.
 *   - Handles are opaque, own device memory, are not thread-safe, and are released with their *_free.
 *   - Aliasing: a `_dev` entry with separate element input and output buffers says next to it whether in == out is allowed.
 */
#ifndef MULTILINEAR_B200_H
#define MULTILINEAR_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ML_LOG_BLOWUP 1    /* src/fri/mod.rs:16 */
#define ML_NUM_QUERIES 128 /* src/fri/mod.rs:17 */
#define ML_MAX_PEERS 16   /* ranks of a sharded prover */

enum {
    ML_OK = 0,
    ML_ERR_NOT_POW2 = 1,     /* assert!(n.is_power_of_two()) — ntt/mod.rs:71-74,134; merkle_tree/mod.rs:66-69; fri/mod.rs:60-63 */
    ML_ERR_SIZE = 2,         /* mismatched sizes — merkle_tree/mod.rs:94-108; sumcheck.rs:131; polynomials.rs:127-131,166-170 */
    ML_ERR_OUT_OF_RANGE = 3, /* Option::None — ntt/mod.rs:46-48; merkle_tree/mod.rs:35-37,144-146 */
    ML_ERR_NOT_RS_CODE = 4,  /* assert "not an RS code" — fri/mod.rs:119-122 */
    ML_ERR_GENERATOR = 5,    /* `gen` is not a primitive n-th root of unity (the DIT network assumes it) */
    ML_ERR_CUDA = 6,         /* CUDA runtime error / no device / extension not built for this GPU */
    ML_ERR_ALLOC = 7,
    ML_ERR_ARG = 8,
    ML_ERR_PEER = 9          /* sharded prover: a peer rank's memory cannot be mapped, or a peer did not arrive in time */
};
/* verifier results (FriProofError, src/fri/mod.rs:251-258) */
enum {
    ML_V_OK = 0,
    ML_V_QUERY_MISMATCH = 101,
    ML_V_WRONG_NUM_QUERIES = 102,
    ML_V_WRONG_NUM_PATHS = 103,
    ML_V_INCLUSION_HASH = 104,
    ML_V_INCLUSION_INDEX = 105,
    ML_V_LAST_RANDOM = 106,
    ML_V_SUMCHECK = 107 /* assert_eq!(delta * last_elem, pol.evaluate(r)) — multilinear_pcs.rs:180-184 */
};

const char *ml_last_error(void);
const char *ml_version(void);
int ml_device_count(int *count);
int ml_set_device(int device);                 /* one process per GPU: call once with LOCAL_RANK */
int ml_device_name(char *out, size_t cap);
int ml_synchronize(void);
/* number of kernels this library has launched in the calling process (bench.py's `gpu_launches`) */
uint64_t ml_kernel_launches(void);

/* Streams.  Host-pointer entry points run on a per-device library stream unless the calling thread installed its
 * own with ml_set_thread_stream; `_dev` entry points take the stream explicitly.  Several host threads may drive
 * independent commits on different streams of one GPU (the library is thread-safe across handles). */
int ml_stream_create(void **out);
int ml_stream_destroy(void *stream);
int ml_stream_synchronize(void *stream);
int ml_set_thread_stream(void *stream, int enable);
/* A handle made by a `_dev` entry (ml_fri_*, ml_merkle_*, ml_sumcheck_*, ml_wsumcheck_*) records that entry's stream and frees its
 * device memory on it: free the handle before destroying its stream.  The handle's methods run on the library stream
 * (ml_wsumcheck_* on the recorded one) and return once their results are complete. */

/* Device memory the library caches.  Scratch and handle-owned buffers are stream-ordered allocations: streams made by
 * ml_stream_create get a private cudaMemPool (destroyed by ml_stream_destroy); any other stream (caller-owned, e.g. a
 * framework's stream) allocates from the device's default pool.  Freed blocks stay cached for reuse — invisible to other allocators in the
 * process — until released: ml_trim_pools returns cached blocks of the current device down to keep_bytes per pool,
 * ml_release_pools synchronises the device and returns all of them, ml_set_pool_release_threshold bounds what stays cached at
 * every synchronisation point (default: unbounded).  ml_pool_stats: bytes reserved from the driver / in use, current device. */
int ml_trim_pools(size_t keep_bytes);
int ml_release_pools(void);
int ml_set_pool_release_threshold(uint64_t bytes);
int ml_pool_stats(uint64_t *reserved_bytes, uint64_t *used_bytes);

/* raw device memory for callers that keep data resident (bench, multi-GPU orchestration) */
int ml_dev_alloc(size_t bytes, void **out);
int ml_dev_free(void *p);
int ml_dev_upload(void *dst_dev, const void *src_host, size_t bytes);
int ml_dev_download(void *dst_host, const void *src_dev, size_t bytes);
int ml_host_alloc_pinned(size_t bytes, void **out);
int ml_host_free_pinned(void *p);
/* page-lock / unlock memory the caller allocated itself (Vec<Field128>, numpy array), so host-pointer entry points upload from it
 * at pinned-memory speed; unregister before freeing it.  Unregistered (pageable) inputs work too, through the driver's staging copies. */
int ml_host_register(void *p, size_t bytes);
int ml_host_unregister(void *p);

/* ---- field (src/field.rs:66-154; winter-math f128).  Element-wise vector ops run on the GPU. ---- */
int ml_fe_add_vec(const uint8_t *a, const uint8_t *b, size_t n, uint8_t *out);
int ml_fe_sub_vec(const uint8_t *a, const uint8_t *b, size_t n, uint8_t *out);
int ml_fe_mul_vec(const uint8_t *a, const uint8_t *b, size_t n, uint8_t *out);
int ml_fe_inv_vec(const uint8_t *a, size_t n, uint8_t *out);                    /* inv(0) = 0 */
int ml_fe_pow_vec(const uint8_t *a, const uint8_t exp_le[16], size_t n, uint8_t *out); /* NttField::pow, ntt/mod.rs:56-58 */
int ml_fe_from_i64_vec(const int64_t *v, size_t n, uint8_t *out);               /* From<i64>, field.rs:150-154 */
/* n 256-bit little-endian integers (32 bytes each) -> v mod M; variant selects the device reduction (1: multiply by the limbs
 * of 2^128 - M, 2: shift form, the one every kernel uses) so the tests can drive both through adversarial inputs */
int ml_fe_from_wide_vec(const uint8_t *v, size_t n, int variant, uint8_t *out);
int ml_synthetic_elements_dev(uint64_t seed, size_t n, void *out_dev, void *stream); /* bench input generator */

/* ---- NTT (src/ntt/mod.rs) ----
 * RESTRICTION (differs from the reference's generic signatures): `gen` must be the root the reference's own callers pass,
 * pow_2_generator(log2 n) (n = the transform length; 2n for reed_solomon), or its inverse; anything else returns
 * ML_ERR_GENERATOR instead of computing with it.  The kernels take their twiddles from per-size root tables kept in HBM. */
int ml_pow2_generator(uint64_t log_size, uint8_t out[16]);            /* NttField::pow_2_generator :42-54 */
int ml_pow2_generator_powers(uint64_t log_size, uint8_t *out);        /* pow_2_generator_powers :18-28 (2^log_size elements) */
int ml_pow2_generator_powers_dev(uint64_t log_size, void *out_dev, void *stream);
int ml_bit_reverse_permutation(uint8_t *values, size_t n, size_t elem_bytes); /* bit_reverse_permutation :113-123 */
int ml_ntt(const uint8_t *coeffs, size_t n, const uint8_t gen[16], uint8_t *evals);   /* Polynomial::ntt :69-110 */
int ml_intt(const uint8_t *evals, size_t n, const uint8_t gen[16], uint8_t *coeffs);  /* LagrangePolynomial::intt :132-173 */
int ml_ntt_dev(const void *coeffs_dev, size_t n, const uint8_t gen[16], void *evals_dev, void *stream);   /* in place allowed */
int ml_intt_dev(const void *evals_dev, size_t n, const uint8_t gen[16], void *coeffs_dev, void *stream);   /* in place allowed */
int ml_poly_evaluate(const uint8_t *coeffs, size_t n, const uint8_t x[16], uint8_t out[16]); /* Polynomial::evaluate :62-67 */
/* univariate helpers of src/polynomials.rs on the domain 0..n-1 (the sumcheck round polynomials, n <= 4 in the crate) */
int ml_poly_interpolate(const uint8_t *evals, size_t n, uint8_t *coeffs_out);          /* PolynomialEvals::interpolate :51-86 (host scalars, n <= 2^14) */
int ml_poly_evaluate_over_domain(const uint8_t *coeffs, size_t n, uint8_t *evals_out);  /* Polynomial::evaluate_over_domain :16-28 */
int ml_reed_solomon(const uint8_t *coeffs, size_t n, const uint8_t gen[16], uint8_t *code /* 2n */); /* src/fri/mod.rs:19-28 */
/* in place allowed: code_dev == coeffs_dev, a buffer of 2n elements whose first n are the coefficients */
int ml_reed_solomon_dev(const void *coeffs_dev, size_t n, const uint8_t gen[16], void *code_dev, void *stream);

/* ---- multilinear polynomials (src/polynomials.rs) ---- */
int ml_mle_to_coefficient(const uint8_t *evals, size_t len, uint8_t *coeffs);   /* MultilinearPolynomialEvals::to_coefficient :150-163 */
int ml_mle_to_evaluation(const uint8_t *coeffs, size_t len, uint8_t *evals);    /* MultilinearPolynomial::to_evaluation :111-124 */
int ml_mle_to_coefficient_dev(const void *evals_dev, size_t len, void *coeffs_dev, void *stream);   /* in place allowed */
int ml_mle_to_evaluation_dev(const void *coeffs_dev, size_t len, void *evals_dev, void *stream);    /* in place allowed */
int ml_mle_evals_evaluate(const uint8_t *evals, size_t len, const uint8_t *args, size_t n_args, uint8_t out[16]);   /* :165-187 */
int ml_mle_coeffs_evaluate(const uint8_t *coeffs, size_t len, const uint8_t *args, size_t n_args, uint8_t out[16]); /* :126-146 */
int ml_mle_evals_evaluate_dev(const void *evals_dev, size_t len, const uint8_t *args, size_t n_args, uint8_t out[16], void *stream);

/* ---- transcript (src/transcript.rs) — strictly sequential SHA-256 over <= a few hundred bytes; host state ---- */
typedef struct ml_transcript ml_transcript;
int ml_transcript_new(ml_transcript **out);                                     /* Transcript::new :17-21 */
int ml_transcript_clone(const ml_transcript *t, ml_transcript **out);           /* #[derive(Clone)] :5 */
void ml_transcript_free(ml_transcript *t);
int ml_transcript_absorb(ml_transcript *t, const uint8_t *bytes, size_t len);   /* absorb :31-33 */
int ml_transcript_random(const ml_transcript *t, uint8_t out[32]);              /* random :23-29 */
int ml_transcript_next_challenge(ml_transcript *t, uint8_t out[16]);            /* next_challenge :35-38 */

/* ---- Merkle (src/merkle_tree/mod.rs) ---- */
typedef struct ml_merkle ml_merkle;
int ml_merkle_commit(const uint8_t *data, size_t item_bytes, size_t n_items, ml_merkle **out);  /* Merkle::commit :65-85 */
int ml_merkle_batch_commit(const uint8_t *const *data, size_t n_batches, size_t item_bytes, size_t n_items, ml_merkle **out); /* batch_commit :92-131 */
/* leaves are ReedSolomonPairs (code[i], code[i + n/2]) of a device-resident code — commit_rs_code, src/fri/mod.rs:45-55.
 * The tree keeps code_dev (ml_merkle_open reads the values from it): the code must stay allocated and unchanged until
 * ml_merkle_free. */
int ml_merkle_commit_rs_code_dev(const void *code_dev, size_t n, void *stream, ml_merkle **out);
void ml_merkle_free(ml_merkle *m);
int ml_merkle_root(const ml_merkle *m, uint8_t out[32]);                        /* root :27-29 */
size_t ml_merkle_num_layers(const ml_merkle *m);                                /* layers.len() :9 */
size_t ml_merkle_layer_len(const ml_merkle *m, size_t layer);
int ml_merkle_layer(const ml_merkle *m, size_t layer, uint8_t *out /* layer_len*32 */);
/* open / batch_open (:31-58, :134-175).  value: item_bytes (n_batches*item_bytes for a batched tree);
 * digests: path_len*32; dirs[i] = side the sibling is on.  ML_ERR_OUT_OF_RANGE = None. */
int ml_merkle_open(const ml_merkle *m, size_t index, uint8_t *value, uint8_t *digests, uint8_t *dirs, size_t *path_len);
/* MerkleInclusionPath::verify / batch_verify (:216-246, :253-293); returns ML_V_* (host, O(log n)) */
int ml_merkle_path_verify(const uint8_t *value, size_t value_bytes, const uint8_t *digests, const uint8_t *dirs,
                          size_t path_len, const uint8_t root[32], size_t index);

/* ---- FRI (src/fri/mod.rs) ---- */
typedef struct ml_fri ml_fri;             /* FriProverData :10-14 — all trees stay in HBM */
typedef struct ml_fri_proof ml_fri_proof; /* FriProof :239-249 */
int ml_fri_init(const uint8_t *code, size_t n, ml_transcript *t, ml_fri **out);                      /* init :58-76 */
int ml_fri_init_dev(const void *code_dev, size_t n, ml_transcript *t, void *stream, ml_fri **out);   /* code is copied */
/* fold_step :79-134.  gen_pows may be NULL (the backend keeps its own root tables in HBM).  RESTRICTION: when given it must be
 * pow_2_generator_powers(log2 domain) — length = original domain size, entries spot-checked (21 positions) against the
 * domain generator's powers, ML_ERR_SIZE / ML_ERR_GENERATOR otherwise; the kernels never read the caller's table.
 * Host-pointer entry points block the calling thread: inputs of 16 MB and more are uploaded one at a time per device
 * (after the calling thread's stream has drained) and results are read back before returning. */
int ml_fri_fold_step(ml_fri *f, const uint8_t *gen_pows, size_t gen_pows_len, size_t k, const uint8_t r[16], ml_transcript *t);
int ml_fri_fold(const uint8_t *gen_pows, size_t gen_pows_len, const uint8_t *code, size_t n, ml_transcript *t, ml_fri **out); /* fold :136-145 */
int ml_fri_fold_dev(const void *code_dev, size_t n, ml_transcript *t, void *stream, ml_fri **out);
void ml_fri_free(ml_fri *f);
size_t ml_fri_num_trees(const ml_fri *f);
int ml_fri_tree(const ml_fri *f, size_t i, const ml_merkle **tree /* borrowed */);
int ml_fri_tree_data(const ml_fri *f, size_t i, uint8_t *pairs_out /* leaves*32 */);                 /* merkle_trees[i].data */
int ml_fri_fold_roots(const ml_fri *f, uint8_t *out /* num_trees*32 */);                             /* fold_roots :147-152 */
int ml_fri_last_element(const ml_fri *f, uint8_t out[16], int *is_some);
/* open_query_at :154-174 — flat output: for tree j: value 32 B, then path_len_j digests, then path_len_j dirs */
int ml_fri_open_query_at(const ml_fri *f, size_t index, uint8_t *values /* trees*32 */, uint8_t *digests, uint8_t *dirs,
                         size_t *path_lens /* trees */);
int ml_fri_prove(const uint8_t *code, size_t n, const uint8_t *gen_pows, size_t gen_pows_len, ml_transcript *t, ml_fri_proof **out); /* prove :261-285 */
int ml_fri_prove_dev(const void *code_dev, size_t n, ml_transcript *t, void *stream, ml_fri_proof **out);
/* reed_solomon (:19-28) + FriProof::prove (:261-285) with the code kept in HBM between the two calls */
int ml_rs_fri_prove(const uint8_t *coeffs, size_t n, ml_transcript *t, ml_fri_proof **out);
int ml_rs_fri_prove_dev(const void *coeffs_dev, size_t n, ml_transcript *t, void *stream, ml_fri_proof **out);
/* reed_solomon + FriProverData::fold (:136-145): the commit phase only (all roots + last element), no queries */
int ml_rs_fri_fold_dev(const void *coeffs_dev, size_t n, ml_transcript *t, void *stream, ml_fri **out);
int ml_fri_verify(const ml_fri_proof *p);                                                            /* verify :287-309, returns ML_V_* */
void ml_fri_proof_free(ml_fri_proof *p);
size_t ml_fri_proof_num_commitments(const ml_fri_proof *p);
int ml_fri_proof_commitments(const ml_fri_proof *p, uint8_t *out);
int ml_fri_proof_last(const ml_fri_proof *p, uint8_t last_elem[16], uint8_t last_random[32]);
/* wire format of `bincode::serde::encode_to_vec(&proof, standard().with_little_endian().with_fixed_int_encoding())` (:367-391) */
size_t ml_fri_proof_serialized_len(const ml_fri_proof *p);
int ml_fri_proof_serialize(const ml_fri_proof *p, uint8_t *out);
int ml_fri_proof_deserialize(const uint8_t *blob, size_t len, ml_fri_proof **out); /* a proof made elsewhere (e.g. by the Rust crate): ML_ERR_ARG if malformed */

/* ---- sumcheck tables, PCS specialisation: width 1, composition |x| x[0] (src/constraint_system/sumcheck.rs:127-277) ---- */
typedef struct ml_sumcheck ml_sumcheck;
int ml_sumcheck_build_tables_for_pcs(const uint8_t *inputs, size_t n_vars, const uint8_t *evals, size_t height, ml_sumcheck **out); /* :128-145 */
int ml_sumcheck_build_tables_for_pcs_dev(const uint8_t *inputs, size_t n_vars, const void *evals_dev, size_t height, void *stream, ml_sumcheck **out);
void ml_sumcheck_free(ml_sumcheck *s);
size_t ml_sumcheck_height(const ml_sumcheck *s);
int ml_sumcheck_tables(const ml_sumcheck *s, uint8_t *matrix_out, uint8_t *delta_out);  /* current `height` entries each */
int ml_sumcheck_partial_sum(const ml_sumcheck *s, const uint8_t r[16], uint8_t out[16]);   /* partial_sum :204-232 */
int ml_sumcheck_fold(ml_sumcheck *s, const uint8_t r[16]);                                 /* fold :234-247 */
/* compute_sumcheck_polynomial :174-202 — total_degree 1..16, else ML_ERR_ARG (the PCS uses 2, multilinear_pcs.rs:57; at 0 the
 * reference panics) */
int ml_sumcheck_compute_polynomial(ml_sumcheck *s, size_t total_degree, uint8_t previous_sum[16], ml_transcript *t,
                                   uint8_t *nonzero_coeffs_out /* total_degree*16 */, uint8_t r_out[16]);
/* compute_sumcheck_polynomials :147-172 — composition_degree 0..15, else ML_ERR_ARG.  The PCS degree 1 runs every round on the
 * device; any other degree runs one host round per variable */
int ml_sumcheck_compute_polynomials(ml_sumcheck *s, size_t composition_degree, ml_transcript *t, const uint8_t sum[16],
                                    uint8_t *coeffs_out /* rounds*(composition_degree+1)*16 */, uint8_t *randoms_out /* rounds*16 */);
int ml_delta_evaluate(const uint8_t *data, const uint8_t *points, size_t n, uint8_t out[16]); /* Delta::evaluate, evaluation.rs:80-90 (host) */

/* ---- multilinear PCS (src/fri/multilinear_pcs.rs) ---- */
typedef struct ml_pcs_proof ml_pcs_proof; /* PCSProof :79-87 */
int ml_pcs_prove(const uint8_t *inputs, size_t n_vars, const uint8_t output[16], const uint8_t *evals, size_t n,
                 ml_transcript *t, ml_pcs_proof **out);                                     /* PCSProof::prove :90-136 */
int ml_pcs_prove_dev(const uint8_t *inputs, size_t n_vars, const uint8_t output[16], const void *evals_dev, size_t n,
                     ml_transcript *t, void *stream, ml_pcs_proof **out);
int ml_pcs_verify(const ml_pcs_proof *p, ml_transcript *t);                                 /* PCSProof::verify :138-190, returns ML_V_* */
void ml_pcs_proof_free(ml_pcs_proof *p);
const ml_fri_proof *ml_pcs_proof_fri(const ml_pcs_proof *p);
size_t ml_pcs_proof_num_rounds(const ml_pcs_proof *p);
int ml_pcs_proof_sumcheck_coeffs(const ml_pcs_proof *p, uint8_t *out /* rounds*2*16 */);    /* SumcheckPolynomial.nonzero_coeffs */

/* ---- stream-ordered provers: FriProof::prove / PCSProof::prove enqueued on a caller's stream ----
 * The transcript state as bytes: the 104-byte running SHA-256 state (eight state words, the 64-byte block buffer, the u64 byte
 * count), laid out identically on the host and on the device.  A state exported here can be copied into device memory and handed
 * to the calls below, and a state they leave in device memory can be copied back and imported. */
size_t ml_transcript_state_bytes(void);                                   /* 104 */
int ml_transcript_export(const ml_transcript *t, uint8_t *state_out);
int ml_transcript_import(const uint8_t *state, ml_transcript **out);
/* A plan owns every device buffer one prove of a 2^log_domain code needs (N = 2^log_domain): the code and Merkle tree of every
 * FRI layer (N, N/2, ... 4), the fold chain's scratch and the query phase's buffers, plus the sumcheck tables with pcs != 0.  It
 * is allocated once at creation on the current device with cudaMalloc, not from the stream pools, so ml_trim_pools never touches
 * it; creation also builds the root and NTT pass tables of the size.  ml_prove_plan_device_bytes is what it holds (about 96 N
 * bytes, 112 N with pcs).  ml_prove_plan_create: ML_ERR_SIZE for log_domain outside 2..40, ML_ERR_ALLOC when the plan does not
 * fit (nothing is left allocated), ML_ERR_CUDA without a device.  ml_prove_plan_free synchronises the plan's device.
 *
 * Each call computes what its blocking twin computes and leaves it in device memory, in stream order on `stream`:
 *   ml_rs_fri_prove_async = ml_rs_fri_prove_dev (coeffs_dev: N/2 coefficients),
 *   ml_fri_prove_async    = ml_fri_prove_dev    (code_dev: N elements),
 *   ml_pcs_prove_async    = ml_pcs_prove_dev    (inputs_dev: n_vars = log_domain - 1 points, output_dev: the claim, 1 element,
 *                                                evals_dev: N/2 evaluations); needs a plan made with pcs != 0.
 *   proof_dev (ml_prove_plan_proof_bytes bytes) receives the FriProof bincode blob, byte-identical to ml_fri_proof_serialize of
 *   the blocking twin's proof (for the PCS call: of ml_pcs_proof_fri); sumcheck_dev (2 * n_vars elements) receives
 *   ml_pcs_proof_sumcheck_coeffs; transcript_dev holds ml_transcript_state_bytes() of state on entry and is updated in place to
 *   the state the host transcript has after the blocking call; *status_dev receives ML_OK, or ML_ERR_NOT_RS_CODE when the code's
 *   last fold is not constant (the proof and transcript contents are then unspecified; the plan proves normally next time).
 * Inputs are only read.
 * Host-side rejections enqueue nothing and return: ML_ERR_ARG for a NULL plan or buffer, a device buffer that is not 16-byte
 * aligned, an output range (transcript, proof, sumcheck, status) overlapping any other buffer of the call, a PCS call on a plan
 * made with pcs = 0, or a current device other than the plan's.
 * No host work during an enqueue call: it makes no device allocation, no synchronisation, no host->device copy from host memory
 * and no host read of device data, so it returns once its kernels are enqueued and may be captured into a CUDA graph with
 * cudaStreamCaptureModeGlobal.  (A kernel launch error is returned as ML_ERR_CUDA; work enqueued before it stays enqueued.)
 * One proof in flight per plan: calls on one plan must be ordered by the caller (calls on one stream are); for overlap use one
 * plan per stream.  A captured graph keeps the pointers it was captured with, so each replay proves what those buffers hold at
 * replay time. */
typedef struct ml_prove_plan ml_prove_plan;
int ml_prove_plan_create(size_t log_domain, int pcs, ml_prove_plan **out);
void ml_prove_plan_free(ml_prove_plan *p);
size_t ml_prove_plan_device_bytes(const ml_prove_plan *p);
size_t ml_prove_plan_proof_bytes(const ml_prove_plan *p);   /* == ml_fri_proof_serialized_len of the proof it writes */
int ml_rs_fri_prove_async(ml_prove_plan *p, const void *coeffs_dev, void *transcript_dev, void *proof_dev, int *status_dev, void *stream);
int ml_fri_prove_async(ml_prove_plan *p, const void *code_dev, void *transcript_dev, void *proof_dev, int *status_dev, void *stream);
int ml_pcs_prove_async(ml_prove_plan *p, const void *inputs_dev, const void *output_dev, const void *evals_dev, void *transcript_dev,
                       void *proof_dev, void *sumcheck_dev, int *status_dev, void *stream);

/* ---- batched FRI / PCS (src/fri/batched_fri.rs, src/fri/batched_pcs.rs) ---- */
typedef struct ml_bfri_proof ml_bfri_proof; /* BatchedFriProof batched_fri.rs:21-27 */
int ml_fingerprint(const uint8_t r[16], const uint8_t *coeffs, size_t n, uint8_t out[16]);  /* fingerprint batched_fri.rs:30-38 (host, tiny) */
int ml_batched_fri_prove(const uint8_t *const *codes, size_t n_codes, size_t n, const uint8_t *gen_pows, size_t gen_pows_len,
                         ml_transcript *t, ml_bfri_proof **out);                            /* BatchedFriProof::prove batched_fri.rs:286-318 */
int ml_batched_fri_verify(const ml_bfri_proof *p);                                          /* batched_fri.rs:320-354 */
/* BatchedFriProverData (batched_fri.rs:9-14) step by step, host transcript — init :41-99, batched_fold_step :101-181 (the
 * remaining steps are ml_fri_fold_step on ml_bfri_fri_data), fold :183-205 (device transcript), open_query_at :207-225 */
typedef struct ml_bfri ml_bfri;
int ml_bfri_init(const uint8_t *const *codes, size_t n_codes, size_t n, ml_transcript *t, ml_bfri **out);
int ml_bfri_batched_fold_step(ml_bfri *h, const uint8_t *gen_pows, size_t gen_pows_len, const uint8_t r[16], ml_transcript *t);
int ml_bfri_fold(const uint8_t *gen_pows, size_t gen_pows_len, const uint8_t *const *codes, size_t n_codes, size_t n, ml_transcript *t, ml_bfri **out);
void ml_bfri_free(ml_bfri *h);
ml_fri *ml_bfri_fri_data(ml_bfri *h);                   /* borrowed: fold_step / fold_roots / last_element work on it */
const ml_merkle *ml_bfri_batch_layer(const ml_bfri *h); /* borrowed: root, layers */
size_t ml_bfri_num_codes(const ml_bfri *h);
int ml_bfri_fingerprint_r(const ml_bfri *h, uint8_t out[16]);
int ml_bfri_open_query_at(const ml_bfri *h, size_t index, uint8_t *batch_values /* n_codes*32 */, uint8_t *batch_digests, uint8_t *batch_dirs,
                          size_t *batch_path_len, uint8_t *values /* trees*32 */, uint8_t *digests, uint8_t *dirs, size_t *path_lens /* trees */);
void ml_bfri_proof_free(ml_bfri_proof *p);
int ml_bfri_proof_batch_commitment(const ml_bfri_proof *p, uint8_t out[32]);
size_t ml_bfri_proof_num_commitments(const ml_bfri_proof *p);
int ml_bfri_proof_commitments(const ml_bfri_proof *p, uint8_t *out);
int ml_bfri_proof_last(const ml_bfri_proof *p, uint8_t last_elem[16], uint8_t last_random[32]);
size_t ml_bfri_proof_serialized_len(const ml_bfri_proof *p);
int ml_bfri_proof_serialize(const ml_bfri_proof *p, uint8_t *out);
/* inverse of ml_bfri_proof_serialize (a blob made by the Rust crate, by ml_batched_*_prove_async or by the serializer): ML_ERR_ARG on
 * malformed input (truncated or trailing bytes, a wrong length prefix, a direction above 1, a non-canonical field element) */
int ml_bfri_proof_deserialize(const uint8_t *blob, size_t len, ml_bfri_proof **out);

typedef struct ml_bpcs_proof ml_bpcs_proof; /* BatchedPCSProof batched_pcs.rs:22-29 */
int ml_batched_pcs_prove(const uint8_t *inputs, size_t n_vars, const uint8_t *outputs, size_t n_polys,
                         const uint8_t *const *evals, size_t n, ml_transcript *t, ml_bpcs_proof **out); /* batched_pcs.rs:130-180 */
int ml_batched_pcs_prove_dev(const uint8_t *inputs, size_t n_vars, const uint8_t *outputs, size_t n_polys,
                             const void *const *evals_dev, size_t n, ml_transcript *t, void *stream, ml_bpcs_proof **out);
int ml_batched_pcs_verify(const ml_bpcs_proof *p, ml_transcript *t);                        /* batched_pcs.rs:182-253 */
void ml_bpcs_proof_free(ml_bpcs_proof *p);
const ml_bfri_proof *ml_bpcs_proof_fri(const ml_bpcs_proof *p);
size_t ml_bpcs_proof_num_rounds(const ml_bpcs_proof *p);
int ml_bpcs_proof_sumcheck_coeffs(const ml_bpcs_proof *p, uint8_t *out);

/* ---- stream-ordered batched provers: BatchedFriProof::prove / BatchedPCSProof::prove enqueued on a caller's stream ----
 * The batched counterpart of the stream-ordered provers above, for B = n_codes codes of N = 2^log_domain elements.  A plan is
 * made for one kind of call:
 *   ML_BPLAN_CODES: ml_batched_fri_prove_async    = ml_batched_fri_prove (codes_dev: B device pointers, N elements each; the
 *                   codes are read in place),
 *   ML_BPLAN_RS:    ml_batched_rs_fri_prove_async = reed_solomon of each + ml_batched_fri_prove, as ml_bfri_shard_rs_prove_dev
 *                   at one rank (coeffs_dev: B device pointers, N/2 coefficients each),
 *   ML_BPLAN_PCS:   ml_batched_pcs_prove_async    = ml_batched_pcs_prove_dev (inputs_dev: n_vars = log_domain - 1 points,
 *                   outputs_dev: B claimed values, evals_dev: B device pointers, N/2 evaluations each).
 * codes_dev / coeffs_dev / evals_dev are HOST arrays of device pointers, as ml_batched_pcs_prove_dev takes them; the call reads
 * the array before it returns.  A plan owns, in one cudaMalloc outside the stream pools: the batch tree (32 N bytes, also the
 * encodes' scratch), FRI layers N/2 .. 4 with their trees, for RS and PCS plans the B codes (16 B N bytes: 8 GiB at 64 x 2^22),
 * for PCS plans the sumcheck tables, and the chain and query buffers; ml_batched_prove_plan_device_bytes is the total.
 * ml_batched_prove_plan_create: ML_ERR_SIZE for log_domain outside 3..40 or n_codes outside 1..2^20, ML_ERR_ARG for an unknown
 * kind, ML_ERR_ALLOC when the plan does not fit (nothing is left allocated), ML_ERR_CUDA without a device.
 *
 * proof_dev (ml_batched_prove_plan_proof_bytes bytes) receives the BatchedFriProof bincode blob, byte-identical to
 * ml_bfri_proof_serialize of the blocking twin's proof (for PCS: of ml_bpcs_proof_fri); sumcheck_dev (2 * n_vars elements)
 * receives ml_bpcs_proof_sumcheck_coeffs; transcript_dev and *status_dev as for the single provers (ML_ERR_NOT_RS_CODE is possible
 * only for ML_BPLAN_CODES).  Inputs are only read.
 * Host-side rejections enqueue nothing and return ML_ERR_ARG: a NULL plan, buffer, array or pointer in the array; a device buffer
 * that is not 16-byte aligned; an output (transcript, proof, sumcheck, status) overlapping any input, including each of the
 * n_codes pointed-to buffers, or another output; a call of another kind than the plan's; a current device other than the plan's.
 * An enqueue makes no allocation, no synchronisation, no host->device copy from host memory and no host read of device data, and
 * may be captured into a CUDA graph with cudaStreamCaptureModeGlobal.  One proof in flight per plan, as above. */
enum { ML_BPLAN_CODES = 0, ML_BPLAN_RS = 1, ML_BPLAN_PCS = 2 };
typedef struct ml_batched_prove_plan ml_batched_prove_plan;
int ml_batched_prove_plan_create(size_t log_domain, size_t n_codes, int kind, ml_batched_prove_plan **out);
void ml_batched_prove_plan_free(ml_batched_prove_plan *p);
size_t ml_batched_prove_plan_device_bytes(const ml_batched_prove_plan *p);
size_t ml_batched_prove_plan_proof_bytes(const ml_batched_prove_plan *p);  /* == ml_bfri_proof_serialized_len of its proof */
int ml_batched_fri_prove_async(ml_batched_prove_plan *p, const void *const *codes_dev, void *transcript_dev, void *proof_dev, int *status_dev,
                               void *stream);
int ml_batched_rs_fri_prove_async(ml_batched_prove_plan *p, const void *const *coeffs_dev, void *transcript_dev, void *proof_dev,
                                  int *status_dev, void *stream);
int ml_batched_pcs_prove_async(ml_batched_prove_plan *p, const void *inputs_dev, const void *outputs_dev, const void *const *evals_dev,
                               void *transcript_dev, void *proof_dev, void *sumcheck_dev, int *status_dev, void *stream);

/* ---- sumcheck tables of arbitrary trace width (System path; SURVEY.md §8f row 4).
 * Replaces SumcheckTables as built by System::build_tables (src/constraint_system/sumcheck.rs:22-38) with
 * partial_sum (:204-232), fold (:234-247) and compute_sumcheck_polynomials (:147-202).  The reference passes the
 * composition as a Rust closure (`&impl Fn(&[F]) -> F`, :176); a closure cannot cross a C ABI, so the caller states the
 * polynomial it computes over the row:  comp(x) = sum_t coefs[t] * prod_{k < term_lens[t]} x[term_cols[...]]
 * (term_cols is the concatenation of the terms' column lists; a term of length 0 is the constant coefs[t]).
 * System::evaluate_composition (evaluation.rs:5-12) = sum_k constraint_mask[k] * expr_k(row) has exactly this form once
 * the masks and trace challenges are folded into the coefficients.  matrix: the trace, row-major [height][width].
 * Limits: width 1..16 (ML_ERR_ARG); at most 64 terms and 256 column references in all (ML_ERR_ARG); a column >= width is
 * ML_ERR_OUT_OF_RANGE.  A rejected ml_wsumcheck_set_composition leaves the previous composition in place.
 * ml_wsumcheck_compute_polynomials: composition_degree 0..15 (ML_ERR_ARG above); coeffs_out holds
 * n_vars * (composition_degree + 1) elements.  Degrees 0..3 run every round on the device; 4..15 run one host round per
 * variable.  A term may be longer than composition_degree: the result is then what the reference computes with that degree. */
typedef struct ml_wsumcheck ml_wsumcheck;
int ml_wsumcheck_build(const uint8_t *row_point, size_t n_vars, const uint8_t *matrix, size_t width, size_t height, ml_wsumcheck **out);
int ml_wsumcheck_build_dev(const uint8_t *row_point, size_t n_vars, const void *matrix_dev, size_t width, size_t height, void *stream, ml_wsumcheck **out);
void ml_wsumcheck_free(ml_wsumcheck *w);
size_t ml_wsumcheck_height(const ml_wsumcheck *w);
size_t ml_wsumcheck_width(const ml_wsumcheck *w);
int ml_wsumcheck_set_composition(ml_wsumcheck *w, size_t n_terms, const uint8_t *coefs, const uint32_t *term_lens, const uint32_t *term_cols);
int ml_wsumcheck_tables(const ml_wsumcheck *w, uint8_t *matrix_out, uint8_t *delta_out);
int ml_wsumcheck_partial_sum(ml_wsumcheck *w, const uint8_t r[16], uint8_t out[16]);                 /* :204-232 */
int ml_wsumcheck_fold(ml_wsumcheck *w, const uint8_t r[16]);                                         /* :234-247 */
int ml_wsumcheck_compute_polynomials(ml_wsumcheck *w, size_t composition_degree, ml_transcript *t, const uint8_t sum[16],
                                     uint8_t *coeffs_out, uint8_t *randoms_out);                     /* :147-202 */

/* ---- BatchedPCSProof::prove sharded over the GPUs of one box (BASELINE config 5; batched_pcs.rs:130-180) ----
 * G ranks (a power of two <= ML_MAX_PEERS), one GPU each.  Rank g encodes the polynomials j with j mod G == g, then owns leaf rows
 * [g*n/G, (g+1)*n/G) of the batched tree: their hashing, fingerprints, first fold and openings.  All exchange is kernels storing
 * into the owner's peer-visible arena over NVLink followed by device-side flags — no NCCL, no host barrier (csrc/shard.cu).
 * A handle hosts the ranks of ONE process:
 *   - all G ranks (n_local == world): a single-process caller such as the Rust crate; ready after ml_shard_create.  Devices may
 *     repeat (virtual ranks on one GPU, used by the tests);
 *   - one rank (n_local == 1): one process per GPU.  Every process exports its record (ml_shard_export), the caller all-gathers the
 *     records with whatever transport it has (72 bytes per rank) and hands all of them to ml_shard_connect.
 * The proof is byte-identical to ml_batched_pcs_prove's.  Calls on one handle are sequential; in the multi-process mode every
 * rank must make the same calls in the same order (a rank that does not arrive makes the others fail with ML_ERR_PEER after
 * MLB_SHARD_TIMEOUT_S seconds, default 20). */
typedef struct ml_shard ml_shard;
int ml_shard_create(int world, int n_local, const int *local_ranks, const int *local_devices, size_t n_polys, size_t n_vars, ml_shard **out);
void ml_shard_free(ml_shard *sh);      /* multi-process: all ranks must have returned from their last call (caller's barrier) */
size_t ml_shard_record_bytes(void);    /* 72 */
int ml_shard_num_local(const ml_shard *sh);
int ml_shard_export(ml_shard *sh, uint8_t *records_out /* num_local * 72 */);
int ml_shard_connect(ml_shard *sh, const uint8_t *records, size_t n_records /* world */);
void *ml_shard_stream(const ml_shard *sh, int local_index);   /* the local rank's main stream (for CUDA-event timing) */
size_t ml_shard_arena_bytes(const ml_shard *sh);
/* local_evals_dev: for every local rank in handle order, its n_polys/world polynomials (device pointers, n = 2^n_vars elements
 * each) in increasing global index (rank, rank + world, ...); they must be complete before the call (no stream ordering). */
int ml_shard_batch_commit_dev(ml_shard *sh, const void *const *local_evals_dev, uint8_t root_out[32]); /* Merkle::batch_commit root of the encoded batch */
int ml_shard_batched_pcs_prove_dev(ml_shard *sh, const uint8_t *inputs, size_t n_vars, const uint8_t *outputs, size_t n_polys,
                                   const void *const *local_evals_dev, ml_transcript *t, ml_bpcs_proof **out /* NULL unless rank 0 is local */);
/* host pointers, evals[j] for all n_polys polynomials; needs a handle that hosts every rank — the drop-in for batched_pcs.rs:130 */
int ml_shard_batched_pcs_prove(ml_shard *sh, const uint8_t *inputs, size_t n_vars, const uint8_t *outputs, size_t n_polys,
                               const uint8_t *const *evals, ml_transcript *t, ml_bpcs_proof **out);

/* ---- PCSProof::prove of ONE polynomial sharded over the GPUs of one box (multilinear_pcs.rs:90-136) ----
 * G ranks (a power of two <= ML_MAX_PEERS), one GPU each; rank b holds the contiguous block evals[b*n/G, (b+1)*n/G).  The blocks
 * are encoded locally and combined into the global code by a column exchange (rank r owns code columns [r*N/G^2, (r+1)*N/G^2),
 * N = 2n); the first log2(G) fold rounds run sharded (Merkle subtrees, sumcheck tables and FRI folds stay on their owners; the
 * round polynomial and challenge are computed identically on every rank), then rank 0 runs the rest of the fold chain from N/G
 * elements and the openings, reading the sharded layers from the owners' arenas (csrc/pcs_shard.cu).  Rank r therefore holds
 * about 1/G of the encoded layers, trees and tables; rank 0 additionally the tail from N/G elements.
 * The proof is byte-identical to ml_pcs_prove's and an ordinary ml_pcs_proof (ml_pcs_verify, the serializer work unchanged).
 * Handles, records, calls and errors as for ml_shard_* above (the same 72-byte IPC records, MLB_SHARD_TIMEOUT_S bounds every
 * wait).  Minimum size: n_vars >= max(1, 2*log2 G): G = 1: 1, 2: 2, 4: 4, 8: 6, 16: 8 (ML_ERR_SIZE below). */
typedef struct ml_pcs_shard ml_pcs_shard;
int ml_pcs_shard_create(int world, int n_local, const int *local_ranks, const int *local_devices, size_t n_vars, ml_pcs_shard **out);
void ml_pcs_shard_free(ml_pcs_shard *sh);   /* multi-process: all ranks must have returned from their last call (caller's barrier) */
int ml_pcs_shard_export(ml_pcs_shard *sh, uint8_t *records_out /* num_local * ml_shard_record_bytes() */);
int ml_pcs_shard_connect(ml_pcs_shard *sh, const uint8_t *records, size_t n_records /* world */);
void *ml_pcs_shard_stream(const ml_pcs_shard *sh, int local_index);  /* the local rank's main stream (for CUDA-event timing) */
size_t ml_pcs_shard_arena_bytes(const ml_pcs_shard *sh);
/* local_evals_dev[i]: local rank i's block evals[rank*n/G, (rank+1)*n/G) (device pointer, complete before the call).  Every process
 * passes the same claim and its own transcript copy; all copies end in rank 0's final state. */
int ml_pcs_shard_prove_dev(ml_pcs_shard *sh, const uint8_t *inputs, size_t n_vars, const uint8_t output[16],
                           const void *const *local_evals_dev, ml_transcript *t, ml_pcs_proof **out /* NULL unless rank 0 is local */);
/* host evals (all n) and a handle that hosts every rank: the drop-in for multilinear_pcs.rs:90 */
int ml_pcs_shard_prove(ml_pcs_shard *sh, const uint8_t *inputs, size_t n_vars, const uint8_t output[16],
                       const uint8_t *evals, size_t n, ml_transcript *t, ml_pcs_proof **out);

/* ---- BatchedPCSProof::prove with every polynomial split by block over the GPUs of one box (batched_pcs.rs:130-180) ----
 * G ranks (a power of two <= ML_MAX_PEERS), one GPU each; rank b holds the block evals_j[b*n/G, (b+1)*n/G) of EVERY polynomial j,
 * so any batch size B >= 1 runs on any G (ml_shard_* splits by polynomial and needs G | B).  Each code is encoded, exchanged and
 * combined as in ml_pcs_shard_*; layer 0 is one batched Merkle tree over the B codes whose segment subtrees stay with their owners;
 * rho, the fingerprinted sumcheck tables and the first log2(G) fold rounds are sharded, then rank 0 runs the rest of the fold
 * chain from N/G elements and the openings (csrc/bpcs_shard.cu).  Rank r holds about 1/G of every code, of the batch tree and of
 * the tables; the arena holds each code twice (layer 0 and its receive slice, ml_bpcs_shard_arena_bytes).
 * The proof is byte-identical to ml_batched_pcs_prove's and an ordinary ml_bpcs_proof (ml_batched_pcs_verify, the serializer
 * work unchanged).  Handles, records, calls and errors as for ml_shard_* above.  Minimum size: n_vars >= max(1, 2*log2 G):
 * G = 1: 1, 2: 2, 4: 4, 8: 6, 16: 8 (ML_ERR_SIZE below, and for n_polys = 0). */
typedef struct ml_bpcs_shard ml_bpcs_shard;
int ml_bpcs_shard_create(int world, int n_local, const int *local_ranks, const int *local_devices, size_t n_polys, size_t n_vars,
                         ml_bpcs_shard **out);
void ml_bpcs_shard_free(ml_bpcs_shard *sh);   /* multi-process: all ranks must have returned from their last call (caller's barrier) */
int ml_bpcs_shard_export(ml_bpcs_shard *sh, uint8_t *records_out /* num_local * ml_shard_record_bytes() */);
int ml_bpcs_shard_connect(ml_bpcs_shard *sh, const uint8_t *records, size_t n_records /* world */);
void *ml_bpcs_shard_stream(const ml_bpcs_shard *sh, int local_index);  /* the local rank's main stream (for CUDA-event timing) */
size_t ml_bpcs_shard_arena_bytes(const ml_bpcs_shard *sh);
/* local_evals_dev[i * n_polys + j]: local rank i's block of polynomial j (device pointers, complete before the call; rank-major).
 * Every process passes the same claim and its own transcript copy; all copies end in rank 0's final state. */
int ml_bpcs_shard_prove_dev(ml_bpcs_shard *sh, const uint8_t *inputs, size_t n_vars, const uint8_t *outputs, size_t n_polys,
                            const void *const *local_evals_dev, ml_transcript *t, ml_bpcs_proof **out /* NULL unless rank 0 is local */);
/* host evals[j] (all n of each polynomial) and a handle that hosts every rank: the drop-in for batched_pcs.rs:130 */
int ml_bpcs_shard_prove(ml_bpcs_shard *sh, const uint8_t *inputs, size_t n_vars, const uint8_t *outputs, size_t n_polys,
                        const uint8_t *const *evals, size_t n, ml_transcript *t, ml_bpcs_proof **out);

/* ---- FriProof::prove of ONE polynomial sharded over the GPUs of one box (fri/mod.rs:261-285), from its coefficients
 * (reed_solomon + prove, fri/mod.rs:19-28) or from its code ----
 * G ranks (a power of two <= ML_MAX_PEERS), one GPU each; n = 2^log_n coefficients, code length N = 2n.  From coefficients, rank
 * b holds the block coeffs[b*n/G, (b+1)*n/G): a cyclic transpose over the peers gives each rank one residue class of the
 * coefficients mod G, which it RS-encodes at length N/G; the column exchange and the combine of ml_pcs_shard_* (without its
 * Moebius step) give the global code.  From a code, rank b holds the block code[b*N/G, (b+1)*N/G), stored straight into the
 * owners' layer 0.  The first log2(G) fold rounds run sharded (Merkle subtrees and folds stay on their owners; every rank absorbs
 * the layer root and draws the same challenge), then rank 0 runs the rest of the fold chain from N/G elements and the openings
 * (csrc/fri_shard.cu).  Rank r holds about 1/G of the encoded layers and trees; rank 0 additionally the tail from N/G elements;
 * there are no sumcheck tables (ml_fri_shard_arena_bytes).
 * The proof is byte-identical to ml_rs_fri_prove's / ml_fri_prove's and an ordinary ml_fri_proof (ml_fri_verify and the
 * serializer work unchanged).  A code that is not an RS code gives ML_ERR_NOT_RS_CODE on every rank, in every process, within
 * the call; the handle proves normally afterwards.  Handles, records, calls and errors as for ml_pcs_shard_* above.  Minimum
 * size: log_n >= max(1, 2*log2 G): G = 1: 1, 2: 2, 4: 4, 8: 6, 16: 8 (ML_ERR_SIZE below). */
typedef struct ml_fri_shard ml_fri_shard;
int ml_fri_shard_create(int world, int n_local, const int *local_ranks, const int *local_devices, size_t log_n, ml_fri_shard **out);
void ml_fri_shard_free(ml_fri_shard *sh);   /* multi-process: all ranks must have returned from their last call (caller's barrier) */
int ml_fri_shard_export(ml_fri_shard *sh, uint8_t *records_out /* num_local * ml_shard_record_bytes() */);
int ml_fri_shard_connect(ml_fri_shard *sh, const uint8_t *records, size_t n_records /* world */);
void *ml_fri_shard_stream(const ml_fri_shard *sh, int local_index);  /* the local rank's main stream (for CUDA-event timing) */
size_t ml_fri_shard_arena_bytes(const ml_fri_shard *sh);
/* local_coeffs_dev[i]: local rank i's block coeffs[rank*n/G, (rank+1)*n/G) (device pointer, complete before the call; only read).
 * Every process passes its own transcript copy; all copies end in rank 0's final state. */
int ml_fri_shard_rs_prove_dev(ml_fri_shard *sh, const void *const *local_coeffs_dev, ml_transcript *t, ml_fri_proof **out /* NULL unless rank 0 is local */);
/* local_code_dev[i]: local rank i's block code[rank*N/G, (rank+1)*N/G) (device pointer, complete before the call; only read) */
int ml_fri_shard_prove_dev(ml_fri_shard *sh, const void *const *local_code_dev, ml_transcript *t, ml_fri_proof **out /* NULL unless rank 0 is local */);
/* host coefficients (all n) and a handle that hosts every rank: reed_solomon + prove (= ml_rs_fri_prove) */
int ml_fri_shard_rs_prove(ml_fri_shard *sh, const uint8_t *coeffs, size_t n, ml_transcript *t, ml_fri_proof **out);
/* host code (n = its length, N) and a handle that hosts every rank: the drop-in for fri/mod.rs:261.  gen_pows follows the
 * RESTRICTION of ml_fri_prove (NULL, or the domain generator's powers: ML_ERR_SIZE / ML_ERR_GENERATOR otherwise). */
int ml_fri_shard_prove(ml_fri_shard *sh, const uint8_t *code, size_t n, const uint8_t *gen_pows, size_t gen_pows_len,
                       ml_transcript *t, ml_fri_proof **out);

/* ---- BatchedFriProof::prove of B codes sharded by block over the GPUs of one box (batched_fri.rs:286-318), from the
 * polynomials' coefficients (reed_solomon of each + prove) or from their codes ----
 * G ranks (a power of two <= ML_MAX_PEERS), one GPU each; B = n_codes (1 <= B <= 2^20) polynomials of n = 2^log_n coefficients
 * each, code length N = 2n.  Rank b holds block b of every polynomial: coefficients [b*n/G, (b+1)*n/G) or code elements
 * [b*N/G, (b+1)*N/G).  Each code is built and placed as by ml_fri_shard_*; layer 0 is one batched Merkle tree over the B codes
 * whose subtrees stay with their owners (as ml_bpcs_shard_*); every rank absorbs the batch root, draws rho and the first
 * challenge; round 0 folds the fingerprinted pairs on their owners, rounds 1 .. log2(G)-1 run sharded, then rank 0 runs the rest
 * of the fold chain from N/G elements and the openings (csrc/bfri_shard.cu).  Rank r holds B received slices and the B layer-0
 * blocks (2B * 16 N/G bytes; the transposed coefficients share the layer-0 space) plus about 1/G of the other layers and trees;
 * rank 0 additionally the tail from N/G elements; there are no sumcheck tables (ml_bfri_shard_arena_bytes).
 * The proof is byte-identical to ml_batched_fri_prove's on the same codes (on reed_solomon of each polynomial for the coefficient
 * entries) and an ordinary ml_bfri_proof (ml_batched_fri_verify and the serializer work unchanged).  A code that is not an RS
 * code gives ML_ERR_NOT_RS_CODE on every rank, in every process, within the call; the handle proves normally afterwards.
 * Handles, records, calls and errors as for ml_pcs_shard_* above.  Minimum size: log_n >= max(1, 2*log2 G) (ML_ERR_SIZE below);
 * log_n = 1 at G = 1 has no folded layer and gives ML_ERR_OUT_OF_RANGE, as ml_batched_fri_prove does. */
typedef struct ml_bfri_shard ml_bfri_shard;
int ml_bfri_shard_create(int world, int n_local, const int *local_ranks, const int *local_devices, size_t n_codes, size_t log_n,
                         ml_bfri_shard **out);
void ml_bfri_shard_free(ml_bfri_shard *sh);   /* multi-process: all ranks must have returned from their last call (caller's barrier) */
int ml_bfri_shard_export(ml_bfri_shard *sh, uint8_t *records_out /* num_local * ml_shard_record_bytes() */);
int ml_bfri_shard_connect(ml_bfri_shard *sh, const uint8_t *records, size_t n_records /* world */);
void *ml_bfri_shard_stream(const ml_bfri_shard *sh, int local_index);  /* the local rank's main stream (for CUDA-event timing) */
size_t ml_bfri_shard_arena_bytes(const ml_bfri_shard *sh);
/* local_coeffs_dev[i * n_codes + j]: local rank i's block of the coefficients of polynomial j, n/G elements (device pointers,
 * complete before the call; only read).  Every process passes its own transcript copy; all copies end in rank 0's final state. */
int ml_bfri_shard_rs_prove_dev(ml_bfri_shard *sh, const void *const *local_coeffs_dev, ml_transcript *t, ml_bfri_proof **out /* NULL unless rank 0 is local */);
/* local_codes_dev[i * n_codes + j]: local rank i's block of code j, N/G elements (device pointers, complete before the call; only read) */
int ml_bfri_shard_prove_dev(ml_bfri_shard *sh, const void *const *local_codes_dev, ml_transcript *t, ml_bfri_proof **out /* NULL unless rank 0 is local */);
/* host coefficients (n_codes arrays of n) and a handle that hosts every rank: reed_solomon of each + prove */
int ml_bfri_shard_rs_prove(ml_bfri_shard *sh, const uint8_t *const *coeffs, size_t n_codes, size_t n, ml_transcript *t, ml_bfri_proof **out);
/* host codes (n_codes arrays of n = N elements) and a handle that hosts every rank: the drop-in for batched_fri.rs:286.  gen_pows
 * follows the RESTRICTION of ml_fri_prove (NULL, or the domain generator's powers: ML_ERR_SIZE / ML_ERR_GENERATOR otherwise). */
int ml_bfri_shard_prove(ml_bfri_shard *sh, const uint8_t *const *codes, size_t n_codes, size_t n, const uint8_t *gen_pows,
                        size_t gen_pows_len, ml_transcript *t, ml_bfri_proof **out);

/* ---- the width-w System sumcheck sharded over the GPUs of one box (SumcheckTables::compute_sumcheck_polynomials,
 * src/constraint_system/sumcheck.rs:147-202) ----
 * G ranks (a power of two <= ML_MAX_PEERS), one GPU each; rank b holds the contiguous row block matrix[b*h/G, (b+1)*h/G) of the
 * row-major [h][width] trace (at width 1 the block ml_pcs_shard_prove_dev takes).  The rows go to CYCLIC tables (rank g owns rows
 * i = g mod G), so every fold pair is local and the single-GPU round kernels run on each rank; each round's td point sums are
 * exchanged through the arenas, the round polynomial and challenge are computed identically on every rank, and once the tables
 * have 2^12 rows they are all-gathered and every rank runs the last rounds itself (csrc/wsumcheck_shard.cu).  Rank r holds about
 * (width + 1) * 16 * h / G bytes of tables; the caller's blocks are only read (they stay valid for a following PCS call).
 * One call computes exactly what ml_wsumcheck_build + ml_wsumcheck_set_composition + ml_wsumcheck_compute_polynomials compute:
 * every coefficient, every challenge and the final transcript, and EVERY process gets the whole result.
 * Handles, records, calls and errors as for ml_pcs_shard_* above.  width 1..16; n_vars >= max(1, log2 G) (ML_ERR_SIZE below);
 * composition_degree 0..3 (ML_ERR_ARG above); composition limits and errors as for ml_wsumcheck_set_composition. */
typedef struct ml_wsumcheck_shard ml_wsumcheck_shard;
int ml_wsumcheck_shard_create(int world, int n_local, const int *local_ranks, const int *local_devices, size_t width, size_t n_vars,
                              ml_wsumcheck_shard **out);
void ml_wsumcheck_shard_free(ml_wsumcheck_shard *sh);   /* multi-process: all ranks must have returned from their last call (caller's barrier) */
int ml_wsumcheck_shard_export(ml_wsumcheck_shard *sh, uint8_t *records_out /* num_local * ml_shard_record_bytes() */);
int ml_wsumcheck_shard_connect(ml_wsumcheck_shard *sh, const uint8_t *records, size_t n_records /* world */);
void *ml_wsumcheck_shard_stream(const ml_wsumcheck_shard *sh, int local_index);  /* the local rank's main stream (for CUDA-event timing) */
size_t ml_wsumcheck_shard_arena_bytes(const ml_wsumcheck_shard *sh);
/* the composition, as for ml_wsumcheck_set_composition; uploaded to every local rank */
int ml_wsumcheck_shard_set_composition(ml_wsumcheck_shard *sh, size_t n_terms, const uint8_t *coefs, const uint32_t *term_lens, const uint32_t *term_cols);
/* local_blocks_dev[i]: local rank i's row block (device pointer, complete before the call).  Every process passes the same row
 * point, sum and transcript copy; coeffs_out: n_vars * (composition_degree + 1) elements, randoms_out: n_vars */
int ml_wsumcheck_shard_compute_polynomials_dev(ml_wsumcheck_shard *sh, const uint8_t *row_point, size_t n_vars, const void *const *local_blocks_dev,
                                               size_t composition_degree, ml_transcript *t, const uint8_t sum[16], uint8_t *coeffs_out,
                                               uint8_t *randoms_out);
/* host rows (all height) and a handle that hosts every rank */
int ml_wsumcheck_shard_compute_polynomials(ml_wsumcheck_shard *sh, const uint8_t *row_point, size_t n_vars, const uint8_t *matrix, size_t width,
                                           size_t height, size_t composition_degree, ml_transcript *t, const uint8_t sum[16], uint8_t *coeffs_out,
                                           uint8_t *randoms_out);

/* ---- batched commit building blocks (round-1 API, kept): one rank's share of `Merkle::batch_commit`
 * (merkle_tree/mod.rs:110-131) over leaf range [leaf_begin, leaf_begin+leaf_count) of all codes.
 * codes_dev[j] points at code j's rows for this range laid out as pairs: leaf_count x 32 bytes.
 * Writes the subtree root of the range (leaf_count a power of two); ranks then all-gather the roots
 * and call ml_merkle_top_from_roots. */
int ml_batched_leaf_subtree_dev(const void *const *pairs_dev, size_t n_codes, size_t leaf_count, void *stream, uint8_t root_out[32]);
/* pairs (code[i], code[i+n/2]) of one local code written in exchange order [dest rank][local poly][row][32 B]; an out_dev
 * buffer (n_local_polys * n_code * 16 bytes) that overlaps the code is ML_ERR_ARG */
int ml_pack_pairs_dev(const void *code_dev, size_t n_code, size_t n_ranks, size_t n_local_polys, size_t local_index, void *out_dev, void *stream);
/* to_coefficient + bit_reverse + reed_solomon of one polynomial given by evaluations (batched_pcs.rs:144-149); code_dev holds 2n elements.
 * In place allowed: code_dev == evals_dev, a buffer of 2n elements whose first n are the evaluations. */
int ml_pcs_encode_dev(const void *evals_dev, size_t n, void *code_dev, void *stream);
int ml_merkle_top_from_roots(const uint8_t *roots, size_t n_roots, uint8_t root_out[32]);
/* the subtree root left in device memory (32 bytes at root_dev) for the all-gather, no host round trip; root_dev may lie inside
 * the pairs (it is written after the subtree is complete) */
int ml_batched_leaf_subtree_root_dev(const void *const *pairs_dev, size_t n_codes, size_t leaf_count, void *root_dev, void *stream);
/* Exchange fused into the pack pass: pairs of one code stored straight into the leaf-range owners' receive buffers
 * through NVLink peer mappings (no send buffer, no collective).  peer_bases[g] is rank g's receive buffer
 * ([global polynomial][row][32 B], rows = n_code/2/n_ranks) as mapped into this process (own buffer for g == rank);
 * max_ctas bounds the grid so the store pass shares the GPU with the next polynomial's NTT (0 = default).  A destination slice
 * (rows pairs of global_poly) that overlaps the code is ML_ERR_ARG. */
int ml_pack_pairs_peer_dev(const void *code_dev, size_t n_code, size_t n_ranks, size_t global_poly, void *const *peer_bases, unsigned max_ctas, void *stream);
/* peer-visible device buffers (CUDA IPC): owner allocates + publishes the 64-byte handle; peers map / unmap it */
int ml_ipc_alloc(size_t bytes, void **dev_out, uint8_t handle_out[64]);
int ml_ipc_open(const uint8_t handle[64], void **dev_out);
int ml_ipc_close(void *dev);
int ml_ipc_free(void *dev);

#ifdef __cplusplus
}
#endif
#endif
