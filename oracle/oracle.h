/*
 * ORACLE — TEST INFRASTRUCTURE ONLY.  CPU restatement of the polynomial-
 * commitment hot path of fr34za/multilinear (reference at /root/reference).
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * `--impl reference` legs may load this library; the product
 * (multilinear_b200/) never links, imports or calls it.
 *
 * PARITY UNPINNED — see oracle/field.h: the reference is Rust, cannot be built in this image and asserts no concrete value.
 * rust/golden_dump.rs + tests/golden/check_against_rust.py let a maintainer with cargo pin the golden vectors against the crate.
 * Every function cites the reference
 * file:line whose loop it restates.  Field elements cross the ABI as 16
 * little-endian bytes (src/field.rs:33-38), digests as 32 bytes.
 */
#ifndef ORACLE_H
#define ORACLE_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OR_LOG_BLOWUP 1    /* src/fri/mod.rs:16 */
#define OR_NUM_QUERIES 128 /* src/fri/mod.rs:17 */

/* status codes shared with include/multilinear_b200.h */
enum { OR_OK = 0, OR_ERR_NOT_POW2 = 1, OR_ERR_SIZE = 2, OR_ERR_RANGE = 3, OR_ERR_NOT_RS = 4, OR_ERR_GEN = 5 };
/* verifier results (FriProofError, src/fri/mod.rs:251-258) */
enum { OR_V_OK = 0, OR_V_QUERY_MISMATCH = 101, OR_V_WRONG_NUM_QUERIES = 102, OR_V_WRONG_NUM_PATHS = 103,
       OR_V_INCLUSION_HASH = 104, OR_V_INCLUSION_INDEX = 105, OR_V_LAST_RANDOM = 106, OR_V_SUMCHECK = 107 };

void or_set_threads(int n); /* OpenMP threads for the hot loops (1 = the reference's behaviour) */
int or_get_threads(void);

/* ---- field (src/field.rs, winter-math f128) ---- */
void or_fe_add(const uint8_t a[16], const uint8_t b[16], uint8_t out[16]);
void or_fe_sub(const uint8_t a[16], const uint8_t b[16], uint8_t out[16]);
void or_fe_mul(const uint8_t a[16], const uint8_t b[16], uint8_t out[16]);
void or_fe_div(const uint8_t a[16], const uint8_t b[16], uint8_t out[16]);
void or_fe_neg(const uint8_t a[16], uint8_t out[16]);
void or_fe_pow(const uint8_t a[16], const uint8_t exp_le[16], uint8_t out[16]);
void or_fe_from_i64(int64_t v, uint8_t out[16]);
void or_fe_from_u128(const uint8_t v_le[16], uint8_t out[16]);
void or_fe_mul_vec(const uint8_t *a, const uint8_t *b, size_t n, uint8_t *out);
void or_fe_add_vec(const uint8_t *a, const uint8_t *b, size_t n, uint8_t *out);
void or_fe_sub_vec(const uint8_t *a, const uint8_t *b, size_t n, uint8_t *out);
void or_synthetic_elements(uint64_t seed, size_t n, uint8_t *out); /* splitmix64 pairs, reduced by new() */

/* ---- NTT (src/ntt/mod.rs) ---- */
int or_pow2_generator(uint64_t log_size, uint8_t out[16]);          /* :42-54 ; OR_ERR_RANGE = None */
int or_pow2_generator_powers(uint64_t log_size, uint8_t *out);      /* :18-28 */
int or_bit_reverse_permutation(uint8_t *values, size_t n, size_t elem_bytes); /* :113-123 */
int or_ntt(const uint8_t *coeffs, size_t n, const uint8_t gen[16], uint8_t *evals);  /* :69-110 */
int or_intt(const uint8_t *evals, size_t n, const uint8_t gen[16], uint8_t *coeffs); /* :132-173 */
int or_poly_evaluate(const uint8_t *coeffs, size_t n, const uint8_t x[16], uint8_t out[16]); /* :62-67 */
int or_reed_solomon(const uint8_t *coeffs, size_t n, const uint8_t gen[16], uint8_t *code); /* src/fri/mod.rs:19-28 */

/* ---- multilinear polynomials (src/polynomials.rs) ---- */
int or_mle_to_coefficient(const uint8_t *evals, size_t len, uint8_t *coeffs);   /* :150-163 */
int or_mle_to_evaluation(const uint8_t *coeffs, size_t len, uint8_t *evals);    /* :111-124 */
int or_mle_evals_evaluate(const uint8_t *evals, size_t len, const uint8_t *args, size_t n_args, uint8_t out[16]);   /* :165-187 */
int or_mle_coeffs_evaluate(const uint8_t *coeffs, size_t len, const uint8_t *args, size_t n_args, uint8_t out[16]); /* :126-146 */
int or_interpolate(const uint8_t *evals, size_t n, uint8_t *coeffs);            /* :51-86 */

/* ---- SHA-256 / transcript (src/transcript.rs) ---- */
void or_sha256_oneshot(const uint8_t *data, size_t len, uint8_t out[32]);
typedef struct or_transcript or_transcript;
or_transcript *or_transcript_new(void);                                  /* :17-21 */
or_transcript *or_transcript_clone(const or_transcript *t);              /* #[derive(Clone)] :5 */
void or_transcript_free(or_transcript *t);
void or_transcript_absorb(or_transcript *t, const uint8_t *bytes, size_t len); /* :31-33 */
void or_transcript_random(const or_transcript *t, uint8_t out[32]);      /* :23-29 */
void or_transcript_next_challenge(or_transcript *t, uint8_t out[16]);    /* :35-38 */

/* ---- Merkle (src/merkle_tree/mod.rs) ---- */
typedef struct or_merkle or_merkle;
or_merkle *or_merkle_commit(const uint8_t *data, size_t item_bytes, size_t n_items); /* :65-85 ; NULL = panic */
or_merkle *or_merkle_batch_commit(const uint8_t *const *data, size_t n_batches, size_t item_bytes, size_t n_items); /* :92-131 */
void or_merkle_free(or_merkle *m);
void or_merkle_root(const or_merkle *m, uint8_t out[32]);                /* :27-29 */
size_t or_merkle_num_layers(const or_merkle *m);
size_t or_merkle_layer_len(const or_merkle *m, size_t layer);
void or_merkle_layer(const or_merkle *m, size_t layer, uint8_t *out);
/* open / batch_open (:31-58, :134-175): value is item_bytes (n_batches*item_bytes for a batched tree);
 * dirs[i] = 0 Left / 1 Right = side the SIBLING is on.  OR_ERR_RANGE = None. */
int or_merkle_open(const or_merkle *m, size_t index, uint8_t *value, uint8_t *digests, uint8_t *dirs, size_t *path_len);
/* MerkleInclusionPath::verify / batch_verify (:216-246, :253-293) */
int or_merkle_path_verify(const uint8_t *value, size_t value_bytes, const uint8_t *digests, const uint8_t *dirs,
                          size_t path_len, const uint8_t root[32], size_t index);

/* ---- FRI (src/fri/mod.rs) ---- */
typedef struct or_fri or_fri;
typedef struct or_fri_proof or_fri_proof;
or_fri *or_fri_init(const uint8_t *code, size_t n, or_transcript *t);    /* :58-76 */
int or_fri_fold_step(or_fri *f, const uint8_t *gen_pows, size_t gen_pows_len, size_t k, const uint8_t r[16], or_transcript *t); /* :79-134 */
or_fri *or_fri_fold(const uint8_t *gen_pows, size_t gen_pows_len, const uint8_t *code, size_t n, or_transcript *t, int *status); /* :136-145 */
void or_fri_free(or_fri *f);
size_t or_fri_num_trees(const or_fri *f);
const or_merkle *or_fri_tree(const or_fri *f, size_t i);
void or_fri_tree_data(const or_fri *f, size_t i, uint8_t *pairs_out);    /* merkle_trees[i].data as 32-byte pairs */
void or_fri_fold_roots(const or_fri *f, uint8_t *out);                   /* :147-152 */
int or_fri_last_element(const or_fri *f, uint8_t out[16]);               /* 1 if Some */
or_fri_proof *or_fri_prove(const uint8_t *code, size_t n, const uint8_t *gen_pows, size_t gen_pows_len, or_transcript *t, int *status); /* :261-285 */
int or_fri_verify(const or_fri_proof *p);                                /* :287-309 */
void or_fri_proof_free(or_fri_proof *p);
size_t or_fri_proof_serialized_len(const or_fri_proof *p);
void or_fri_proof_serialize(const or_fri_proof *p, uint8_t *out);        /* bincode fixed-int LE of FriProof (:239-249, :367-369) */
size_t or_fri_proof_num_commitments(const or_fri_proof *p);
void or_fri_proof_commitments(const or_fri_proof *p, uint8_t *out);
void or_fri_proof_last(const or_fri_proof *p, uint8_t last_elem[16], uint8_t last_random[32]);

/* ---- sumcheck tables, PCS specialisation (src/constraint_system/sumcheck.rs:127-277) ---- */
typedef struct or_sumcheck or_sumcheck;
or_sumcheck *or_sumcheck_build_tables_for_pcs(const uint8_t *inputs, size_t n_vars, const uint8_t *evals, size_t height); /* :128-145 */
void or_sumcheck_free(or_sumcheck *s);
size_t or_sumcheck_height(const or_sumcheck *s);
void or_sumcheck_tables(const or_sumcheck *s, uint8_t *matrix_out, uint8_t *delta_out); /* current height entries each */
void or_sumcheck_partial_sum(const or_sumcheck *s, const uint8_t r[16], uint8_t out[16]); /* :204-232, composition x[0] */
void or_sumcheck_fold(or_sumcheck *s, const uint8_t r[16]);                               /* :234-247 */
/* :174-202; total_degree 0 (the reference reads evals[1] of one point and panics): OR_ERR_SIZE, nothing touched */
int or_sumcheck_compute_polynomial(or_sumcheck *s, size_t total_degree, uint8_t previous_sum[16], or_transcript *t,
                                   uint8_t *nonzero_coeffs_out, uint8_t r_out[16]);
void or_sumcheck_compute_polynomials(or_sumcheck *s, size_t composition_degree, or_transcript *t, const uint8_t sum[16],
                                     uint8_t *coeffs_out, uint8_t *randoms_out);          /* :147-172 */
void or_delta_evaluate(const uint8_t *data, const uint8_t *points, size_t n, uint8_t out[16]); /* evaluation.rs:80-90 */

/* ---- width-w sumcheck tables (System path, src/constraint_system/sumcheck.rs:21-38, 147-247); the composition closure is
 * restated as a sparse polynomial over the row: sum_t coef[t] * prod_k x[cols[..]] ---- */
typedef struct or_wsumcheck or_wsumcheck;
or_wsumcheck *or_wsumcheck_build(const uint8_t *row_point, size_t n_vars, const uint8_t *matrix, size_t width, size_t height); /* :22-38 */
void or_wsumcheck_free(or_wsumcheck *s);
size_t or_wsumcheck_height(const or_wsumcheck *s);
void or_wsumcheck_tables(const or_wsumcheck *s, uint8_t *matrix_out, uint8_t *delta_out);
int or_wsumcheck_set_composition(or_wsumcheck *s, size_t n_terms, const uint8_t *coefs, const uint32_t *term_lens, const uint32_t *term_cols);
void or_wsumcheck_partial_sum(const or_wsumcheck *s, const uint8_t r[16], uint8_t out[16]);   /* :204-232 */
void or_wsumcheck_fold(or_wsumcheck *s, const uint8_t r[16]);                                 /* :234-247 */
void or_wsumcheck_compute_polynomials(or_wsumcheck *s, size_t composition_degree, or_transcript *t, const uint8_t sum[16],
                                      uint8_t *coeffs_out, uint8_t *randoms_out);             /* :147-202 */
void or_trace_evaluate(const uint8_t *matrix, size_t width, size_t height, const uint8_t *points, uint8_t *out); /* evaluation.rs:33-48 */
void or_mask_evaluate(size_t index, size_t n_vars, const uint8_t *points, uint8_t out[16]);   /* evaluation.rs:56-73 */

/* ---- multilinear PCS (src/fri/multilinear_pcs.rs) ---- */
typedef struct or_pcs_proof or_pcs_proof;
or_pcs_proof *or_pcs_prove(const uint8_t *inputs, size_t n_vars, const uint8_t output[16], const uint8_t *evals, size_t n,
                           or_transcript *t, int *status);               /* :90-136 */
int or_pcs_verify(const or_pcs_proof *p, or_transcript *t);              /* :138-190 */
void or_pcs_proof_free(or_pcs_proof *p);
const or_fri_proof *or_pcs_proof_fri(const or_pcs_proof *p);
size_t or_pcs_proof_num_rounds(const or_pcs_proof *p);
void or_pcs_proof_sumcheck_coeffs(const or_pcs_proof *p, uint8_t *out);  /* rounds x 2 x 16 bytes */

/* ---- batched FRI / PCS (src/fri/batched_fri.rs, src/fri/batched_pcs.rs) ---- */
typedef struct or_bfri_proof or_bfri_proof;
void or_fingerprint(const uint8_t r[16], const uint8_t *coeffs, size_t n, uint8_t out[16]); /* batched_fri.rs:30-38 */
or_bfri_proof *or_batched_fri_prove(const uint8_t *const *codes, size_t n_codes, size_t n, const uint8_t *gen_pows,
                                    size_t gen_pows_len, or_transcript *t, int *status);   /* batched_fri.rs:286-318 */
int or_batched_fri_verify(const or_bfri_proof *p);                       /* batched_fri.rs:320-354 */
void or_bfri_proof_free(or_bfri_proof *p);
size_t or_bfri_proof_serialized_len(const or_bfri_proof *p);
void or_bfri_proof_serialize(const or_bfri_proof *p, uint8_t *out);
void or_bfri_proof_batch_commitment(const or_bfri_proof *p, uint8_t out[32]);
size_t or_bfri_proof_num_commitments(const or_bfri_proof *p);
void or_bfri_proof_commitments(const or_bfri_proof *p, uint8_t *out);
void or_bfri_proof_last(const or_bfri_proof *p, uint8_t last_elem[16], uint8_t last_random[32]);

typedef struct or_bpcs_proof or_bpcs_proof;
or_bpcs_proof *or_batched_pcs_prove(const uint8_t *inputs, size_t n_vars, const uint8_t *outputs, size_t n_polys,
                                    const uint8_t *const *evals, size_t n, or_transcript *t, int *status); /* batched_pcs.rs:130-180 */
int or_batched_pcs_verify(const or_bpcs_proof *p, or_transcript *t);    /* batched_pcs.rs:182-253 */
void or_bpcs_proof_free(or_bpcs_proof *p);
const or_bfri_proof *or_bpcs_proof_fri(const or_bpcs_proof *p);
size_t or_bpcs_proof_num_rounds(const or_bpcs_proof *p);
void or_bpcs_proof_sumcheck_coeffs(const or_bpcs_proof *p, uint8_t *out);

#ifdef __cplusplus
}
#endif
#endif
