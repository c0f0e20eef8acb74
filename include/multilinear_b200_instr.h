/*
 * multilinear_b200_instr.h — INSTRUMENTATION, not part of the drop-in boundary (include/multilinear_b200.h).
 * Used by bench.py and tools/ only.  ml_profile_* and ml_trace_dump read timing state kept inside
 * libmultilinear_b200.so (they are exported from it but no reference function maps to them);
 * ml_microbench lives in its own library, multilinear_b200/libmlb_instr.so, and is not linked into the product.
 */
#ifndef MULTILINEAR_B200_INSTR_H
#define MULTILINEAR_B200_INSTR_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* host-side phase trace of the host-pointer prove path (recorded when MLB_TRACE is set in the environment); prints to stderr */
void ml_trace_dump(void);

/* ---- per-kernel-group timing ----
 * ml_profile_*: when enabled, every kernel group is bracketed by CUDA events on its launch stream;
 * ml_profile_get sums device time, launches and algorithmic HBM bytes (input read once + output written once)
 * per group id: 0 ntt_pass, 1 merkle_leaf_subtree, 2 merkle_nodes, 3 merkle_top, 4 fri_fold, 5 sumcheck_sums,
 * 6 sumcheck_fold, 7 mobius, 8 eq_table, 9 bit_reverse, 10 query_gather, 11 fused_tail, 12 transcript_step.
 * ml_microbench (libmlb_instr.so): integer-pipe speed-of-light loops ("modmul", "butterfly", "sha_leaf", "sha_node", "copy"). */
int ml_profile_enable(int on);
int ml_profile_reset(void);
int ml_profile_get(int id, double *total_ms, uint64_t *launches, double *alg_bytes);
int ml_profile_get_max(int id, double *mean_ms, uint64_t *launches, double *alg_bytes); /* the group's largest launches */
int ml_microbench(const char *what, size_t n, int iters, double *ms_out, double *work_out);

/* sharded prover (ml_shard_*): device time in ms between the phase marks of the last call on the first local rank's stream —
 * commit: S0 encode+pack, S1 row subtree, S2 batch root; prove: S0, S1, S2 root + rho, S2 fingerprint partials, S3 reduce,
 * S4 wait for the matrix, chain incl. S5 first fold, openings + proof (the last three on rank 0 only).  Returns how many. */
struct ml_shard;
int ml_shard_phase_ms(const struct ml_shard *sh, double *out, int cap);
/* sharded single PCS prover (ml_pcs_shard_*): the same for [S0 encode + exchange + tables, S1 combine, sharded rounds, tail fold
 * chain (rank 0), openings + proof (rank 0)] */
struct ml_pcs_shard;
int ml_pcs_shard_phase_ms(const struct ml_pcs_shard *sh, double *out, int cap);
/* block-sharded batched PCS prover (ml_bpcs_shard_*): [S0 encodes + exchange, S1 combine + batch tree, S2/S3 batch root + rho +
 * fingerprinted tables, sharded rounds, tail fold chain (rank 0), openings + proof (rank 0)] */
struct ml_bpcs_shard;
int ml_bpcs_shard_phase_ms(const struct ml_bpcs_shard *sh, double *out, int cap);
/* sharded FRI prover (ml_fri_shard_*): [S0 transpose + encode + exchange (from a code: the placement into layer 0), S1 combine
 * (from a code: the wait), sharded rounds, tail fold chain (rank 0), openings + proof (rank 0)] */
struct ml_fri_shard;
int ml_fri_shard_phase_ms(const struct ml_fri_shard *sh, double *out, int cap);
/* sharded batched FRI prover (ml_bfri_shard_*): [S0 transposes + encodes + exchange (from codes: the placement into layer 0), S1
 * combine + batch tree, S2 batch root, sharded rounds, tail fold chain (rank 0), openings + proof (rank 0)] */
struct ml_bfri_shard;
int ml_bfri_shard_phase_ms(const struct ml_bfri_shard *sh, double *out, int cap);

#ifdef __cplusplus
}
#endif
#endif
