//! `src/cuda.rs` for fr34za/multilinear — the CUDA backend behind the crate's own signatures.
//!
//! The `extern "C"` block is GENERATED from include/multilinear_b200.h (tools/abi_tools.py --write) and checked against it by
//! tests/test_abi.py (names, arity, pointer-ness), so it cannot drift from the library.  Below it: one wrapper per hot-path
//! signature of SURVEY.md §8(b), each citing the function whose body it replaces.  Source only — the graft image has no Rust
//! toolchain; the same symbols are exercised through ctypes (multilinear_b200/api.py), C (examples/pcs_prove.c) and C++
//! (include/multilinear_b200.hpp, tests/cpp/reference_tests.cpp).  INTEGRATION.md shows where each wrapper is called from.
//!
//! Data crossing the boundary: `&[Field128]` as (ptr, len) of 16-byte little-endian canonical elements (src/field.rs:33-38),
//! `HashDigest` as 32 bytes, `Direction` as u8 (0 = Left, 1 = Right), proofs as the bincode bytes of the crate's own serde derives
//! (src/fri/mod.rs:367-369) decoded with the crate's own `Deserialize` — the proof structs are never rebuilt field by field.
#![allow(dead_code, clippy::missing_safety_doc)]
use std::os::raw::{c_char, c_int, c_uint, c_void};

use crate::constraint_system::sumcheck::SumcheckPolynomial;
use crate::field::{Field, Field128};
use crate::fri::batched_fri::{BatchedFriProof, BatchedQueryProof};
use crate::fri::batched_pcs::{BatchedPCSClaim, BatchedPCSProof};
use crate::fri::multilinear_pcs::PCSProof;
use crate::fri::{FriProof, QueryProof, ReedSolomonPair, LOG_BLOWUP};
use crate::merkle_tree::{Direction, HashDigest, Merkle, MerkleInclusionPath};
use crate::ntt::{LagrangePolynomial, Polynomial};
use crate::polynomials::{MultilinearPolynomial, MultilinearPolynomialEvals};

macro_rules! opaque { ($($n:ident),*) => { $(#[repr(C)] pub struct $n { _p: [u8; 0] })* } }
opaque!(MlTranscript, MlMerkle, MlFri, MlFriProof, MlSumcheck, MlWSumcheck, MlPcsProof, MlBfriProof, MlBpcsProof, MlShard, MlBfri, MlPcsShard, MlBpcsShard, MlWSumcheckShard, MlFriShard, MlBfriShard, MlProvePlan, MlBatchedProvePlan);

const _: () = assert!(std::mem::size_of::<Field128>() == 16 && std::mem::align_of::<Field128>() == 16);
const _: () = assert!(std::mem::size_of::<ReedSolomonPair<Field128>>() == 32); // #[repr(C)], src/fri/mod.rs:30-35
const _: () = assert!(std::mem::size_of::<HashDigest>() == 32); // src/merkle_tree/mod.rs:5
const _: () = assert!(cfg!(target_endian = "little"));

#[link(name = "multilinear_b200")]
extern "C" {
    // ---- GENERATED from include/multilinear_b200.h by tools/abi_tools.py (do not edit by hand)
    pub fn ml_batched_fri_prove(codes: *const *const u8, n_codes: usize, n: usize, gen_pows: *const u8, gen_pows_len: usize, t: *mut MlTranscript, out: *mut *mut MlBfriProof) -> c_int;
    pub fn ml_batched_fri_prove_async(p: *mut MlBatchedProvePlan, codes_dev: *const *const c_void, transcript_dev: *mut c_void, proof_dev: *mut c_void, status_dev: *mut c_int, stream: *mut c_void) -> c_int;
    pub fn ml_batched_fri_verify(p: *const MlBfriProof) -> c_int;
    pub fn ml_batched_leaf_subtree_dev(pairs_dev: *const *const c_void, n_codes: usize, leaf_count: usize, stream: *mut c_void, root_out: *mut u8) -> c_int;
    pub fn ml_batched_leaf_subtree_root_dev(pairs_dev: *const *const c_void, n_codes: usize, leaf_count: usize, root_dev: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn ml_batched_pcs_prove(inputs: *const u8, n_vars: usize, outputs: *const u8, n_polys: usize, evals: *const *const u8, n: usize, t: *mut MlTranscript, out: *mut *mut MlBpcsProof) -> c_int;
    pub fn ml_batched_pcs_prove_async(p: *mut MlBatchedProvePlan, inputs_dev: *const c_void, outputs_dev: *const c_void, evals_dev: *const *const c_void, transcript_dev: *mut c_void, proof_dev: *mut c_void, sumcheck_dev: *mut c_void, status_dev: *mut c_int, stream: *mut c_void) -> c_int;
    pub fn ml_batched_pcs_prove_dev(inputs: *const u8, n_vars: usize, outputs: *const u8, n_polys: usize, evals_dev: *const *const c_void, n: usize, t: *mut MlTranscript, stream: *mut c_void, out: *mut *mut MlBpcsProof) -> c_int;
    pub fn ml_batched_pcs_verify(p: *const MlBpcsProof, t: *mut MlTranscript) -> c_int;
    pub fn ml_batched_prove_plan_create(log_domain: usize, n_codes: usize, kind: c_int, out: *mut *mut MlBatchedProvePlan) -> c_int;
    pub fn ml_batched_prove_plan_device_bytes(p: *const MlBatchedProvePlan) -> usize;
    pub fn ml_batched_prove_plan_free(p: *mut MlBatchedProvePlan);
    pub fn ml_batched_prove_plan_proof_bytes(p: *const MlBatchedProvePlan) -> usize;
    pub fn ml_batched_rs_fri_prove_async(p: *mut MlBatchedProvePlan, coeffs_dev: *const *const c_void, transcript_dev: *mut c_void, proof_dev: *mut c_void, status_dev: *mut c_int, stream: *mut c_void) -> c_int;
    pub fn ml_bfri_batch_layer(h: *const MlBfri) -> *const MlMerkle;
    pub fn ml_bfri_batched_fold_step(h: *mut MlBfri, gen_pows: *const u8, gen_pows_len: usize, r: *const u8, t: *mut MlTranscript) -> c_int;
    pub fn ml_bfri_fingerprint_r(h: *const MlBfri, out: *mut u8) -> c_int;
    pub fn ml_bfri_fold(gen_pows: *const u8, gen_pows_len: usize, codes: *const *const u8, n_codes: usize, n: usize, t: *mut MlTranscript, out: *mut *mut MlBfri) -> c_int;
    pub fn ml_bfri_free(h: *mut MlBfri);
    pub fn ml_bfri_fri_data(h: *mut MlBfri) -> *mut MlFri;
    pub fn ml_bfri_init(codes: *const *const u8, n_codes: usize, n: usize, t: *mut MlTranscript, out: *mut *mut MlBfri) -> c_int;
    pub fn ml_bfri_num_codes(h: *const MlBfri) -> usize;
    pub fn ml_bfri_open_query_at(h: *const MlBfri, index: usize, batch_values: *mut u8, batch_digests: *mut u8, batch_dirs: *mut u8, batch_path_len: *mut usize, values: *mut u8, digests: *mut u8, dirs: *mut u8, path_lens: *mut usize) -> c_int;
    pub fn ml_bfri_proof_batch_commitment(p: *const MlBfriProof, out: *mut u8) -> c_int;
    pub fn ml_bfri_proof_commitments(p: *const MlBfriProof, out: *mut u8) -> c_int;
    pub fn ml_bfri_proof_deserialize(blob: *const u8, len: usize, out: *mut *mut MlBfriProof) -> c_int;
    pub fn ml_bfri_proof_free(p: *mut MlBfriProof);
    pub fn ml_bfri_proof_last(p: *const MlBfriProof, last_elem: *mut u8, last_random: *mut u8) -> c_int;
    pub fn ml_bfri_proof_num_commitments(p: *const MlBfriProof) -> usize;
    pub fn ml_bfri_proof_serialize(p: *const MlBfriProof, out: *mut u8) -> c_int;
    pub fn ml_bfri_proof_serialized_len(p: *const MlBfriProof) -> usize;
    pub fn ml_bfri_shard_arena_bytes(sh: *const MlBfriShard) -> usize;
    pub fn ml_bfri_shard_connect(sh: *mut MlBfriShard, records: *const u8, n_records: usize) -> c_int;
    pub fn ml_bfri_shard_create(world: c_int, n_local: c_int, local_ranks: *const c_int, local_devices: *const c_int, n_codes: usize, log_n: usize, out: *mut *mut MlBfriShard) -> c_int;
    pub fn ml_bfri_shard_export(sh: *mut MlBfriShard, records_out: *mut u8) -> c_int;
    pub fn ml_bfri_shard_free(sh: *mut MlBfriShard);
    pub fn ml_bfri_shard_prove(sh: *mut MlBfriShard, codes: *const *const u8, n_codes: usize, n: usize, gen_pows: *const u8, gen_pows_len: usize, t: *mut MlTranscript, out: *mut *mut MlBfriProof) -> c_int;
    pub fn ml_bfri_shard_prove_dev(sh: *mut MlBfriShard, local_codes_dev: *const *const c_void, t: *mut MlTranscript, out: *mut *mut MlBfriProof) -> c_int;
    pub fn ml_bfri_shard_rs_prove(sh: *mut MlBfriShard, coeffs: *const *const u8, n_codes: usize, n: usize, t: *mut MlTranscript, out: *mut *mut MlBfriProof) -> c_int;
    pub fn ml_bfri_shard_rs_prove_dev(sh: *mut MlBfriShard, local_coeffs_dev: *const *const c_void, t: *mut MlTranscript, out: *mut *mut MlBfriProof) -> c_int;
    pub fn ml_bfri_shard_stream(sh: *const MlBfriShard, local_index: c_int) -> *mut c_void;
    pub fn ml_bit_reverse_permutation(values: *mut u8, n: usize, elem_bytes: usize) -> c_int;
    pub fn ml_bpcs_proof_free(p: *mut MlBpcsProof);
    pub fn ml_bpcs_proof_fri(p: *const MlBpcsProof) -> *const MlBfriProof;
    pub fn ml_bpcs_proof_num_rounds(p: *const MlBpcsProof) -> usize;
    pub fn ml_bpcs_proof_sumcheck_coeffs(p: *const MlBpcsProof, out: *mut u8) -> c_int;
    pub fn ml_bpcs_shard_arena_bytes(sh: *const MlBpcsShard) -> usize;
    pub fn ml_bpcs_shard_connect(sh: *mut MlBpcsShard, records: *const u8, n_records: usize) -> c_int;
    pub fn ml_bpcs_shard_create(world: c_int, n_local: c_int, local_ranks: *const c_int, local_devices: *const c_int, n_polys: usize, n_vars: usize, out: *mut *mut MlBpcsShard) -> c_int;
    pub fn ml_bpcs_shard_export(sh: *mut MlBpcsShard, records_out: *mut u8) -> c_int;
    pub fn ml_bpcs_shard_free(sh: *mut MlBpcsShard);
    pub fn ml_bpcs_shard_prove(sh: *mut MlBpcsShard, inputs: *const u8, n_vars: usize, outputs: *const u8, n_polys: usize, evals: *const *const u8, n: usize, t: *mut MlTranscript, out: *mut *mut MlBpcsProof) -> c_int;
    pub fn ml_bpcs_shard_prove_dev(sh: *mut MlBpcsShard, inputs: *const u8, n_vars: usize, outputs: *const u8, n_polys: usize, local_evals_dev: *const *const c_void, t: *mut MlTranscript, out: *mut *mut MlBpcsProof) -> c_int;
    pub fn ml_bpcs_shard_stream(sh: *const MlBpcsShard, local_index: c_int) -> *mut c_void;
    pub fn ml_delta_evaluate(data: *const u8, points: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn ml_dev_alloc(bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn ml_dev_download(dst_host: *mut c_void, src_dev: *const c_void, bytes: usize) -> c_int;
    pub fn ml_dev_free(p: *mut c_void) -> c_int;
    pub fn ml_dev_upload(dst_dev: *mut c_void, src_host: *const c_void, bytes: usize) -> c_int;
    pub fn ml_device_count(count: *mut c_int) -> c_int;
    pub fn ml_device_name(out: *mut c_char, cap: usize) -> c_int;
    pub fn ml_fe_add_vec(a: *const u8, b: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn ml_fe_from_i64_vec(v: *const i64, n: usize, out: *mut u8) -> c_int;
    pub fn ml_fe_from_wide_vec(v: *const u8, n: usize, variant: c_int, out: *mut u8) -> c_int;
    pub fn ml_fe_inv_vec(a: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn ml_fe_mul_vec(a: *const u8, b: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn ml_fe_pow_vec(a: *const u8, exp_le: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn ml_fe_sub_vec(a: *const u8, b: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn ml_fingerprint(r: *const u8, coeffs: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn ml_fri_fold(gen_pows: *const u8, gen_pows_len: usize, code: *const u8, n: usize, t: *mut MlTranscript, out: *mut *mut MlFri) -> c_int;
    pub fn ml_fri_fold_dev(code_dev: *const c_void, n: usize, t: *mut MlTranscript, stream: *mut c_void, out: *mut *mut MlFri) -> c_int;
    pub fn ml_fri_fold_roots(f: *const MlFri, out: *mut u8) -> c_int;
    pub fn ml_fri_fold_step(f: *mut MlFri, gen_pows: *const u8, gen_pows_len: usize, k: usize, r: *const u8, t: *mut MlTranscript) -> c_int;
    pub fn ml_fri_free(f: *mut MlFri);
    pub fn ml_fri_init(code: *const u8, n: usize, t: *mut MlTranscript, out: *mut *mut MlFri) -> c_int;
    pub fn ml_fri_init_dev(code_dev: *const c_void, n: usize, t: *mut MlTranscript, stream: *mut c_void, out: *mut *mut MlFri) -> c_int;
    pub fn ml_fri_last_element(f: *const MlFri, out: *mut u8, is_some: *mut c_int) -> c_int;
    pub fn ml_fri_num_trees(f: *const MlFri) -> usize;
    pub fn ml_fri_open_query_at(f: *const MlFri, index: usize, values: *mut u8, digests: *mut u8, dirs: *mut u8, path_lens: *mut usize) -> c_int;
    pub fn ml_fri_proof_commitments(p: *const MlFriProof, out: *mut u8) -> c_int;
    pub fn ml_fri_proof_deserialize(blob: *const u8, len: usize, out: *mut *mut MlFriProof) -> c_int;
    pub fn ml_fri_proof_free(p: *mut MlFriProof);
    pub fn ml_fri_proof_last(p: *const MlFriProof, last_elem: *mut u8, last_random: *mut u8) -> c_int;
    pub fn ml_fri_proof_num_commitments(p: *const MlFriProof) -> usize;
    pub fn ml_fri_proof_serialize(p: *const MlFriProof, out: *mut u8) -> c_int;
    pub fn ml_fri_proof_serialized_len(p: *const MlFriProof) -> usize;
    pub fn ml_fri_prove(code: *const u8, n: usize, gen_pows: *const u8, gen_pows_len: usize, t: *mut MlTranscript, out: *mut *mut MlFriProof) -> c_int;
    pub fn ml_fri_prove_async(p: *mut MlProvePlan, code_dev: *const c_void, transcript_dev: *mut c_void, proof_dev: *mut c_void, status_dev: *mut c_int, stream: *mut c_void) -> c_int;
    pub fn ml_fri_prove_dev(code_dev: *const c_void, n: usize, t: *mut MlTranscript, stream: *mut c_void, out: *mut *mut MlFriProof) -> c_int;
    pub fn ml_fri_shard_arena_bytes(sh: *const MlFriShard) -> usize;
    pub fn ml_fri_shard_connect(sh: *mut MlFriShard, records: *const u8, n_records: usize) -> c_int;
    pub fn ml_fri_shard_create(world: c_int, n_local: c_int, local_ranks: *const c_int, local_devices: *const c_int, log_n: usize, out: *mut *mut MlFriShard) -> c_int;
    pub fn ml_fri_shard_export(sh: *mut MlFriShard, records_out: *mut u8) -> c_int;
    pub fn ml_fri_shard_free(sh: *mut MlFriShard);
    pub fn ml_fri_shard_prove(sh: *mut MlFriShard, code: *const u8, n: usize, gen_pows: *const u8, gen_pows_len: usize, t: *mut MlTranscript, out: *mut *mut MlFriProof) -> c_int;
    pub fn ml_fri_shard_prove_dev(sh: *mut MlFriShard, local_code_dev: *const *const c_void, t: *mut MlTranscript, out: *mut *mut MlFriProof) -> c_int;
    pub fn ml_fri_shard_rs_prove(sh: *mut MlFriShard, coeffs: *const u8, n: usize, t: *mut MlTranscript, out: *mut *mut MlFriProof) -> c_int;
    pub fn ml_fri_shard_rs_prove_dev(sh: *mut MlFriShard, local_coeffs_dev: *const *const c_void, t: *mut MlTranscript, out: *mut *mut MlFriProof) -> c_int;
    pub fn ml_fri_shard_stream(sh: *const MlFriShard, local_index: c_int) -> *mut c_void;
    pub fn ml_fri_tree(f: *const MlFri, i: usize, tree: *mut *const MlMerkle) -> c_int;
    pub fn ml_fri_tree_data(f: *const MlFri, i: usize, pairs_out: *mut u8) -> c_int;
    pub fn ml_fri_verify(p: *const MlFriProof) -> c_int;
    pub fn ml_host_alloc_pinned(bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn ml_host_free_pinned(p: *mut c_void) -> c_int;
    pub fn ml_host_register(p: *mut c_void, bytes: usize) -> c_int;
    pub fn ml_host_unregister(p: *mut c_void) -> c_int;
    pub fn ml_intt(evals: *const u8, n: usize, gen_: *const u8, coeffs: *mut u8) -> c_int;
    pub fn ml_intt_dev(evals_dev: *const c_void, n: usize, gen_: *const u8, coeffs_dev: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn ml_ipc_alloc(bytes: usize, dev_out: *mut *mut c_void, handle_out: *mut u8) -> c_int;
    pub fn ml_ipc_close(dev: *mut c_void) -> c_int;
    pub fn ml_ipc_free(dev: *mut c_void) -> c_int;
    pub fn ml_ipc_open(handle: *const u8, dev_out: *mut *mut c_void) -> c_int;
    pub fn ml_kernel_launches() -> u64;
    pub fn ml_last_error() -> *const c_char;
    pub fn ml_merkle_batch_commit(data: *const *const u8, n_batches: usize, item_bytes: usize, n_items: usize, out: *mut *mut MlMerkle) -> c_int;
    pub fn ml_merkle_commit(data: *const u8, item_bytes: usize, n_items: usize, out: *mut *mut MlMerkle) -> c_int;
    pub fn ml_merkle_commit_rs_code_dev(code_dev: *const c_void, n: usize, stream: *mut c_void, out: *mut *mut MlMerkle) -> c_int;
    pub fn ml_merkle_free(m: *mut MlMerkle);
    pub fn ml_merkle_layer(m: *const MlMerkle, layer: usize, out: *mut u8) -> c_int;
    pub fn ml_merkle_layer_len(m: *const MlMerkle, layer: usize) -> usize;
    pub fn ml_merkle_num_layers(m: *const MlMerkle) -> usize;
    pub fn ml_merkle_open(m: *const MlMerkle, index: usize, value: *mut u8, digests: *mut u8, dirs: *mut u8, path_len: *mut usize) -> c_int;
    pub fn ml_merkle_path_verify(value: *const u8, value_bytes: usize, digests: *const u8, dirs: *const u8, path_len: usize, root: *const u8, index: usize) -> c_int;
    pub fn ml_merkle_root(m: *const MlMerkle, out: *mut u8) -> c_int;
    pub fn ml_merkle_top_from_roots(roots: *const u8, n_roots: usize, root_out: *mut u8) -> c_int;
    pub fn ml_mle_coeffs_evaluate(coeffs: *const u8, len: usize, args: *const u8, n_args: usize, out: *mut u8) -> c_int;
    pub fn ml_mle_evals_evaluate(evals: *const u8, len: usize, args: *const u8, n_args: usize, out: *mut u8) -> c_int;
    pub fn ml_mle_evals_evaluate_dev(evals_dev: *const c_void, len: usize, args: *const u8, n_args: usize, out: *mut u8, stream: *mut c_void) -> c_int;
    pub fn ml_mle_to_coefficient(evals: *const u8, len: usize, coeffs: *mut u8) -> c_int;
    pub fn ml_mle_to_coefficient_dev(evals_dev: *const c_void, len: usize, coeffs_dev: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn ml_mle_to_evaluation(coeffs: *const u8, len: usize, evals: *mut u8) -> c_int;
    pub fn ml_mle_to_evaluation_dev(coeffs_dev: *const c_void, len: usize, evals_dev: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn ml_ntt(coeffs: *const u8, n: usize, gen_: *const u8, evals: *mut u8) -> c_int;
    pub fn ml_ntt_dev(coeffs_dev: *const c_void, n: usize, gen_: *const u8, evals_dev: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn ml_pack_pairs_dev(code_dev: *const c_void, n_code: usize, n_ranks: usize, n_local_polys: usize, local_index: usize, out_dev: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn ml_pack_pairs_peer_dev(code_dev: *const c_void, n_code: usize, n_ranks: usize, global_poly: usize, peer_bases: *const *mut c_void, max_ctas: c_uint, stream: *mut c_void) -> c_int;
    pub fn ml_pcs_encode_dev(evals_dev: *const c_void, n: usize, code_dev: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn ml_pcs_proof_free(p: *mut MlPcsProof);
    pub fn ml_pcs_proof_fri(p: *const MlPcsProof) -> *const MlFriProof;
    pub fn ml_pcs_proof_num_rounds(p: *const MlPcsProof) -> usize;
    pub fn ml_pcs_proof_sumcheck_coeffs(p: *const MlPcsProof, out: *mut u8) -> c_int;
    pub fn ml_pcs_prove(inputs: *const u8, n_vars: usize, output: *const u8, evals: *const u8, n: usize, t: *mut MlTranscript, out: *mut *mut MlPcsProof) -> c_int;
    pub fn ml_pcs_prove_async(p: *mut MlProvePlan, inputs_dev: *const c_void, output_dev: *const c_void, evals_dev: *const c_void, transcript_dev: *mut c_void, proof_dev: *mut c_void, sumcheck_dev: *mut c_void, status_dev: *mut c_int, stream: *mut c_void) -> c_int;
    pub fn ml_pcs_prove_dev(inputs: *const u8, n_vars: usize, output: *const u8, evals_dev: *const c_void, n: usize, t: *mut MlTranscript, stream: *mut c_void, out: *mut *mut MlPcsProof) -> c_int;
    pub fn ml_pcs_shard_arena_bytes(sh: *const MlPcsShard) -> usize;
    pub fn ml_pcs_shard_connect(sh: *mut MlPcsShard, records: *const u8, n_records: usize) -> c_int;
    pub fn ml_pcs_shard_create(world: c_int, n_local: c_int, local_ranks: *const c_int, local_devices: *const c_int, n_vars: usize, out: *mut *mut MlPcsShard) -> c_int;
    pub fn ml_pcs_shard_export(sh: *mut MlPcsShard, records_out: *mut u8) -> c_int;
    pub fn ml_pcs_shard_free(sh: *mut MlPcsShard);
    pub fn ml_pcs_shard_prove(sh: *mut MlPcsShard, inputs: *const u8, n_vars: usize, output: *const u8, evals: *const u8, n: usize, t: *mut MlTranscript, out: *mut *mut MlPcsProof) -> c_int;
    pub fn ml_pcs_shard_prove_dev(sh: *mut MlPcsShard, inputs: *const u8, n_vars: usize, output: *const u8, local_evals_dev: *const *const c_void, t: *mut MlTranscript, out: *mut *mut MlPcsProof) -> c_int;
    pub fn ml_pcs_shard_stream(sh: *const MlPcsShard, local_index: c_int) -> *mut c_void;
    pub fn ml_pcs_verify(p: *const MlPcsProof, t: *mut MlTranscript) -> c_int;
    pub fn ml_poly_evaluate(coeffs: *const u8, n: usize, x: *const u8, out: *mut u8) -> c_int;
    pub fn ml_poly_evaluate_over_domain(coeffs: *const u8, n: usize, evals_out: *mut u8) -> c_int;
    pub fn ml_poly_interpolate(evals: *const u8, n: usize, coeffs_out: *mut u8) -> c_int;
    pub fn ml_pool_stats(reserved_bytes: *mut u64, used_bytes: *mut u64) -> c_int;
    pub fn ml_pow2_generator(log_size: u64, out: *mut u8) -> c_int;
    pub fn ml_pow2_generator_powers(log_size: u64, out: *mut u8) -> c_int;
    pub fn ml_pow2_generator_powers_dev(log_size: u64, out_dev: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn ml_prove_plan_create(log_domain: usize, pcs: c_int, out: *mut *mut MlProvePlan) -> c_int;
    pub fn ml_prove_plan_device_bytes(p: *const MlProvePlan) -> usize;
    pub fn ml_prove_plan_free(p: *mut MlProvePlan);
    pub fn ml_prove_plan_proof_bytes(p: *const MlProvePlan) -> usize;
    pub fn ml_reed_solomon(coeffs: *const u8, n: usize, gen_: *const u8, code: *mut u8) -> c_int;
    pub fn ml_reed_solomon_dev(coeffs_dev: *const c_void, n: usize, gen_: *const u8, code_dev: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn ml_release_pools() -> c_int;
    pub fn ml_rs_fri_fold_dev(coeffs_dev: *const c_void, n: usize, t: *mut MlTranscript, stream: *mut c_void, out: *mut *mut MlFri) -> c_int;
    pub fn ml_rs_fri_prove(coeffs: *const u8, n: usize, t: *mut MlTranscript, out: *mut *mut MlFriProof) -> c_int;
    pub fn ml_rs_fri_prove_async(p: *mut MlProvePlan, coeffs_dev: *const c_void, transcript_dev: *mut c_void, proof_dev: *mut c_void, status_dev: *mut c_int, stream: *mut c_void) -> c_int;
    pub fn ml_rs_fri_prove_dev(coeffs_dev: *const c_void, n: usize, t: *mut MlTranscript, stream: *mut c_void, out: *mut *mut MlFriProof) -> c_int;
    pub fn ml_set_device(device: c_int) -> c_int;
    pub fn ml_set_pool_release_threshold(bytes: u64) -> c_int;
    pub fn ml_set_thread_stream(stream: *mut c_void, enable: c_int) -> c_int;
    pub fn ml_shard_arena_bytes(sh: *const MlShard) -> usize;
    pub fn ml_shard_batch_commit_dev(sh: *mut MlShard, local_evals_dev: *const *const c_void, root_out: *mut u8) -> c_int;
    pub fn ml_shard_batched_pcs_prove(sh: *mut MlShard, inputs: *const u8, n_vars: usize, outputs: *const u8, n_polys: usize, evals: *const *const u8, t: *mut MlTranscript, out: *mut *mut MlBpcsProof) -> c_int;
    pub fn ml_shard_batched_pcs_prove_dev(sh: *mut MlShard, inputs: *const u8, n_vars: usize, outputs: *const u8, n_polys: usize, local_evals_dev: *const *const c_void, t: *mut MlTranscript, out: *mut *mut MlBpcsProof) -> c_int;
    pub fn ml_shard_connect(sh: *mut MlShard, records: *const u8, n_records: usize) -> c_int;
    pub fn ml_shard_create(world: c_int, n_local: c_int, local_ranks: *const c_int, local_devices: *const c_int, n_polys: usize, n_vars: usize, out: *mut *mut MlShard) -> c_int;
    pub fn ml_shard_export(sh: *mut MlShard, records_out: *mut u8) -> c_int;
    pub fn ml_shard_free(sh: *mut MlShard);
    pub fn ml_shard_num_local(sh: *const MlShard) -> c_int;
    pub fn ml_shard_record_bytes() -> usize;
    pub fn ml_shard_stream(sh: *const MlShard, local_index: c_int) -> *mut c_void;
    pub fn ml_stream_create(out: *mut *mut c_void) -> c_int;
    pub fn ml_stream_destroy(stream: *mut c_void) -> c_int;
    pub fn ml_stream_synchronize(stream: *mut c_void) -> c_int;
    pub fn ml_sumcheck_build_tables_for_pcs(inputs: *const u8, n_vars: usize, evals: *const u8, height: usize, out: *mut *mut MlSumcheck) -> c_int;
    pub fn ml_sumcheck_build_tables_for_pcs_dev(inputs: *const u8, n_vars: usize, evals_dev: *const c_void, height: usize, stream: *mut c_void, out: *mut *mut MlSumcheck) -> c_int;
    pub fn ml_sumcheck_compute_polynomial(s: *mut MlSumcheck, total_degree: usize, previous_sum: *mut u8, t: *mut MlTranscript, nonzero_coeffs_out: *mut u8, r_out: *mut u8) -> c_int;
    pub fn ml_sumcheck_compute_polynomials(s: *mut MlSumcheck, composition_degree: usize, t: *mut MlTranscript, sum: *const u8, coeffs_out: *mut u8, randoms_out: *mut u8) -> c_int;
    pub fn ml_sumcheck_fold(s: *mut MlSumcheck, r: *const u8) -> c_int;
    pub fn ml_sumcheck_free(s: *mut MlSumcheck);
    pub fn ml_sumcheck_height(s: *const MlSumcheck) -> usize;
    pub fn ml_sumcheck_partial_sum(s: *const MlSumcheck, r: *const u8, out: *mut u8) -> c_int;
    pub fn ml_sumcheck_tables(s: *const MlSumcheck, matrix_out: *mut u8, delta_out: *mut u8) -> c_int;
    pub fn ml_synchronize() -> c_int;
    pub fn ml_synthetic_elements_dev(seed: u64, n: usize, out_dev: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn ml_transcript_absorb(t: *mut MlTranscript, bytes: *const u8, len: usize) -> c_int;
    pub fn ml_transcript_clone(t: *const MlTranscript, out: *mut *mut MlTranscript) -> c_int;
    pub fn ml_transcript_export(t: *const MlTranscript, state_out: *mut u8) -> c_int;
    pub fn ml_transcript_free(t: *mut MlTranscript);
    pub fn ml_transcript_import(state: *const u8, out: *mut *mut MlTranscript) -> c_int;
    pub fn ml_transcript_new(out: *mut *mut MlTranscript) -> c_int;
    pub fn ml_transcript_next_challenge(t: *mut MlTranscript, out: *mut u8) -> c_int;
    pub fn ml_transcript_random(t: *const MlTranscript, out: *mut u8) -> c_int;
    pub fn ml_transcript_state_bytes() -> usize;
    pub fn ml_trim_pools(keep_bytes: usize) -> c_int;
    pub fn ml_version() -> *const c_char;
    pub fn ml_wsumcheck_build(row_point: *const u8, n_vars: usize, matrix: *const u8, width: usize, height: usize, out: *mut *mut MlWSumcheck) -> c_int;
    pub fn ml_wsumcheck_build_dev(row_point: *const u8, n_vars: usize, matrix_dev: *const c_void, width: usize, height: usize, stream: *mut c_void, out: *mut *mut MlWSumcheck) -> c_int;
    pub fn ml_wsumcheck_compute_polynomials(w: *mut MlWSumcheck, composition_degree: usize, t: *mut MlTranscript, sum: *const u8, coeffs_out: *mut u8, randoms_out: *mut u8) -> c_int;
    pub fn ml_wsumcheck_fold(w: *mut MlWSumcheck, r: *const u8) -> c_int;
    pub fn ml_wsumcheck_free(w: *mut MlWSumcheck);
    pub fn ml_wsumcheck_height(w: *const MlWSumcheck) -> usize;
    pub fn ml_wsumcheck_partial_sum(w: *mut MlWSumcheck, r: *const u8, out: *mut u8) -> c_int;
    pub fn ml_wsumcheck_set_composition(w: *mut MlWSumcheck, n_terms: usize, coefs: *const u8, term_lens: *const u32, term_cols: *const u32) -> c_int;
    pub fn ml_wsumcheck_shard_arena_bytes(sh: *const MlWSumcheckShard) -> usize;
    pub fn ml_wsumcheck_shard_compute_polynomials(sh: *mut MlWSumcheckShard, row_point: *const u8, n_vars: usize, matrix: *const u8, width: usize, height: usize, composition_degree: usize, t: *mut MlTranscript, sum: *const u8, coeffs_out: *mut u8, randoms_out: *mut u8) -> c_int;
    pub fn ml_wsumcheck_shard_compute_polynomials_dev(sh: *mut MlWSumcheckShard, row_point: *const u8, n_vars: usize, local_blocks_dev: *const *const c_void, composition_degree: usize, t: *mut MlTranscript, sum: *const u8, coeffs_out: *mut u8, randoms_out: *mut u8) -> c_int;
    pub fn ml_wsumcheck_shard_connect(sh: *mut MlWSumcheckShard, records: *const u8, n_records: usize) -> c_int;
    pub fn ml_wsumcheck_shard_create(world: c_int, n_local: c_int, local_ranks: *const c_int, local_devices: *const c_int, width: usize, n_vars: usize, out: *mut *mut MlWSumcheckShard) -> c_int;
    pub fn ml_wsumcheck_shard_export(sh: *mut MlWSumcheckShard, records_out: *mut u8) -> c_int;
    pub fn ml_wsumcheck_shard_free(sh: *mut MlWSumcheckShard);
    pub fn ml_wsumcheck_shard_set_composition(sh: *mut MlWSumcheckShard, n_terms: usize, coefs: *const u8, term_lens: *const u32, term_cols: *const u32) -> c_int;
    pub fn ml_wsumcheck_shard_stream(sh: *const MlWSumcheckShard, local_index: c_int) -> *mut c_void;
    pub fn ml_wsumcheck_tables(w: *const MlWSumcheck, matrix_out: *mut u8, delta_out: *mut u8) -> c_int;
    pub fn ml_wsumcheck_width(w: *const MlWSumcheck) -> usize;
    // ---- END GENERATED
}

type F = Field128;

/// status -> the reference's behaviour: statuses 1 (not a power of two), 2 (size mismatch) and 4 (not an RS code) are its
/// assert!/panic! sites, so they panic with the library's message; 3 (`None`) is handled by the callers that return Option.
pub fn check(st: c_int) {
    if st != 0 {
        let msg = unsafe { std::ffi::CStr::from_ptr(ml_last_error()) }.to_string_lossy().into_owned();
        panic!("{msg}");
    }
}
fn p(x: &[F]) -> *const u8 {
    x.as_ptr().cast()
}
fn pm(x: &mut [F]) -> *mut u8 {
    x.as_mut_ptr().cast()
}
fn zeros(n: usize) -> Vec<F> {
    vec![F::from(0u128); n]
}
fn bincode_cfg() -> impl bincode::config::Config {
    bincode::config::standard().with_little_endian().with_fixed_int_encoding() // src/fri/mod.rs:367-369
}

// ------------------------------------------------------------------ src/ntt/mod.rs, src/fri/mod.rs:19-28
/// `NttField::pow_2_generator_powers` (src/ntt/mod.rs:18-28)
pub fn pow_2_generator_powers(log_size: u64) -> Option<Vec<F>> {
    if log_size > 40 {
        return None;
    }
    let mut out = zeros(1usize << log_size);
    check(unsafe { ml_pow2_generator_powers(log_size, pm(&mut out)) });
    Some(out)
}
/// `bit_reverse_permutation` (src/ntt/mod.rs:113-123)
pub fn bit_reverse_permutation(values: &mut [F]) {
    check(unsafe { ml_bit_reverse_permutation(pm(values), values.len(), 16) });
}
/// body of `Polynomial::ntt` (src/ntt/mod.rs:69-110)
pub fn ntt(poly: &Polynomial<F>, gen: F) -> LagrangePolynomial<F> {
    let mut evals = zeros(poly.coeffs.len());
    check(unsafe { ml_ntt(p(&poly.coeffs), poly.coeffs.len(), gen.as_ref().as_ptr(), pm(&mut evals)) });
    LagrangePolynomial { gen, evals }
}
/// body of `LagrangePolynomial::intt` (src/ntt/mod.rs:132-173)
pub fn intt(l: &LagrangePolynomial<F>) -> Polynomial<F> {
    let mut coeffs = zeros(l.evals.len());
    check(unsafe { ml_intt(p(&l.evals), l.evals.len(), l.gen.as_ref().as_ptr(), pm(&mut coeffs)) });
    Polynomial { coeffs }
}
/// body of `reed_solomon` (src/fri/mod.rs:19-28)
pub fn reed_solomon(coeffs: Vec<F>, gen: F) -> Vec<F> {
    let n = coeffs.len();
    let mut code = zeros(n << LOG_BLOWUP);
    check(unsafe { ml_reed_solomon(p(&coeffs), n, gen.as_ref().as_ptr(), pm(&mut code)) });
    code
}

// ------------------------------------------------------------------ src/polynomials.rs
/// `MultilinearPolynomialEvals::to_coefficient` (:150-163); the reference works on `next_power_of_two` many entries
pub fn to_coefficient(e: &MultilinearPolynomialEvals<F>) -> MultilinearPolynomial<F> {
    let mut coeffs = zeros(e.evals.len());
    check(unsafe { ml_mle_to_coefficient(p(&e.evals), e.evals.len(), pm(&mut coeffs)) });
    MultilinearPolynomial { coeffs }
}
/// `MultilinearPolynomial::to_evaluation` (:111-124)
pub fn to_evaluation(c: &MultilinearPolynomial<F>) -> MultilinearPolynomialEvals<F> {
    let mut evals = zeros(c.coeffs.len());
    check(unsafe { ml_mle_to_evaluation(p(&c.coeffs), c.coeffs.len(), pm(&mut evals)) });
    MultilinearPolynomialEvals { evals }
}
/// `MultilinearPolynomialEvals::evaluate` (:165-187)
pub fn mle_evaluate(e: &MultilinearPolynomialEvals<F>, args: &[F]) -> F {
    let mut out = zeros(1);
    check(unsafe { ml_mle_evals_evaluate(p(&e.evals), e.evals.len(), p(args), args.len(), pm(&mut out)) });
    out[0]
}
/// `MultilinearPolynomial::evaluate` (:126-146)
pub fn mle_coeffs_evaluate(c: &MultilinearPolynomial<F>, args: &[F]) -> F {
    let mut out = zeros(1);
    check(unsafe { ml_mle_coeffs_evaluate(p(&c.coeffs), c.coeffs.len(), p(args), args.len(), pm(&mut out)) });
    out[0]
}
/// `PolynomialEvals::interpolate` (:51-86) and `Polynomial::evaluate_over_domain` (:16-28) on boxed slices
pub fn interpolate(evals: &[F]) -> Box<[F]> {
    let mut c = zeros(evals.len());
    check(unsafe { ml_poly_interpolate(p(evals), evals.len(), pm(&mut c)) });
    c.into_boxed_slice()
}
pub fn evaluate_over_domain(coeffs: &[F]) -> Box<[F]> {
    let mut e = zeros(coeffs.len());
    check(unsafe { ml_poly_evaluate_over_domain(p(coeffs), coeffs.len(), pm(&mut e)) });
    e.into_boxed_slice()
}

// ------------------------------------------------------------------ src/transcript.rs
/// Drop-in for `Transcript` (src/transcript.rs:5-39): the SHA-256 state lives behind the C ABI so that prover calls can advance it
/// on the device; `new` / `random` / `absorb` / `next_challenge` / `Clone` keep their meaning.
pub struct Transcript {
    pub(crate) h: *mut MlTranscript,
}
impl Transcript {
    pub fn new() -> Self {
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_transcript_new(&mut h) });
        Self { h }
    }
    pub fn random(&self) -> [u8; 32] {
        let mut out = [0u8; 32];
        check(unsafe { ml_transcript_random(self.h, out.as_mut_ptr()) });
        out
    }
    pub fn absorb(&mut self, values: &[u8]) {
        check(unsafe { ml_transcript_absorb(self.h, values.as_ptr(), values.len()) });
    }
    pub fn next_challenge<T: Field>(&mut self) -> T {
        let mut le = [0u8; 16];
        check(unsafe { ml_transcript_next_challenge(self.h, le.as_mut_ptr()) });
        T::from(u128::from_le_bytes(le))
    }
    /// the running SHA-256 state (ml_transcript_state_bytes() bytes), as the stream-ordered provers take it in device memory
    pub fn export_state(&self) -> Vec<u8> {
        let mut out = vec![0u8; unsafe { ml_transcript_state_bytes() }];
        check(unsafe { ml_transcript_export(self.h, out.as_mut_ptr()) });
        out
    }
    /// a transcript continuing from an exported state (e.g. one a stream-ordered prove left in device memory)
    pub fn import_state(state: &[u8]) -> Self {
        assert_eq!(state.len(), unsafe { ml_transcript_state_bytes() });
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_transcript_import(state.as_ptr(), &mut h) });
        Self { h }
    }
}
impl Default for Transcript {
    fn default() -> Self {
        Self::new()
    }
}
impl Clone for Transcript {
    fn clone(&self) -> Self {
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_transcript_clone(self.h, &mut h) });
        Self { h }
    }
}
impl Drop for Transcript {
    fn drop(&mut self) {
        unsafe { ml_transcript_free(self.h) }
    }
}

// ------------------------------------------------------------------ src/merkle_tree/mod.rs
fn digest(b: &[u8]) -> HashDigest {
    HashDigest::clone_from_slice(b)
}
/// every layer of a device tree as the reference's `layers: Vec<Vec<HashDigest>>` (src/merkle_tree/mod.rs:8-11)
unsafe fn download_layers(m: *const MlMerkle) -> Vec<Vec<HashDigest>> {
    let mut layers = Vec::new();
    for l in 0..ml_merkle_num_layers(m) {
        let len = ml_merkle_layer_len(m, l);
        let mut raw = vec![0u8; 32 * len];
        check(ml_merkle_layer(m, l, raw.as_mut_ptr()));
        layers.push(raw.chunks_exact(32).map(digest).collect());
    }
    layers
}
/// body of `Merkle::commit` (src/merkle_tree/mod.rs:65-85): leaves hashed and reduced on the GPU, the struct rebuilt on the host
/// (items must all have the same byte length, which holds for every `T` the crate commits to)
pub fn merkle_commit<T: AsRef<[u8]>>(data: Vec<T>) -> Merkle<T> {
    assert!(data.len().is_power_of_two(), "Data length must be a power of two");
    let item = data[0].as_ref().len();
    let flat: Vec<u8> = data.iter().flat_map(|x| x.as_ref().iter().copied()).collect();
    let mut h = std::ptr::null_mut();
    check(unsafe { ml_merkle_commit(flat.as_ptr(), item, data.len(), &mut h) });
    let layers = unsafe { download_layers(h) };
    unsafe { ml_merkle_free(h) };
    Merkle { layers, data }
}
/// body of `Merkle::<Vec<T>>::batch_commit` (src/merkle_tree/mod.rs:92-131); `data` stays [batch][index] as the reference keeps it
/// (`batch_open` extracts the column, :134-175)
pub fn merkle_batch_commit<T: AsRef<[u8]>>(data: Vec<Vec<T>>) -> Merkle<Vec<T>> {
    assert!(!data.is_empty(), "Data must not be empty");
    let n = data[0].len();
    assert!(n.is_power_of_two(), "Each batch length must be a power of two");
    assert!(data.iter().all(|b| b.len() == n), "All batches must have the same length");
    let item = data[0][0].as_ref().len();
    let flats: Vec<Vec<u8>> = data.iter().map(|b| b.iter().flat_map(|x| x.as_ref().iter().copied()).collect()).collect();
    let ptrs: Vec<*const u8> = flats.iter().map(|f| f.as_ptr()).collect();
    let mut h = std::ptr::null_mut();
    check(unsafe { ml_merkle_batch_commit(ptrs.as_ptr(), data.len(), item, n, &mut h) });
    let layers = unsafe { download_layers(h) };
    unsafe { ml_merkle_free(h) };
    Merkle { layers, data }
}
fn path_from(digests: &[u8], dirs: &[u8]) -> Vec<(HashDigest, Direction)> {
    digests.chunks_exact(32).zip(dirs).map(|(d, &s)| (digest(d), if s == 0 { Direction::Left } else { Direction::Right })).collect()
}

// ------------------------------------------------------------------ src/fri/mod.rs
/// `FriProverData<F>` with every tree resident in HBM (src/fri/mod.rs:10-14): init / fold_step / fold / fold_roots / open_query_at
pub struct CudaFriProverData {
    h: *mut MlFri,
}
impl CudaFriProverData {
    /// `FriProverData::init` (:58-76)
    pub fn init(code: &[F], transcript: &mut Transcript) -> Self {
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_fri_init(p(code), code.len(), transcript.h, &mut h) });
        Self { h }
    }
    /// `fold_step` (:79-134)
    pub fn fold_step(&mut self, gen_pows: &[F], k: usize, r: F, transcript: &mut Transcript) {
        check(unsafe { ml_fri_fold_step(self.h, p(gen_pows), gen_pows.len(), k, r.as_ref().as_ptr(), transcript.h) });
    }
    /// `fold` (:136-145) — one call, the whole chain stays on the device
    pub fn fold(gen_pows: &[F], code: &[F], transcript: &mut Transcript) -> Self {
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_fri_fold(p(gen_pows), gen_pows.len(), p(code), code.len(), transcript.h, &mut h) });
        Self { h }
    }
    /// `fold_roots` (:147-152)
    pub fn fold_roots(&self) -> Vec<HashDigest> {
        let n = unsafe { ml_fri_num_trees(self.h) };
        let mut raw = vec![0u8; 32 * n];
        check(unsafe { ml_fri_fold_roots(self.h, raw.as_mut_ptr()) });
        raw.chunks_exact(32).map(digest).collect()
    }
    pub fn last_element(&self) -> Option<F> {
        let (mut out, mut some) = (zeros(1), 0);
        check(unsafe { ml_fri_last_element(self.h, pm(&mut out), &mut some) });
        (some != 0).then_some(out[0])
    }
    /// `open_query_at` (:154-174)
    pub fn open_query_at(&self, index: usize) -> QueryProof<F> {
        let trees = unsafe { ml_fri_num_trees(self.h) };
        let (mut values, mut lens) = (vec![0u8; 32 * trees], vec![0usize; trees]);
        let (mut digests, mut dirs) = (vec![0u8; 32 * 64 * trees], vec![0u8; 64 * trees]);
        check(unsafe { ml_fri_open_query_at(self.h, index, values.as_mut_ptr(), digests.as_mut_ptr(), dirs.as_mut_ptr(), lens.as_mut_ptr()) });
        let (mut paths, mut off) = (Vec::with_capacity(trees), 0);
        for j in 0..trees {
            let v = &values[32 * j..32 * j + 32];
            let value = ReedSolomonPair { value: fe(&v[..16]), minus_value: fe(&v[16..]) };
            paths.push(MerkleInclusionPath { value, path: path_from(&digests[32 * off..32 * (off + lens[j])], &dirs[off..off + lens[j]]) });
            off += lens[j];
        }
        QueryProof { paths }
    }
    /// the reference's struct, rebuilt on the host (`merkle_trees[i].data`, `.layers`, :10-14) for code that reads its fields
    pub fn into_reference(self) -> crate::fri::FriProverData<F> {
        let mut merkle_trees = Vec::new();
        for i in 0..unsafe { ml_fri_num_trees(self.h) } {
            let mut t: *const MlMerkle = std::ptr::null();
            check(unsafe { ml_fri_tree(self.h, i, &mut t) });
            let leaves = unsafe { ml_merkle_layer_len(t, 0) };
            let mut raw = vec![0u8; 32 * leaves];
            check(unsafe { ml_fri_tree_data(self.h, i, raw.as_mut_ptr()) });
            let data = raw.chunks_exact(32).map(|v| ReedSolomonPair { value: fe(&v[..16]), minus_value: fe(&v[16..]) }).collect();
            merkle_trees.push(Merkle { layers: unsafe { download_layers(t) }, data });
        }
        crate::fri::FriProverData { merkle_trees, last_element: self.last_element() }
    }
}
impl Drop for CudaFriProverData {
    fn drop(&mut self) {
        unsafe { ml_fri_free(self.h) }
    }
}
fn fe(le: &[u8]) -> F {
    F::from(u128::from_le_bytes(le.try_into().unwrap()))
}
unsafe fn fri_proof_from(h: *const MlFriProof) -> FriProof<F> {
    let mut blob = vec![0u8; ml_fri_proof_serialized_len(h)];
    check(ml_fri_proof_serialize(h, blob.as_mut_ptr()));
    bincode::serde::decode_from_slice(&blob, bincode_cfg()).expect("FriProof blob").0
}
/// body of `FriProof::prove` (src/fri/mod.rs:261-285)
pub fn fri_prove(code: &[F], gen_pows: &[F], transcript: &mut Transcript) -> FriProof<F> {
    let mut h = std::ptr::null_mut();
    check(unsafe { ml_fri_prove(p(code), code.len(), p(gen_pows), gen_pows.len(), transcript.h, &mut h) });
    let proof = unsafe { fri_proof_from(h) };
    unsafe { ml_fri_proof_free(h) };
    proof
}
/// `reed_solomon` + `FriProof::prove` with the code kept in HBM between the two (the commit the headline metric times)
pub fn rs_fri_prove(coeffs: &[F], transcript: &mut Transcript) -> FriProof<F> {
    let mut h = std::ptr::null_mut();
    check(unsafe { ml_rs_fri_prove(p(coeffs), coeffs.len(), transcript.h, &mut h) });
    let proof = unsafe { fri_proof_from(h) };
    unsafe { ml_fri_proof_free(h) };
    proof
}

// ------------------------------------------------------------------ src/constraint_system/sumcheck.rs (PCS specialisation)
/// `SumcheckTables<F>` of width 1 with the composition `|x| x[0]` (sumcheck.rs:127-247), tables resident in HBM
pub struct CudaSumcheckTables {
    h: *mut MlSumcheck,
}
impl CudaSumcheckTables {
    /// `build_tables_for_pcs` (:128-145)
    pub fn build_tables_for_pcs(inputs: &[F], poly: &MultilinearPolynomialEvals<F>) -> Self {
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_sumcheck_build_tables_for_pcs(p(inputs), inputs.len(), p(&poly.evals), poly.evals.len(), &mut h) });
        Self { h }
    }
    /// `partial_sum` (:204-232) for the composition `x[0]`
    pub fn partial_sum(&self, r: F) -> F {
        let mut out = zeros(1);
        check(unsafe { ml_sumcheck_partial_sum(self.h, r.as_ref().as_ptr(), pm(&mut out)) });
        out[0]
    }
    /// `fold` (:234-247)
    pub fn fold(&mut self, r: F) {
        check(unsafe { ml_sumcheck_fold(self.h, r.as_ref().as_ptr()) });
    }
    /// `compute_sumcheck_polynomial` (:174-202): returns (polynomial, r) and updates `previous_sum`
    pub fn compute_sumcheck_polynomial(&mut self, total_degree: usize, previous_sum: &mut F, transcript: &mut Transcript) -> (SumcheckPolynomial<F>, F) {
        let (mut nz, mut r, mut prev) = (zeros(total_degree), zeros(1), [*previous_sum]);
        check(unsafe { ml_sumcheck_compute_polynomial(self.h, total_degree, pm(&mut prev), transcript.h, pm(&mut nz), pm(&mut r)) });
        *previous_sum = prev[0];
        (SumcheckPolynomial { nonzero_coeffs: nz.into_boxed_slice() }, r[0])
    }
    /// `compute_sumcheck_polynomials` (:147-172): all rounds with the transcript advanced on the device
    pub fn compute_sumcheck_polynomials(&mut self, composition_degree: usize, transcript: &mut Transcript, sum: F) -> (Vec<SumcheckPolynomial<F>>, Vec<F>) {
        let rounds = unsafe { ml_sumcheck_height(self.h) }.trailing_zeros() as usize;
        let td = composition_degree + 1;
        let (mut coeffs, mut randoms) = (zeros(rounds * td), zeros(rounds));
        check(unsafe { ml_sumcheck_compute_polynomials(self.h, composition_degree, transcript.h, sum.as_ref().as_ptr(), pm(&mut coeffs), pm(&mut randoms)) });
        (coeffs.chunks_exact(td).map(|c| SumcheckPolynomial { nonzero_coeffs: c.into() }).collect(), randoms)
    }
}
impl Drop for CudaSumcheckTables {
    fn drop(&mut self) {
        unsafe { ml_sumcheck_free(self.h) }
    }
}

// ------------------------------------------------------------------ src/fri/multilinear_pcs.rs, batched_fri.rs, batched_pcs.rs
fn sumcheck_polys(flat: &[F]) -> Vec<SumcheckPolynomial<F>> {
    flat.chunks_exact(2).map(|c| SumcheckPolynomial { nonzero_coeffs: c.into() }).collect() // total_degree = 2 (multilinear_pcs.rs:57)
}
/// body of `PCSProof::prove` (src/fri/multilinear_pcs.rs:90-136)
pub fn pcs_prove(inputs: Vec<F>, output: F, poly: MultilinearPolynomialEvals<F>, transcript: &mut Transcript) -> PCSProof<F> {
    let mut h = std::ptr::null_mut();
    check(unsafe { ml_pcs_prove(p(&inputs), inputs.len(), output.as_ref().as_ptr(), p(&poly.evals), poly.evals.len(), transcript.h, &mut h) });
    unsafe { pcs_proof_from(h, inputs, output) }
}
unsafe fn pcs_proof_from(h: *mut MlPcsProof, inputs: Vec<F>, output: F) -> PCSProof<F> {
    let fri_proof = fri_proof_from(ml_pcs_proof_fri(h));
    let mut flat = zeros(2 * ml_pcs_proof_num_rounds(h));
    check(ml_pcs_proof_sumcheck_coeffs(h, pm(&mut flat)));
    ml_pcs_proof_free(h);
    PCSProof { fri_proof, sumcheck_polynomials: sumcheck_polys(&flat), inputs, output }
}
/// `PCSProof::prove` of ONE polynomial over all GPUs of the box from one process (ml_pcs_shard_*, csrc/pcs_shard.cu): rank g holds
/// the block evals[g*n/G, (g+1)*n/G); the first log2(G) fold rounds run sharded, rank 0 runs the rest.  Lower latency than
/// `pcs_prove` from n_vars ~ 20 up, and polynomials too large for one GPU.  The handle is built once per n_vars and reused; the
/// proof bytes equal `pcs_prove`'s.
pub struct ShardedPcsProver {
    h: *mut MlPcsShard,
}
impl ShardedPcsProver {
    pub fn new(n_vars: usize) -> Self {
        let mut count = 0;
        check(unsafe { ml_device_count(&mut count) });
        let mut world = 1usize << (usize::BITS - 1 - (count.max(1) as usize).leading_zeros()); // largest power of two <= GPUs
        while world > 1 && n_vars < 2 * world.trailing_zeros() as usize {
            world >>= 1; // n_vars >= 2 log2(world)
        }
        let world = world.min(16) as c_int;
        let ids: Vec<c_int> = (0..world).collect();
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_pcs_shard_create(world, world, ids.as_ptr(), ids.as_ptr(), n_vars, &mut h) });
        Self { h }
    }
    pub fn prove(&mut self, inputs: Vec<F>, output: F, poly: MultilinearPolynomialEvals<F>, transcript: &mut Transcript) -> PCSProof<F> {
        let mut h = std::ptr::null_mut();
        check(unsafe {
            ml_pcs_shard_prove(self.h, p(&inputs), inputs.len(), output.as_ref().as_ptr(), p(&poly.evals), poly.evals.len(), transcript.h, &mut h)
        });
        unsafe { pcs_proof_from(h, inputs, output) }
    }
}
impl Drop for ShardedPcsProver {
    fn drop(&mut self) {
        unsafe { ml_pcs_shard_free(self.h) }
    }
}
/// `FriProof::prove` of ONE polynomial over all GPUs of the box from one process (ml_fri_shard_*, csrc/fri_shard.cu), from its
/// 2^log_n coefficients (`reed_solomon` + prove) or from its code of 2^(log_n+1) elements: rank g holds the block g of G; the first
/// log2(G) fold rounds run sharded, rank 0 runs the rest.  The handle is built once per log_n and reused; the proof bytes equal
/// `rs_fri_prove`'s / `fri_prove`'s.
pub struct ShardedFriProver {
    h: *mut MlFriShard,
}
impl ShardedFriProver {
    pub fn new(log_n: usize) -> Self {
        let mut count = 0;
        check(unsafe { ml_device_count(&mut count) });
        let mut world = 1usize << (usize::BITS - 1 - (count.max(1) as usize).leading_zeros()); // largest power of two <= GPUs
        while world > 1 && log_n < 2 * world.trailing_zeros() as usize {
            world >>= 1; // log_n >= 2 log2(world)
        }
        let world = world.min(16) as c_int;
        let ids: Vec<c_int> = (0..world).collect();
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_fri_shard_create(world, world, ids.as_ptr(), ids.as_ptr(), log_n, &mut h) });
        Self { h }
    }
    /// body of `FriProof::prove` (src/fri/mod.rs:261-285) for a code of the handle's length
    pub fn prove(&mut self, code: &[F], gen_pows: &[F], transcript: &mut Transcript) -> FriProof<F> {
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_fri_shard_prove(self.h, p(code), code.len(), p(gen_pows), gen_pows.len(), transcript.h, &mut h) });
        let proof = unsafe { fri_proof_from(h) };
        unsafe { ml_fri_proof_free(h) };
        proof
    }
    /// `reed_solomon` (src/fri/mod.rs:19-28) + `FriProof::prove` of the handle's number of coefficients
    pub fn rs_prove(&mut self, coeffs: &[F], transcript: &mut Transcript) -> FriProof<F> {
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_fri_shard_rs_prove(self.h, p(coeffs), coeffs.len(), transcript.h, &mut h) });
        let proof = unsafe { fri_proof_from(h) };
        unsafe { ml_fri_proof_free(h) };
        proof
    }
}
impl Drop for ShardedFriProver {
    fn drop(&mut self) {
        unsafe { ml_fri_shard_free(self.h) }
    }
}
/// Stream-ordered `FriProof::prove` / `PCSProof::prove` of one domain size 2^log_domain (ml_prove_plan_*, csrc/plan.cu): the plan
/// owns every device buffer a prove needs; a call only enqueues kernels on `stream` (e.g. a cudarc stream's raw handle) and writes
/// the bincode blob, the final transcript state and the status into the caller's device buffers.  One proof in flight per plan.
pub struct ProvePlan {
    h: *mut MlProvePlan,
}
impl ProvePlan {
    pub fn new(log_domain: usize, pcs: bool) -> Self {
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_prove_plan_create(log_domain, pcs as c_int, &mut h) });
        Self { h }
    }
    /// bytes of the FriProof blob a call writes (`bincode` of the proof, fri/mod.rs:367-369)
    pub fn proof_bytes(&self) -> usize {
        unsafe { ml_prove_plan_proof_bytes(self.h) }
    }
    pub fn device_bytes(&self) -> usize {
        unsafe { ml_prove_plan_device_bytes(self.h) }
    }
    /// `reed_solomon` + `FriProof::prove` of N/2 coefficients in HBM.
    /// # Safety
    /// Every pointer is device memory of the size include/multilinear_b200.h states, 16-byte aligned, and stays valid until the
    /// stream has passed the call.
    pub unsafe fn rs_fri_prove_async(&mut self, coeffs_dev: *const c_void, transcript_dev: *mut c_void, proof_dev: *mut c_void,
                                     status_dev: *mut c_int, stream: *mut c_void) {
        check(ml_rs_fri_prove_async(self.h, coeffs_dev, transcript_dev, proof_dev, status_dev, stream));
    }
    /// `FriProof::prove` of a code of N elements in HBM.
    /// # Safety
    /// As for `rs_fri_prove_async`.
    pub unsafe fn fri_prove_async(&mut self, code_dev: *const c_void, transcript_dev: *mut c_void, proof_dev: *mut c_void,
                                  status_dev: *mut c_int, stream: *mut c_void) {
        check(ml_fri_prove_async(self.h, code_dev, transcript_dev, proof_dev, status_dev, stream));
    }
    /// `PCSProof::prove` of N/2 evaluations in HBM (a plan made with `pcs`); sumcheck_dev receives 2 * n_vars coefficients.
    /// # Safety
    /// As for `rs_fri_prove_async`.
    #[allow(clippy::too_many_arguments)]
    pub unsafe fn pcs_prove_async(&mut self, inputs_dev: *const c_void, output_dev: *const c_void, evals_dev: *const c_void,
                                  transcript_dev: *mut c_void, proof_dev: *mut c_void, sumcheck_dev: *mut c_void, status_dev: *mut c_int,
                                  stream: *mut c_void) {
        check(ml_pcs_prove_async(self.h, inputs_dev, output_dev, evals_dev, transcript_dev, proof_dev, sumcheck_dev, status_dev, stream));
    }
}
impl Drop for ProvePlan {
    fn drop(&mut self) {
        unsafe { ml_prove_plan_free(self.h) }
    }
}
/// Stream-ordered `BatchedFriProof::prove` / `BatchedPCSProof::prove` of n_codes codes of 2^log_domain elements
/// (ml_batched_prove_plan_*, csrc/bplan.cu), for one kind of call: from codes, from coefficients (reed_solomon of each first) or
/// from evaluations (PCS).  A call only enqueues kernels on `stream` and writes the bincode blob, the final transcript state, the
/// status and (PCS) the sumcheck coefficients into the caller's device buffers.  One proof in flight per plan.
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub enum BatchedPlanKind {
    Codes = 0,
    Rs = 1,
    Pcs = 2,
}
pub struct BatchedProvePlan {
    h: *mut MlBatchedProvePlan,
}
impl BatchedProvePlan {
    pub fn new(log_domain: usize, n_codes: usize, kind: BatchedPlanKind) -> Self {
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_batched_prove_plan_create(log_domain, n_codes, kind as c_int, &mut h) });
        Self { h }
    }
    /// bytes of the BatchedFriProof blob a call writes (`bincode` of the proof)
    pub fn proof_bytes(&self) -> usize {
        unsafe { ml_batched_prove_plan_proof_bytes(self.h) }
    }
    pub fn device_bytes(&self) -> usize {
        unsafe { ml_batched_prove_plan_device_bytes(self.h) }
    }
    /// `BatchedFriProof::prove` of n_codes codes of N elements in HBM (a `Codes` plan).
    /// # Safety
    /// Every pointer (those in `codes_dev` too) is device memory of the size include/multilinear_b200.h states, 16-byte aligned,
    /// and stays valid until the stream has passed the call.
    pub unsafe fn batched_fri_prove_async(&mut self, codes_dev: &[*const c_void], transcript_dev: *mut c_void, proof_dev: *mut c_void,
                                          status_dev: *mut c_int, stream: *mut c_void) {
        check(ml_batched_fri_prove_async(self.h, codes_dev.as_ptr(), transcript_dev, proof_dev, status_dev, stream));
    }
    /// `reed_solomon` of each of n_codes polynomials of N/2 coefficients in HBM + `BatchedFriProof::prove` (an `Rs` plan).
    /// # Safety
    /// As for `batched_fri_prove_async`.
    pub unsafe fn batched_rs_fri_prove_async(&mut self, coeffs_dev: &[*const c_void], transcript_dev: *mut c_void, proof_dev: *mut c_void,
                                             status_dev: *mut c_int, stream: *mut c_void) {
        check(ml_batched_rs_fri_prove_async(self.h, coeffs_dev.as_ptr(), transcript_dev, proof_dev, status_dev, stream));
    }
    /// `BatchedPCSProof::prove` of n_codes polynomials of N/2 evaluations in HBM (a `Pcs` plan); sumcheck_dev receives 2 * n_vars
    /// coefficients.
    /// # Safety
    /// As for `batched_fri_prove_async`.
    #[allow(clippy::too_many_arguments)]
    pub unsafe fn batched_pcs_prove_async(&mut self, inputs_dev: *const c_void, outputs_dev: *const c_void, evals_dev: &[*const c_void],
                                          transcript_dev: *mut c_void, proof_dev: *mut c_void, sumcheck_dev: *mut c_void,
                                          status_dev: *mut c_int, stream: *mut c_void) {
        check(ml_batched_pcs_prove_async(self.h, inputs_dev, outputs_dev, evals_dev.as_ptr(), transcript_dev, proof_dev, sumcheck_dev,
                                         status_dev, stream));
    }
}
impl Drop for BatchedProvePlan {
    fn drop(&mut self) {
        unsafe { ml_batched_prove_plan_free(self.h) }
    }
}
/// `BatchedFriProof` does not derive `Deserialize`; its blob is the bincode encoding of its parts in field order, and the parts
/// that do derive it (`Vec<HashDigest>`, `MerkleInclusionPath<Vec<ReedSolomonPair<F>>>`, `QueryProof<F>`, `F`) are decoded one by one
unsafe fn bfri_proof_from(h: *const MlBfriProof) -> BatchedFriProof<F> {
    let mut blob = vec![0u8; ml_bfri_proof_serialized_len(h)];
    check(ml_bfri_proof_serialize(h, blob.as_mut_ptr()));
    let cfg = bincode_cfg();
    let mut at = 32;
    let batch_commitment = digest(&blob[..32]);
    macro_rules! take { ($t:ty) => {{ let (v, n): ($t, usize) = bincode::serde::decode_from_slice(&blob[at..], cfg).expect("BatchedFriProof blob"); at += n; v }} }
    let commitments = take!(Vec<HashDigest>);
    let nq = take!(u64) as usize;
    let mut queries = Vec::with_capacity(nq);
    for _ in 0..nq {
        let batch_path = take!(MerkleInclusionPath<Vec<ReedSolomonPair<F>>>);
        let query_proof = take!(QueryProof<F>);
        queries.push(BatchedQueryProof { batch_path, query_proof });
    }
    let last_elem = take!(F);
    let mut last_random = [0u8; 32];
    last_random.copy_from_slice(&blob[at..at + 32]);
    BatchedFriProof { batch_commitment, commitments, queries, last_elem, last_random }
}
/// body of `BatchedFriProof::prove` (src/fri/batched_fri.rs:286-318)
pub fn batched_fri_prove(codes: &[Vec<F>], gen_pows: &[F], transcript: &mut Transcript) -> BatchedFriProof<F> {
    let ptrs: Vec<*const u8> = codes.iter().map(|c| p(c)).collect();
    let mut h = std::ptr::null_mut();
    check(unsafe { ml_batched_fri_prove(ptrs.as_ptr(), codes.len(), codes[0].len(), p(gen_pows), gen_pows.len(), transcript.h, &mut h) });
    let proof = unsafe { bfri_proof_from(h) };
    unsafe { ml_bfri_proof_free(h) };
    proof
}
/// `BatchedFriProof::prove` of B codes over all GPUs of the box from one process, every code split by block (ml_bfri_shard_*,
/// csrc/bfri_shard.cu), from the codes of 2^(log_n+1) elements or from the polynomials' 2^log_n coefficients (`reed_solomon` of each
/// + prove): rank g holds block g of G of every polynomial; round 0 and the next log2(G)-1 fold rounds run sharded, rank 0 runs the
/// rest.  The handle is built once per shape (n_codes, log_n) and reused; the proof bytes equal `batched_fri_prove`'s.
pub struct ShardedBatchedFriProver {
    h: *mut MlBfriShard,
}
impl ShardedBatchedFriProver {
    pub fn new(n_codes: usize, log_n: usize) -> Self {
        let mut count = 0;
        check(unsafe { ml_device_count(&mut count) });
        let mut world = 1usize << (usize::BITS - 1 - (count.max(1) as usize).leading_zeros()); // largest power of two <= GPUs
        while world > 1 && log_n < 2 * world.trailing_zeros() as usize {
            world >>= 1; // log_n >= 2 log2(world)
        }
        let world = world.min(16) as c_int;
        let ids: Vec<c_int> = (0..world).collect();
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_bfri_shard_create(world, world, ids.as_ptr(), ids.as_ptr(), n_codes, log_n, &mut h) });
        Self { h }
    }
    /// body of `BatchedFriProof::prove` (src/fri/batched_fri.rs:286-318) for codes of the handle's shape
    pub fn prove(&mut self, codes: &[Vec<F>], gen_pows: &[F], transcript: &mut Transcript) -> BatchedFriProof<F> {
        let ptrs: Vec<*const u8> = codes.iter().map(|c| p(c)).collect();
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_bfri_shard_prove(self.h, ptrs.as_ptr(), codes.len(), codes[0].len(), p(gen_pows), gen_pows.len(), transcript.h, &mut h) });
        let proof = unsafe { bfri_proof_from(h) };
        unsafe { ml_bfri_proof_free(h) };
        proof
    }
    /// `reed_solomon` (src/fri/mod.rs:19-28) of every polynomial + `BatchedFriProof::prove`
    pub fn rs_prove(&mut self, coeffs: &[Vec<F>], transcript: &mut Transcript) -> BatchedFriProof<F> {
        let ptrs: Vec<*const u8> = coeffs.iter().map(|c| p(c)).collect();
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_bfri_shard_rs_prove(self.h, ptrs.as_ptr(), coeffs.len(), coeffs[0].len(), transcript.h, &mut h) });
        let proof = unsafe { bfri_proof_from(h) };
        unsafe { ml_bfri_proof_free(h) };
        proof
    }
}
impl Drop for ShardedBatchedFriProver {
    fn drop(&mut self) {
        unsafe { ml_bfri_shard_free(self.h) }
    }
}
/// `BatchedFriProverData<F>` (src/fri/batched_fri.rs:9-14) with the batch layer and every tree resident in HBM:
/// init :41-99, batched_fold_step :101-181, fold :183-205, open_query_at :207-225; `fri_data()` borrows the inner FriProverData
pub struct CudaBatchedFriProverData {
    h: *mut MlBfri,
}
impl CudaBatchedFriProverData {
    pub fn init(codes: &[Vec<F>], transcript: &mut Transcript) -> Self {
        let ptrs: Vec<*const u8> = codes.iter().map(|c| p(c)).collect();
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_bfri_init(ptrs.as_ptr(), codes.len(), codes[0].len(), transcript.h, &mut h) });
        Self { h }
    }
    pub fn batched_fold_step(&mut self, gen_pows: &[F], r: F, transcript: &mut Transcript) {
        check(unsafe { ml_bfri_batched_fold_step(self.h, p(gen_pows), gen_pows.len(), r.as_ref().as_ptr(), transcript.h) });
    }
    /// the remaining steps (`prover_data.fri_data.fold_step(gen_pows, k, r, transcript)`, :198-201)
    pub fn fold_step(&mut self, gen_pows: &[F], k: usize, r: F, transcript: &mut Transcript) {
        check(unsafe { ml_fri_fold_step(ml_bfri_fri_data(self.h), p(gen_pows), gen_pows.len(), k, r.as_ref().as_ptr(), transcript.h) });
    }
    pub fn fold(gen_pows: &[F], codes: &[Vec<F>], transcript: &mut Transcript) -> Self {
        let ptrs: Vec<*const u8> = codes.iter().map(|c| p(c)).collect();
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_bfri_fold(p(gen_pows), gen_pows.len(), ptrs.as_ptr(), codes.len(), codes[0].len(), transcript.h, &mut h) });
        Self { h }
    }
    pub fn fingerprint_r(&self) -> F {
        let mut out = zeros(1);
        check(unsafe { ml_bfri_fingerprint_r(self.h, pm(&mut out)) });
        out[0]
    }
    pub fn batch_root(&self) -> HashDigest {
        let mut raw = [0u8; 32];
        check(unsafe { ml_merkle_root(ml_bfri_batch_layer(self.h), raw.as_mut_ptr()) });
        digest(&raw)
    }
    pub fn fold_roots(&self) -> Vec<HashDigest> {
        let f = unsafe { ml_bfri_fri_data(self.h) };
        let n = unsafe { ml_fri_num_trees(f) };
        let mut raw = vec![0u8; 32 * n];
        check(unsafe { ml_fri_fold_roots(f, raw.as_mut_ptr()) });
        raw.chunks_exact(32).map(digest).collect()
    }
    pub fn open_query_at(&self, index: usize) -> BatchedQueryProof<F> {
        let f = unsafe { ml_bfri_fri_data(self.h) };
        let (trees, b) = (unsafe { ml_fri_num_trees(f) }, unsafe { ml_bfri_num_codes(self.h) });
        let (mut bvals, mut bdigs, mut bdirs, mut blen) = (vec![0u8; 32 * b], vec![0u8; 32 * 64], vec![0u8; 64], 0usize);
        let (mut values, mut lens) = (vec![0u8; 32 * trees], vec![0usize; trees]);
        let (mut digests, mut dirs) = (vec![0u8; 32 * 64 * trees], vec![0u8; 64 * trees]);
        check(unsafe {
            ml_bfri_open_query_at(self.h, index, bvals.as_mut_ptr(), bdigs.as_mut_ptr(), bdirs.as_mut_ptr(), &mut blen, values.as_mut_ptr(),
                                  digests.as_mut_ptr(), dirs.as_mut_ptr(), lens.as_mut_ptr())
        });
        let pair = |v: &[u8]| ReedSolomonPair { value: fe(&v[..16]), minus_value: fe(&v[16..]) };
        let batch_path = MerkleInclusionPath { value: bvals.chunks_exact(32).map(pair).collect(), path: path_from(&bdigs[..32 * blen], &bdirs[..blen]) };
        let (mut paths, mut off) = (Vec::with_capacity(trees), 0);
        for j in 0..trees {
            paths.push(MerkleInclusionPath { value: pair(&values[32 * j..32 * j + 32]), path: path_from(&digests[32 * off..32 * (off + lens[j])], &dirs[off..off + lens[j]]) });
            off += lens[j];
        }
        BatchedQueryProof { batch_path, query_proof: QueryProof { paths } }
    }
}
impl Drop for CudaBatchedFriProverData {
    fn drop(&mut self) {
        unsafe { ml_bfri_free(self.h) }
    }
}
unsafe fn bpcs_proof_from(h: *mut MlBpcsProof, claim: BatchedPCSClaim<F>) -> BatchedPCSProof<F> {
    let fri_proof = bfri_proof_from(ml_bpcs_proof_fri(h));
    let mut flat = zeros(2 * ml_bpcs_proof_num_rounds(h));
    check(ml_bpcs_proof_sumcheck_coeffs(h, pm(&mut flat)));
    ml_bpcs_proof_free(h);
    BatchedPCSProof { fri_proof, sumcheck_polynomials: sumcheck_polys(&flat), claim }
}
/// body of `BatchedPCSProof::prove` (src/fri/batched_pcs.rs:130-180) on one GPU
pub fn batched_pcs_prove(claim: BatchedPCSClaim<F>, poly: &[MultilinearPolynomialEvals<F>], transcript: &mut Transcript) -> BatchedPCSProof<F> {
    let ptrs: Vec<*const u8> = poly.iter().map(|m| p(&m.evals)).collect();
    let mut h = std::ptr::null_mut();
    check(unsafe {
        ml_batched_pcs_prove(p(&claim.inputs), claim.inputs.len(), p(&claim.outputs), poly.len(), ptrs.as_ptr(), poly[0].evals.len(), transcript.h, &mut h)
    });
    unsafe { bpcs_proof_from(h, claim) }
}

/// `BatchedPCSProof::prove` over all GPUs of the box from ONE process (ml_shard_*, csrc/shard.cu): the polynomials are encoded where
/// they land (j mod G), leaves are hashed by leaf range, the exchange is NVLink stores between the GPUs' arenas.  The handle is
/// built once per shape (n_polys, n_vars) and reused; the proof bytes equal `batched_pcs_prove`'s.  Shapes that ml_shard_* cannot
/// split by polynomial (the chosen world is not a power of two or does not divide n_polys) go to `BlockShardedBatchedProver`.
pub struct ShardedBatchedProver {
    h: *mut MlShard,
    block: Option<BlockShardedBatchedProver>,
}
impl ShardedBatchedProver {
    pub fn new(n_polys: usize, n_vars: usize) -> Self {
        let mut count = 0;
        check(unsafe { ml_device_count(&mut count) });
        let world = 1usize << (usize::BITS - 1 - (count.max(1) as usize).leading_zeros()); // largest power of two <= GPUs
        let world = world.min(n_polys).min(16);
        if !world.is_power_of_two() || n_polys % world != 0 {
            return Self { h: std::ptr::null_mut(), block: Some(BlockShardedBatchedProver::new(n_polys, n_vars)) };
        }
        let world = world as c_int;
        let ids: Vec<c_int> = (0..world).collect();
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_shard_create(world, world, ids.as_ptr(), ids.as_ptr(), n_polys, n_vars, &mut h) });
        Self { h, block: None }
    }
    pub fn prove(&mut self, claim: BatchedPCSClaim<F>, poly: &[MultilinearPolynomialEvals<F>], transcript: &mut Transcript) -> BatchedPCSProof<F> {
        if let Some(b) = self.block.as_mut() {
            return b.prove(claim, poly, transcript);
        }
        let ptrs: Vec<*const u8> = poly.iter().map(|m| p(&m.evals)).collect();
        let mut h = std::ptr::null_mut();
        check(unsafe {
            ml_shard_batched_pcs_prove(self.h, p(&claim.inputs), claim.inputs.len(), p(&claim.outputs), poly.len(), ptrs.as_ptr(), transcript.h, &mut h)
        });
        unsafe { bpcs_proof_from(h, claim) }
    }
}
impl Drop for ShardedBatchedProver {
    fn drop(&mut self) {
        if !self.h.is_null() {
            unsafe { ml_shard_free(self.h) }
        }
    }
}

/// `BatchedPCSProof::prove` over all GPUs of the box from ONE process with every polynomial split by block (ml_bpcs_shard_*,
/// csrc/bpcs_shard.cu): rank g holds evals_j[g*n/G, (g+1)*n/G) of every polynomial, so any n_polys >= 1 runs on every GPU.  The
/// handle is built once per shape (n_polys, n_vars) and reused; the proof bytes equal `batched_pcs_prove`'s.
pub struct BlockShardedBatchedProver {
    h: *mut MlBpcsShard,
}
impl BlockShardedBatchedProver {
    pub fn new(n_polys: usize, n_vars: usize) -> Self {
        let mut count = 0;
        check(unsafe { ml_device_count(&mut count) });
        let mut world = 1usize << (usize::BITS - 1 - (count.max(1) as usize).leading_zeros()); // largest power of two <= GPUs
        while world > 1 && n_vars < 2 * world.trailing_zeros() as usize {
            world >>= 1; // n_vars >= 2 log2(world)
        }
        let world = world.min(16) as c_int;
        let ids: Vec<c_int> = (0..world).collect();
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_bpcs_shard_create(world, world, ids.as_ptr(), ids.as_ptr(), n_polys, n_vars, &mut h) });
        Self { h }
    }
    pub fn prove(&mut self, claim: BatchedPCSClaim<F>, poly: &[MultilinearPolynomialEvals<F>], transcript: &mut Transcript) -> BatchedPCSProof<F> {
        let ptrs: Vec<*const u8> = poly.iter().map(|m| p(&m.evals)).collect();
        let mut h = std::ptr::null_mut();
        check(unsafe {
            ml_bpcs_shard_prove(self.h, p(&claim.inputs), claim.inputs.len(), p(&claim.outputs), poly.len(), ptrs.as_ptr(), poly[0].evals.len(),
                                transcript.h, &mut h)
        });
        unsafe { bpcs_proof_from(h, claim) }
    }
}
impl Drop for BlockShardedBatchedProver {
    fn drop(&mut self) {
        unsafe { ml_bpcs_shard_free(self.h) }
    }
}

// ------------------------------------------------------------------ System sumcheck of width > 1 (sumcheck.rs:21-53, 147-247)
/// the composition closure (`&impl Fn(&[F]) -> F`, sumcheck.rs:176) stated as the polynomial it computes over a row:
/// comp(x) = sum_t coef_t * prod_k x[cols_t[k]]  (INTEGRATION.md §4)
pub struct CudaWideSumcheckTables {
    h: *mut MlWSumcheck,
    width: usize,
}
impl CudaWideSumcheckTables {
    /// `System::build_tables` (:22-38): `matrix` row-major [height][width], `row_point` = the n_vars trace challenges of the delta mask
    pub fn build(row_point: &[F], matrix: &[F], width: usize) -> Self {
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_wsumcheck_build(p(row_point), row_point.len(), p(matrix), width, matrix.len() / width, &mut h) });
        Self { h, width }
    }
    pub fn set_composition(&mut self, terms: &[(F, &[u32])]) {
        let coefs: Vec<F> = terms.iter().map(|t| t.0).collect();
        let lens: Vec<u32> = terms.iter().map(|t| t.1.len() as u32).collect();
        let cols: Vec<u32> = terms.iter().flat_map(|t| t.1.iter().copied()).collect();
        check(unsafe { ml_wsumcheck_set_composition(self.h, terms.len(), p(&coefs), lens.as_ptr(), cols.as_ptr()) });
    }
    pub fn partial_sum(&mut self, r: F) -> F {
        let mut out = zeros(1);
        check(unsafe { ml_wsumcheck_partial_sum(self.h, r.as_ref().as_ptr(), pm(&mut out)) });
        out[0]
    }
    pub fn fold(&mut self, r: F) {
        check(unsafe { ml_wsumcheck_fold(self.h, r.as_ref().as_ptr()) });
    }
    /// `compute_sumcheck_polynomials` (:147-172)
    pub fn compute_sumcheck_polynomials(&mut self, composition_degree: usize, transcript: &mut Transcript, sum: F) -> (Vec<SumcheckPolynomial<F>>, Vec<F>) {
        let rounds = unsafe { ml_wsumcheck_height(self.h) }.trailing_zeros() as usize;
        let td = composition_degree + 1;
        let (mut coeffs, mut randoms) = (zeros(rounds * td), zeros(rounds));
        check(unsafe { ml_wsumcheck_compute_polynomials(self.h, composition_degree, transcript.h, sum.as_ref().as_ptr(), pm(&mut coeffs), pm(&mut randoms)) });
        (coeffs.chunks_exact(td).map(|c| SumcheckPolynomial { nonzero_coeffs: c.into() }).collect(), randoms)
    }
}
impl Drop for CudaWideSumcheckTables {
    fn drop(&mut self) {
        unsafe { ml_wsumcheck_free(self.h) }
    }
}
/// The width-w sumcheck over all GPUs of the box from one process (ml_wsumcheck_shard_*, csrc/wsumcheck_shard.cu): rank g holds the
/// row block matrix[g*h/G, (g+1)*h/G); the result equals `CudaWideSumcheckTables::build` + `set_composition` +
/// `compute_sumcheck_polynomials` exactly.  For traces too large for one GPU.  The handle is built once per (width, n_vars).
pub struct ShardedWideSumcheckTables {
    h: *mut MlWSumcheckShard,
    width: usize,
}
impl ShardedWideSumcheckTables {
    pub fn new(width: usize, n_vars: usize) -> Self {
        let mut count = 0;
        check(unsafe { ml_device_count(&mut count) });
        let mut world = 1usize << (usize::BITS - 1 - (count.max(1) as usize).leading_zeros()); // largest power of two <= GPUs
        while world > 1 && n_vars < world.trailing_zeros() as usize {
            world >>= 1; // n_vars >= log2(world)
        }
        let world = world.min(16) as c_int;
        let ids: Vec<c_int> = (0..world).collect();
        let mut h = std::ptr::null_mut();
        check(unsafe { ml_wsumcheck_shard_create(world, world, ids.as_ptr(), ids.as_ptr(), width, n_vars, &mut h) });
        Self { h, width }
    }
    pub fn set_composition(&mut self, terms: &[(F, &[u32])]) {
        let coefs: Vec<F> = terms.iter().map(|t| t.0).collect();
        let lens: Vec<u32> = terms.iter().map(|t| t.1.len() as u32).collect();
        let cols: Vec<u32> = terms.iter().flat_map(|t| t.1.iter().copied()).collect();
        check(unsafe { ml_wsumcheck_shard_set_composition(self.h, terms.len(), p(&coefs), lens.as_ptr(), cols.as_ptr()) });
    }
    /// `compute_sumcheck_polynomials` (:147-172) of the trace `matrix` (row-major [2^n_vars][width]) at `row_point`
    pub fn compute_sumcheck_polynomials(&mut self, row_point: &[F], matrix: &[F], composition_degree: usize, transcript: &mut Transcript, sum: F)
        -> (Vec<SumcheckPolynomial<F>>, Vec<F>) {
        let rounds = row_point.len();
        let td = composition_degree + 1;
        let (mut coeffs, mut randoms) = (zeros(rounds * td), zeros(rounds));
        check(unsafe {
            ml_wsumcheck_shard_compute_polynomials(self.h, p(row_point), rounds, p(matrix), self.width, matrix.len() / self.width, composition_degree,
                                                   transcript.h, sum.as_ref().as_ptr(), pm(&mut coeffs), pm(&mut randoms))
        });
        (coeffs.chunks_exact(td).map(|c| SumcheckPolynomial { nonzero_coeffs: c.into() }).collect(), randoms)
    }
}
impl Drop for ShardedWideSumcheckTables {
    fn drop(&mut self) {
        unsafe { ml_wsumcheck_shard_free(self.h) }
    }
}
