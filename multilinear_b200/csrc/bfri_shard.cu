// One BatchedFriProof::prove (batched_fri.rs:286-318) of B codes, each split by block over G ranks, one GPU each, given by the
// coefficients of B polynomials (reed_solomon of each + prove) or by their codes; the proof is byte-identical to
// ml_batched_fri_prove's.  Notation and the segment layout are pcs_shard.cu's: L = log2 G, n coefficients per polynomial, N = 2n,
// NL = N/G, R = N/G^2.  Rank b holds block b of every polynomial: coefficients [b*n/G, (b+1)*n/G) or code elements [b*NL, (b+1)*NL).
// A batched FRI proof is ml_bpcs_shard's proof without the claim, the sumcheck tables and the Moebius step, so everything but the
// transcript step is a stage of pcs_shard.h: the batched layer 0 of bpcs_shard.cu and the table-free rounds of fri_shard.cu.
//
//   S0, coefficients: cyclic transpose of each of the B blocks into the owners' coefficient slices (coefficient j -> rank
//       rev_L(j mod G), as in fri_shard.cu); flag PC -> all; wait PC; per polynomial j, RS encode at length NL into one of two
//       buffers on the main stream while the side stream stores slice r of code j-1 into rank r's recv slice j-1; flag PX -> all.
//       The coefficient slices live in layer 0, which the combine writes only after every encode of this rank.
//   S0, codes: per code j, rank b's block is run b of every rank's layer-0 code j (stored there directly); flag PX -> all.
//   S1  wait PX; coefficients: twiddle + G-point DFT of every recv slice into layer-0 code j (the combine without its Moebius
//       step); batched subtree of every segment (a leaf hashes the pairs of all B codes); run roots -> all, flag PB.
//   S2  wait PB; top of the batch tree; one thread absorbs the batch root, draws rho and absorbs it (batched_fri.rs:80-86), then
//       draws r_0 with nothing absorbed in between (:194).  Deterministic, so every rank reaches the same transcript.
//   Round 0: fingerprint + first fold of every segment with the GLOBAL leaf index -> layer 1 in the segment layout (rank 0's tail
//       code when L = 1).  Rounds 1 .. L-1 are fri_shard's: subtrees, top, absorb root_k and draw r_k, fold.  Flag PG -> rank 0.
//   Tail (rank 0): wait PG; fold_chain_dev from k = L without tables; queries over N/2 leaves; layer 0 opened from the owners'
//       arenas (B pairs and the path), layers 1 .. L-1 likewise, layers >= L from the tail; the final transcript -> all (flag PF).
//       A failed tail (a code that is not an RS code) hands its status to every rank instead.
//   G = 1 runs the same code without any exchange: the encodes (or copies) go straight into layer 0 as one segment, S2 only
//   absorbs the root and rho, and round 0 runs inside the tail's fold chain as its batched first fold (as ml_batched_fri_prove).
#include <memory>

#include "pcs_shard.h"
#include "transcript.cuh"

using namespace mlb;
using namespace mlbp;
using namespace mlbs;

namespace {

// S2, one thread: batch root -> transcript, rho (batched_fri.rs:80-86); r_out != nullptr: r_0 (:194), r_out = {r_0, r_0 / 2}
__global__ void __launch_bounds__(32) bfri_shard_root_kernel(const uint8_t* __restrict__ root, DevTranscript* tr, fe* rho_out, fe* r_out) {
    if (threadIdx.x != 0) return;
    DevTranscript t = *tr;
    fe rho;
    dt_batch_root(&t, root, nullptr, 0, &rho);
    fe_store(rho_out, rho);
    if (r_out) {
        const fe r = dt_challenge(&t);
        fe_store(r_out, r);
        fe_store(r_out + 1, fe_half(r));
    }
    *tr = t;
}

}  // namespace

struct ml_bfri_shard : BatchCore {};

namespace {

const char* WHO = "ml_bfri_shard";

int log_N_of(const ml_bfri_shard* sh) { return (int)sh->n_vars + ML_LOG_BLOWUP; }

// G = 1: the B codes straight into layer 0
int bfstage_local(ml_bfri_shard* sh, PeerRank& r, const void* const* blocks, bool rs, const uint8_t* tr_state) {
    MLB_TRY(fri_begin(sh, r, tr_state));
    for (size_t j = 0; j < sh->B; j++) {
        fe* code = at(r, sh->lay.layer[0]) + j * sh->NL;
        if (rs) MLB_TRY(ntt_launch(r.ctx, (const fe*)blocks[j], code, log_N_of(sh), false, true, r.st.main));
        else MLB_CUDA(cudaMemcpyAsync(code, blocks[j], sh->NL * 16, cudaMemcpyDeviceToDevice, r.st.main));
    }
    return ML_OK;
}

// S0, coefficients: the caller's B blocks -> the owners' coefficient slices (flag PC)
int bfstage_transpose(ml_bfri_shard* sh, PeerRank& r, const void* const* coeffs, const uint8_t* tr_state) {
    MLB_TRY(fri_begin(sh, r, tr_state));
    const RootTables* rt;
    MLB_TRY(get_root_tables(r.ctx, log_N_of(sh), r.st.main, &rt));  // never a lazy build behind a spinning wait
    for (size_t j = 0; j < sh->B; j++) MLB_TRY(tables_launch(sh, r, (const fe*)coeffs[j], sh->lay.coef + j * sh->nloc * 16, r.st.main, true));
    return peer_signal(sh->grp, r, PC, -1, r.st.main);
}
// S0, coefficients: wait PC; the B encodes, each exchanged while the next one runs (flag PX)
int bfstage_encode(ml_bfri_shard* sh, size_t li) {
    PeerRank& r = sh->local[li];
    MLB_CUDA(cudaSetDevice(r.device));
    MLB_TRY(peer_wait(sh->grp, r, PC, -1, r.st.main));
    const fe* coef = at(r, sh->lay.coef);
    const int log_NL = (int)ilog2(sh->NL);
    return batch_encode_exchange(sh, li, [&](size_t j, fe* y, cudaStream_t s) { return ntt_launch(r.ctx, coef + j * sh->nloc, y, log_NL, false, true, s); });
}
// S0, codes: the caller's B blocks -> run `rank` of every rank's layer-0 codes (flag PX)
int bfstage_place(ml_bfri_shard* sh, PeerRank& r, const void* const* codes, const uint8_t* tr_state) {
    MLB_TRY(fri_begin(sh, r, tr_state));
    const RootTables* rt;
    MLB_TRY(get_root_tables(r.ctx, log_N_of(sh), r.st.main, &rt));
    for (size_t j = 0; j < sh->B; j++) MLB_TRY(place_launch(sh, r, (const fe*)codes[j], sh->lay.layer[0] + j * sh->NL * 16, r.st.main));
    return peer_signal(sh->grp, r, PX, -1, r.st.main);
}

// S2: top of the batch tree, batch root and rho (G > 1: and r_0) into the arena
int bfstage_root(ml_bfri_shard* sh, PeerRank& r) {
    MLB_CUDA(cudaSetDevice(r.device));
    const Layout& a = sh->lay;
    MLB_TRY(top_launch(sh, r, PB, 0, sh->cnt0));
    bfri_shard_root_kernel<<<1, 32, 0, r.st.main>>>(batch_root(sh, r), (DevTranscript*)(r.arena + a.tr), at(r, a.rho), sh->L ? at(r, a.r) : nullptr);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
// round 0 (G > 1): fingerprint + first fold into layer 1; at L = 1 that is rank 0's tail code (flag PG)
int bfstage_fold0(ml_bfri_shard* sh, PeerRank& r) {
    MLB_CUDA(cudaSetDevice(r.device));
    MLB_TRY(batch_fold0_launch(sh, r, at(r, sh->lay.r), fold_target(sh, r, 0), r.st.main));
    if (sh->L > 1) return ML_OK;
    return peer_signal(sh->grp, r, PG, 0, r.st.main);
}

// rank 0: the rest of the fold chain (at G = 1 from the batched first fold), the openings, the final transcript to everybody
int bfprove_tail(ml_bfri_shard* sh, PeerRank& r0, ml_transcript* t, ml_bfri_proof** out) {
    ml_fri* f = new ml_fri();
    struct FriGuard { ml_fri* p; ~FriGuard() { free_fri(p); } } fri_guard{f};
    std::unique_ptr<ml_bfri_proof> p(new ml_bfri_proof());
    ChainHooks hooks;
    if (sh->L == 0)
        hooks.first_fold = [&](const fe* r_dev, fe** next, bool* owns) {
            *owns = false;  // the tail code buffer of the arena
            *next = at(r0, sh->lay.tail_code);
            return batch_fold0_launch(sh, r0, r_dev, *next, r0.st.main);
        };
    uint8_t roots_lo[MAX_L * 32] = {0};
    MLB_TRY(tail_chain(sh, r0, f, hooks, nullptr, roots_lo, t, 4));
    MLB_TRY(assemble_bfri(sh, r0, f, t, p.get(), roots_lo));
    if (&r0 == &sh->local[0]) sh->mark_phase(6);
    MLB_TRY(tail_release(sh, r0, t));  // also releases the other ranks' buffers for the next call
    *out = p.release();
    return ML_OK;
}

// one call on every local rank; blocks[i * B + j]: local rank i's block of polynomial j, coefficients (rs) or code
int bfri_shard_run(ml_bfri_shard* sh, const void* const* blocks, bool rs, ml_transcript* t, ml_bfri_proof** out) {
    MLB_TRY(sh->check_ready());
    DeviceGuard guard;
    *out = nullptr;
    sh->grp.epoch++;
    uint8_t tr_state[sizeof(DevTranscript)];
    memcpy(tr_state, &t->sha, sizeof tr_state);
    const size_t nl = sh->local.size(), B = sh->B;
    sh->n_marks = 0;
    sh->mark_phase(0);
    if (sh->L == 0) {
        MLB_TRY(bfstage_local(sh, sh->local[0], blocks, rs, tr_state));
    } else if (rs) {
        for (size_t i = 0; i < nl; i++) MLB_TRY(bfstage_transpose(sh, sh->local[i], blocks + i * B, tr_state));
        for (size_t i = 0; i < nl; i++) MLB_TRY(bfstage_encode(sh, i));
    } else {
        for (size_t i = 0; i < nl; i++) MLB_TRY(bfstage_place(sh, sh->local[i], blocks + i * B, tr_state));
    }
    sh->mark_phase(1);
    for (size_t i = 0; i < nl; i++) MLB_TRY(batch_commit(sh, sh->local[i], rs, false));
    sh->mark_phase(2);
    for (size_t i = 0; i < nl; i++) MLB_TRY(bfstage_root(sh, sh->local[i]));
    sh->mark_phase(3);
    if (sh->L > 0) {
        for (size_t i = 0; i < nl; i++) MLB_TRY(bfstage_fold0(sh, sh->local[i]));
        for (int k = 1; k < sh->L; k++) {
            for (size_t i = 0; i < nl; i++) MLB_TRY(stage_post(sh, sh->local[i], k, -1));
            for (size_t i = 0; i < nl; i++) MLB_TRY(fri_round(sh, sh->local[i], k));
            for (size_t i = 0; i < nl; i++) MLB_TRY(fri_fold(sh, sh->local[i], k));
        }
    }
    return end_call(sh, t, out, ml_bfri_proof_free, [&](PeerRank& r0) { return bfprove_tail(sh, r0, t, out); });
}

// host arrays src[j] (the whole polynomial j: n coefficients (rs) or code elements), cut into the ranks' blocks
int bfri_shard_host(ml_bfri_shard* sh, const char* entry, const uint8_t* const* src, size_t n_codes, size_t n, bool rs, const uint8_t* gen_pows,
                    size_t gen_pows_len, ml_transcript* t, ml_bfri_proof** out) {
    const size_t want_n = rs ? sh->n : 2 * sh->n, bytes = want_n / sh->world * 16;
    if (n_codes != sh->B || n != want_n) {
        set_error("%s: %zu arrays of %zu elements, the handle takes %zu of %zu", entry, n_codes, n, sh->B, want_n);
        return ML_ERR_SIZE;
    }
    if (!rs) MLB_TRY(check_gen_pows(log_N_of(sh), gen_pows, gen_pows_len));
    return sh->host_call(entry, sh->B, bytes, [&](int rank, size_t j) { return src[j] + (size_t)rank * bytes; },
                         [&](const void* const* dev) { return bfri_shard_run(sh, dev, rs, t, out); });
}

}  // namespace

extern "C" {

int ml_bfri_shard_create(int world, int n_local, const int* local_ranks, const int* local_devices, size_t n_codes, size_t log_n, ml_bfri_shard** out) {
    MLB_TRY(peer_check_world("ml_bfri_shard_create", world, n_local));
    const int L = (int)ilog2((size_t)world);
    if (n_codes < 1 || n_codes > ((size_t)1 << 20)) { set_error("ml_bfri_shard_create: n_codes = %zu, need 1 <= n_codes <= 2^20", n_codes); return ML_ERR_SIZE; }
    if (log_n < 1 || log_n < (size_t)(2 * L) || log_n >= 40) {
        set_error("ml_bfri_shard_create: log_n = %zu, need max(1, 2*log2(world)) = %d <= log_n < 40", log_n, L ? 2 * L : 1);
        return ML_ERR_SIZE;
    }
    DeviceGuard guard;
    ml_bfri_shard* sh = new ml_bfri_shard();
    sh->who = WHO;
    int st = shard_init(sh, world, n_local, local_ranks, local_devices, log_n, n_codes, true);
    if (st == ML_OK) st = batch_init(sh);
    if (st != ML_OK) { delete sh; return st; }
    *out = sh;
    return ML_OK;
}

void ml_bfri_shard_free(ml_bfri_shard* sh) { delete sh; }

int ml_bfri_shard_export(ml_bfri_shard* sh, uint8_t* records_out) { return sh->export_records(records_out); }
int ml_bfri_shard_connect(ml_bfri_shard* sh, const uint8_t* records, size_t n_records) { return sh->connect(records, n_records); }
void* ml_bfri_shard_stream(const ml_bfri_shard* sh, int local_index) { return sh->stream(local_index); }
size_t ml_bfri_shard_arena_bytes(const ml_bfri_shard* sh) { return sh->lay.total; }

// INSTRUMENTATION (include/multilinear_b200_instr.h): device time between the phase marks of the last call on the first local
// rank's main stream, in ms: [S0 transpose + encodes + exchange (or placement), S1 combine + batch tree, S2 batch root, sharded
// rounds, tail chain, openings] (the last two on rank 0 only).  Returns the count.
int ml_bfri_shard_phase_ms(const ml_bfri_shard* sh, double* out, int cap) { return sh->phase_ms(out, cap); }

// reed_solomon of every polynomial + BatchedFriProof::prove (batched_fri.rs:286-318).  Every process calls it with its own
// transcript copy; the proof comes out on the process that hosts rank 0 (*out = NULL elsewhere); every transcript ends in the
// same state.
int ml_bfri_shard_rs_prove_dev(ml_bfri_shard* sh, const void* const* local_coeffs_dev, ml_transcript* t, ml_bfri_proof** out) {
    return bfri_shard_run(sh, local_coeffs_dev, true, t, out);
}
// BatchedFriProof::prove of B codes of N = 2^(log_n + 1) elements
int ml_bfri_shard_prove_dev(ml_bfri_shard* sh, const void* const* local_codes_dev, ml_transcript* t, ml_bfri_proof** out) {
    return bfri_shard_run(sh, local_codes_dev, false, t, out);
}

// host coefficients (n_codes arrays of n) and a handle that hosts every rank
int ml_bfri_shard_rs_prove(ml_bfri_shard* sh, const uint8_t* const* coeffs, size_t n_codes, size_t n, ml_transcript* t, ml_bfri_proof** out) {
    return bfri_shard_host(sh, "ml_bfri_shard_rs_prove", coeffs, n_codes, n, true, nullptr, 0, t, out);
}
// host codes (n_codes arrays of n = 2^(log_n + 1)) and a handle that hosts every rank: the drop-in for batched_fri.rs:286;
// gen_pows as for ml_fri_prove
int ml_bfri_shard_prove(ml_bfri_shard* sh, const uint8_t* const* codes, size_t n_codes, size_t n, const uint8_t* gen_pows, size_t gen_pows_len,
                        ml_transcript* t, ml_bfri_proof** out) {
    return bfri_shard_host(sh, "ml_bfri_shard_prove", codes, n_codes, n, false, gen_pows, gen_pows_len, t, out);
}

}  // extern "C"
