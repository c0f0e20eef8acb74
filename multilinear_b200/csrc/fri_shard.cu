// One FriProof::prove (src/fri/mod.rs:261-285) of one polynomial sharded over G ranks, one GPU each, given by its coefficients
// (reed_solomon + prove, fri/mod.rs:19-28) or by its code; the proof is byte-identical to ml_rs_fri_prove's / ml_fri_prove's.
// Notation and the segment layout are pcs_shard.cu's: L = log2 G, n coefficients, N = 2n, NL = N/G, R = N/G^2, w = w_N.
// Only what a FRI proof does differently lives here; the column exchange, the combine, the segment subtrees, the top hash, the
// fold, the tail and the openings of the sharded layers are the stages of pcs_shard.h.  The placement of a given code and the
// table-free round (fri_round, fri_fold) are shared with bfri_shard.cu through pcs_shard.h.
//
//   Coefficients.  With j = j1 + G*j2 and Y_j1 = reed_solomon(c[j1 + G*j2 : j2 < n/G], w^G) (the RS-encode NTT at length NL),
//       code[k2 + NL*k1] = sum_j1 w_G^(j1*k1) * w^(j1*k2) * Y_j1[k2]:
//   pcs_shard's combine without its Moebius step, once rank b holds residue class j1 = rev_L(b).
//   S0  cyclic transpose of the caller's block: coefficient j -> rank rev_L(j mod G) at j / G (16 n/G bytes out per rank);
//       flag PC -> all; wait PC; RS encode of the n/G received coefficients; slice r of it -> rank r's recv; flag PX -> all.
//   S1  wait PX; twiddle + G-point DFT into layer 0 (G runs of R elements per rank, segment layout).
//   Code.  Rank b's block code[b*NL, (b+1)*NL) is run b of every rank: S0 stores slice [rR, (r+1)R) straight into rank r's
//       layer 0 at run_pos(G, b, j, R) (no receive buffer, no combine); flag PX -> all; S1 is the wait.
//   Rounds k < L: pcs_shard's rounds without tables.  A: segment subtrees, run roots -> all (flag PR_k).  B: top of the layer
//       tree; absorb its root and draw r_k on every rank (the FRI order root_k | r_k, fri/mod.rs:71,133,139-142).  C: fold into
//       layer k+1, or into rank 0's tail code after round L-1 (flag PG -> rank 0).
//   Tail (rank 0): wait PG; fold_chain_dev from k = L without tables, layer L committed but not absorbed; queries over N/2 leaves;
//       layers < L opened by peer loads; the final transcript -> all (flag PF).  A failed tail (a code that is not an RS code
//       ends in a non-constant last fold) hands its status to every rank instead, so every rank returns it at once.
//   G = 1 runs the same code without any exchange: the encode (or a copy of the code) goes straight into the tail.
#include <memory>
#include <string>

#include "pcs_shard.h"

using namespace mlb;
using namespace mlbp;
using namespace mlbs;

namespace {

// S0 of the code entry: slice [dest*R, (dest+1)*R) of this rank's block = run `rank` of rank dest's code at off_layer0
__global__ void __launch_bounds__(256) fri_shard_place_kernel(const fe* __restrict__ code, size_t NL, size_t R, int rank, int world, PeerPtrs peers,
                                                              size_t off_layer0) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < NL; k += stride) {
        const size_t dest = k / R, j = k - dest * R;
        reinterpret_cast<uint4*>(peers.base[dest] + off_layer0)[run_pos((size_t)world, (size_t)rank, j, R)] = __ldg(reinterpret_cast<const uint4*>(code + k));
    }
}

}  // namespace

namespace mlbs {

int fri_begin(ShardCore* sh, PeerRank& r, const uint8_t* tr_state) {
    MLB_CUDA(cudaSetDevice(r.device));
    MLB_TRY(h2d(r.arena + sh->lay.tr, tr_state, sizeof(DevTranscript), r.st.main));
    MLB_CUDA(cudaMemsetAsync(sh->grp.status(r), 0, 16, r.st.main));
    return ML_OK;
}
int place_launch(ShardCore* sh, PeerRank& r, const fe* code, size_t off_code, cudaStream_t s) {
    fri_shard_place_kernel<<<peer_grid(sh->NL), 256, 0, s>>>(code, sh->NL, sh->R, r.rank, sh->world, sh->grp.peers(), off_code);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
int fri_round(ShardCore* sh, PeerRank& r, int k) {
    MLB_CUDA(cudaSetDevice(r.device));
    const Layout& a = sh->lay;
    const int cnt = (sh->world * sh->world) >> (k + 1);
    MLB_TRY(top_launch(sh, r, PR0 + k, k, cnt));
    const uint8_t* root = r.arena + a.top[k] + 32 * merkle_layer_offset((size_t)cnt, ilog2((size_t)cnt));
    return chain_challenge_launch((DevTranscript*)(r.arena + a.tr), root, 32, r.arena + a.roots_out + 32 * k, at(r, a.r), true, r.st.main);
}
int fri_fold(ShardCore* sh, PeerRank& r, int k) {
    MLB_TRY(fold_code(sh, r, k));
    if (k + 1 < sh->L) return ML_OK;
    return peer_signal(sh->grp, r, PG, 0, r.st.main);
}

}  // namespace mlbs

struct ml_fri_shard : ShardCore {};

namespace {

const char* WHO = "ml_fri_shard";

int log_N_of(const ml_fri_shard* sh) { return (int)sh->n_vars + ML_LOG_BLOWUP; }

// G = 1: layer 0 straight into the tail buffer
int fstage_local(ml_fri_shard* sh, PeerRank& r, const fe* src, bool rs, const uint8_t* tr_state) {
    MLB_TRY(fri_begin(sh, r, tr_state));
    fe* code = at(r, sh->lay.tail_code);
    if (rs) return ntt_launch(r.ctx, src, code, log_N_of(sh), false, true, r.st.main);
    MLB_CUDA(cudaMemcpyAsync(code, src, sh->NL * 16, cudaMemcpyDeviceToDevice, r.st.main));
    return ML_OK;
}

// S0, coefficients: the caller's block -> the owners' coefficient buffers (flag PC)
int fstage_transpose(ml_fri_shard* sh, PeerRank& r, const fe* coeffs, const uint8_t* tr_state) {
    MLB_TRY(fri_begin(sh, r, tr_state));
    const RootTables* rt;
    MLB_TRY(get_root_tables(r.ctx, log_N_of(sh), r.st.main, &rt));  // never a lazy build behind a spinning wait
    MLB_TRY(tables_launch(sh, r, coeffs, sh->lay.coef, r.st.main, true));
    return peer_signal(sh->grp, r, PC, -1, r.st.main);
}
// S0, coefficients: wait PC; local RS encode; column exchange (flag PX)
int fstage_encode(ml_fri_shard* sh, PeerRank& r) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    const Layout& a = sh->lay;
    MLB_TRY(peer_wait(sh->grp, r, PC, -1, s));
    MLB_TRY(ntt_launch(r.ctx, at(r, a.coef), at(r, a.ycode), (int)ilog2(sh->NL), false, true, s));
    MLB_TRY(exchange_launch(sh, r, at(r, a.ycode), a.recv, s));
    return peer_signal(sh->grp, r, PX, -1, s);
}
// S0, code: the caller's block -> run `rank` of every rank's layer 0 (flag PX)
int fstage_place(ml_fri_shard* sh, PeerRank& r, const fe* code, const uint8_t* tr_state) {
    MLB_TRY(fri_begin(sh, r, tr_state));
    const RootTables* rt;
    MLB_TRY(get_root_tables(r.ctx, log_N_of(sh), r.st.main, &rt));
    MLB_TRY(place_launch(sh, r, code, sh->lay.layer[0], r.st.main));
    return peer_signal(sh->grp, r, PX, -1, r.st.main);
}
// S1: wait PX; coefficients: combine the received columns into layer 0
int fstage_combine(ml_fri_shard* sh, PeerRank& r, bool rs) {
    MLB_CUDA(cudaSetDevice(r.device));
    const RootTables* rt;
    MLB_TRY(get_root_tables(r.ctx, log_N_of(sh), r.st.main, &rt));
    MLB_TRY(peer_wait(sh->grp, r, PX, -1, r.st.main));
    if (!rs) return ML_OK;
    return combine_launch(sh->L, at(r, sh->lay.recv), sh->R, r.rank, log_N_of(sh), rt, at(r, sh->lay.layer[0]), r.st.main, false);
}
// rank 0: the rest of the fold chain from layer L, the openings, the final transcript to everybody
int fprove_tail(ml_fri_shard* sh, PeerRank& r0, ml_transcript* t, ml_fri_proof** out) {
    ml_fri* f = new ml_fri();
    struct FriGuard { ml_fri* p; ~FriGuard() { free_fri(p); } } fri_guard{f};
    std::unique_ptr<ml_fri_proof> p(new ml_fri_proof());
    uint8_t roots_lo[MAX_L * 32];
    MLB_TRY(tail_chain(sh, r0, f, ChainHooks(), nullptr, roots_lo, t, 3));
    MLB_TRY(assemble_fri(sh, r0, f, t, p.get(), roots_lo));
    if (&r0 == &sh->local[0]) mark_phase(sh, 5);
    MLB_TRY(tail_release(sh, r0, t));  // also releases the other ranks' buffers for the next call
    *out = p.release();
    return ML_OK;
}

// one call on every local rank; blocks[i]: local rank i's block of the coefficients (rs) or of the code
int fri_shard_run(ml_fri_shard* sh, const void* const* blocks, bool rs, ml_transcript* t, ml_fri_proof** out) {
    MLB_TRY(peer_check_ready(sh->grp, WHO));
    DeviceGuard guard;
    *out = nullptr;
    sh->grp.epoch++;
    uint8_t tr_state[sizeof(DevTranscript)];
    memcpy(tr_state, &t->sha, sizeof tr_state);
    const size_t nl = sh->local.size();
    sh->n_marks = 0;
    mark_phase(sh, 0);
    if (sh->L == 0) {
        MLB_TRY(fstage_local(sh, sh->local[0], (const fe*)blocks[0], rs, tr_state));
        mark_phase(sh, 1);
        mark_phase(sh, 2);
    } else {
        if (rs) {
            for (size_t i = 0; i < nl; i++) MLB_TRY(fstage_transpose(sh, sh->local[i], (const fe*)blocks[i], tr_state));
            for (size_t i = 0; i < nl; i++) MLB_TRY(fstage_encode(sh, sh->local[i]));
        } else {
            for (size_t i = 0; i < nl; i++) MLB_TRY(fstage_place(sh, sh->local[i], (const fe*)blocks[i], tr_state));
        }
        mark_phase(sh, 1);
        for (size_t i = 0; i < nl; i++) MLB_TRY(fstage_combine(sh, sh->local[i], rs));
        mark_phase(sh, 2);
        for (int k = 0; k < sh->L; k++) {
            for (size_t i = 0; i < nl; i++) MLB_TRY(stage_post(sh, sh->local[i], k, -1));
            for (size_t i = 0; i < nl; i++) MLB_TRY(fri_round(sh, sh->local[i], k));
            for (size_t i = 0; i < nl; i++) MLB_TRY(fri_fold(sh, sh->local[i], k));
        }
    }
    int st0 = ML_OK;
    std::string msg;
    if (PeerRank* r0 = rank0_of(sh)) {
        st0 = fprove_tail(sh, *r0, t, out);
        if (st0 != ML_OK) {
            msg = ml_last_error();
            tail_fail(sh, *r0, st0);  // the other ranks wait for PF: release them with this status instead of letting them time out
        }
    }
    int st = finish_ranks(sh, t, st0);
    if (st0 != ML_OK) { set_error("%s", msg.c_str()); st = st0; }
    if (st != ML_OK && *out) { ml_fri_proof_free(*out); *out = nullptr; }
    return st;
}

// host blocks of `per` elements each (a handle that hosts every rank)
int fri_shard_host(ml_fri_shard* sh, const uint8_t* src, size_t per, bool rs, ml_transcript* t, ml_fri_proof** out) {
    DeviceGuard guard;
    std::vector<void*> dev(sh->local.size(), nullptr);
    int st = ML_OK;
    for (size_t i = 0; i < sh->local.size() && st == ML_OK; i++) {
        PeerRank& r = sh->local[i];
        if (cudaSetDevice(r.device) != cudaSuccess) { st = ML_ERR_CUDA; break; }
        st = pmalloc(&dev[i], per * 16, r.st.main);
        if (st == ML_OK) st = h2d(dev[i], src + (size_t)r.rank * per * 16, per * 16, r.st.main);
        if (st == ML_OK && cudaStreamSynchronize(r.st.main) != cudaSuccess) st = ML_ERR_CUDA;
    }
    if (st == ML_OK) st = fri_shard_run(sh, dev.data(), rs, t, out);
    for (size_t i = 0; i < sh->local.size(); i++) {
        cudaSetDevice(sh->local[i].device);
        cudaStreamSynchronize(sh->local[i].st.main);
        pfree(dev[i], sh->local[i].st.main);
    }
    return st;
}

int check_hosts_all(const ml_fri_shard* sh, const char* who) {
    if ((int)sh->local.size() != sh->world) { set_error("%s: host-pointer entry needs a handle that hosts every rank", who); return ML_ERR_ARG; }
    return ML_OK;
}

}  // namespace

extern "C" {

int ml_fri_shard_create(int world, int n_local, const int* local_ranks, const int* local_devices, size_t log_n, ml_fri_shard** out) {
    MLB_TRY(peer_check_world("ml_fri_shard_create", world, n_local));
    const int L = (int)ilog2((size_t)world);
    if (log_n < 1 || log_n < (size_t)(2 * L) || log_n >= 40) {
        set_error("ml_fri_shard_create: log_n = %zu, need max(1, 2*log2(world)) = %d <= log_n < 40", log_n, L ? 2 * L : 1);
        return ML_ERR_SIZE;
    }
    DeviceGuard guard;
    ml_fri_shard* sh = new ml_fri_shard();
    sh->who = WHO;
    int st = shard_init(sh, world, n_local, local_ranks, local_devices, log_n, 0, "ml_fri_shard_create", true);
    if (st != ML_OK) { ml_fri_shard_free(sh); return st; }
    *out = sh;
    return ML_OK;
}

void ml_fri_shard_free(ml_fri_shard* sh) {
    if (!sh) return;
    shard_free(sh);
    delete sh;
}

int ml_fri_shard_export(ml_fri_shard* sh, uint8_t* records_out) { return shard_export(sh, records_out); }
int ml_fri_shard_connect(ml_fri_shard* sh, const uint8_t* records, size_t n_records) { return shard_connect(sh, records, n_records, "ml_fri_shard_connect"); }
void* ml_fri_shard_stream(const ml_fri_shard* sh, int local_index) { return shard_stream(sh, local_index); }
size_t ml_fri_shard_arena_bytes(const ml_fri_shard* sh) { return sh->lay.total; }

// INSTRUMENTATION (include/multilinear_b200_instr.h): device time between the phase marks of the last call on the first local
// rank's main stream, in ms: [S0 transpose + encode + exchange (or placement), S1 combine (or the wait), sharded rounds, tail
// chain, openings] (the last two on rank 0 only).  Returns the count.
int ml_fri_shard_phase_ms(const ml_fri_shard* sh, double* out, int cap) { return shard_phase_ms(sh, out, cap); }

// reed_solomon + FriProof::prove (fri/mod.rs:19-28, :261-285).  Every process calls it with its own transcript copy; the proof
// comes out on the process that hosts rank 0 (*out = NULL elsewhere); every transcript ends in the same state.
int ml_fri_shard_rs_prove_dev(ml_fri_shard* sh, const void* const* local_coeffs_dev, ml_transcript* t, ml_fri_proof** out) {
    return fri_shard_run(sh, local_coeffs_dev, true, t, out);
}
// FriProof::prove of a code of N = 2^(log_n + 1) elements
int ml_fri_shard_prove_dev(ml_fri_shard* sh, const void* const* local_code_dev, ml_transcript* t, ml_fri_proof** out) {
    return fri_shard_run(sh, local_code_dev, false, t, out);
}

// host coefficients (all n) and a handle that hosts every rank
int ml_fri_shard_rs_prove(ml_fri_shard* sh, const uint8_t* coeffs, size_t n, ml_transcript* t, ml_fri_proof** out) {
    MLB_TRY(check_hosts_all(sh, "ml_fri_shard_rs_prove"));
    if (n != sh->n) { set_error("ml_fri_shard_rs_prove: %zu coefficients, the handle takes %zu", n, sh->n); return ML_ERR_SIZE; }
    return fri_shard_host(sh, coeffs, sh->nloc, true, t, out);
}
// host code (all n = 2^(log_n + 1) elements) and a handle that hosts every rank: the drop-in for fri/mod.rs:261; gen_pows as
// for ml_fri_prove
int ml_fri_shard_prove(ml_fri_shard* sh, const uint8_t* code, size_t n, const uint8_t* gen_pows, size_t gen_pows_len, ml_transcript* t,
                       ml_fri_proof** out) {
    MLB_TRY(check_hosts_all(sh, "ml_fri_shard_prove"));
    if (n != 2 * sh->n) { set_error("ml_fri_shard_prove: a code of %zu elements, the handle takes %zu", n, 2 * sh->n); return ML_ERR_SIZE; }
    MLB_TRY(check_gen_pows(log_N_of(sh), gen_pows, gen_pows_len));
    return fri_shard_host(sh, code, sh->NL, false, t, out);
}

}  // extern "C"
