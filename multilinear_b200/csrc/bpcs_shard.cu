// One BatchedPCSProof::prove (batched_pcs.rs:130-180) with every polynomial split by block over G ranks, one GPU each; the proof is
// byte-identical to ml_batched_pcs_prove's.  Notation and the segment layout are pcs_shard.cu's; rank b holds the block
// evals_j[b*n/G, (b+1)*n/G) of each of the B polynomials.  Only what a batched proof does differently lives here; the encode
// exchange, the combine, rounds 1 .. L-1, the tail and the openings of layers >= 1 are the stages of pcs_shard.h.  The batched
// layer 0 (pipeline, commit, round-0 fold, openings and the BatchedFriProof) is shared with bfri_shard.cu through pcs_shard.h.
//
//   S0  per polynomial j: encode the local block (encode_into) into one of two buffers on the main stream while the side stream
//       stores slice r of code j-1 into rank r's recv slice j-1 (one recv slice per polynomial); flag PX -> all.
//   S1  wait PX; combine recv slice j into layer-0 code j, in the segment layout, for every j; batched subtree of every segment
//       (a leaf hashes the pairs of all B codes at its position; merkle_batched_rs_launch over the segment's code pointers); run
//       roots -> all, flag PB.
//   S2  wait PB; top of the batch tree; absorb the batch root, draw rho and absorb it, prev = fingerprint(rho, outputs).
//       Deterministic, so every rank reaches the same transcript.
//   S3  Horner fingerprint of the B local evaluation blocks (rho from HBM) into one block; cyclic transpose into the owners'
//       sumcheck tables, flag PT; local eq table.
//   Round 0: wait PT; partial sums -> all, flag PR_0; the round polynomial is absorbed WITHOUT a root (the batch root is in the
//       transcript already); fingerprint + first fold of every segment with the GLOBAL leaf index -> layer 1 in the segment layout
//       (rank 0's tail code when L = 1).  Rounds 1 .. L-1 and the tail are pcs_shard's.  Openings of layer 0 gather the B pairs
//       and the path from the owner's arena (upper path from rank 0's copy of the top tree).
//   G = 1 runs the same code without the exchange: the encodes go straight into layer 0 (one segment of N/2 leaves), the
//       fingerprint straight into the tail tables, and round 0 runs inside the tail's fold chain as its batched first fold.
#include <memory>

#include "pcs_shard.h"
#include "transcript.cuh"

using namespace mlb;
using namespace mlbp;
using namespace mlbs;

namespace {

// S2, one thread: batch root -> transcript, rho, running claim (identical on every rank)
__global__ void __launch_bounds__(32) bpcs_shard_root_kernel(const uint8_t* __restrict__ root, DevTranscript* tr, const fe* __restrict__ outputs,
                                                             int n_outputs, fe* rho_out, fe* prev_out) {
    if (threadIdx.x != 0) return;
    DevTranscript t = *tr;
    fe rho;
    const fe acc = dt_batch_root(&t, root, outputs, n_outputs, &rho);
    fe_store(rho_out, rho);
    fe_store(prev_out, acc);
    *tr = t;
}

// round 0: for every pair (j, j+R) of every segment of layer 0, the Horner fingerprints over the B codes (code c at layer0 + c *
// code_stride) of the values and of the minus-values, then the FRI fold (batched_fri.rs:124-150) with the GLOBAL leaf index
// gi = p*NL + rank*R + j in the twiddle w^(-gi).  Output placement as pcs_shard_fold_kernel's.
__global__ void __launch_bounds__(256) bpcs_shard_fold_kernel(const fe* __restrict__ layer0, int B, size_t code_stride, size_t segs, size_t R, size_t NL,
                                                              int rank, int log_N, const fe* __restrict__ rho_dev, const fe* __restrict__ r_dev,
                                                              const fe* __restrict__ lo, const fe* __restrict__ hi, fe* __restrict__ out) {
    const fe rho = fe_load(rho_dev), rh = fe_load(r_dev + 1);
    const size_t total = segs * R, N = (size_t)1 << log_N, stride = (size_t)gridDim.x * blockDim.x;
    for (size_t x = (size_t)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += stride) {
        const size_t p = x / R, j = x - p * R;
        const fe* c = layer0 + p * 2 * R + j;
        fe a = fe_zero(), b = fe_zero();
        for (int i = 0; i < B; i++, c += code_stride) {
            a = fe_add(fe_mul(a, rho), fe_load_nc(c));
            b = fe_add(fe_mul(b, rho), fe_load_nc(c + R));
        }
        const size_t gi = p * NL + (size_t)rank * R + j;
        fe d = fe_sub(a, b);
        if (gi != 0) d = fe_mul(d, root_pow(lo, hi, N - gi));
        fe_store(out + run_pos(segs, p, j, R), fe_add(fe_half(fe_add(a, b)), fe_mul(rh, d)));
    }
}

// layer-0 opening of query q: the B pairs at leaf idx[q] mod n (laid out as bfri_open_queries: code c's pair at 32 c) and the
// path, from the owner's segment subtree and rank 0's copy of the top tree (cnt run roots); record = B * 32 | 32 * depth
__global__ void __launch_bounds__(64) bpcs_shard_open0_kernel(const unsigned long long* __restrict__ idx, PeerPtrs peers, size_t off_layer0, size_t off_dig0,
                                                              const uint8_t* __restrict__ top0, size_t n, size_t NL, size_t R, int B, int world, int cnt,
                                                              size_t stride, uint8_t* __restrict__ out) {
    const int q = blockIdx.x, t = threadIdx.x;
    const size_t i = idx[q] % n;
    const size_t p = i / NL, k2 = i - p * NL, owner = k2 / R, jj = k2 - owner * R;
    const int log_R = ilog2_dev(R), log_cnt = ilog2_dev((size_t)cnt);
    uint8_t* rec = out + (size_t)q * stride;
    const uint8_t* base = peers.base[owner];
    const fe* seg = reinterpret_cast<const fe*>(base + off_layer0) + p * 2 * R;
    for (int v = t; v < 2 * B; v += blockDim.x)
        *reinterpret_cast<uint4*>(rec + 16 * (size_t)v) = *reinterpret_cast<const uint4*>(seg + (size_t)(v >> 1) * NL + jj + ((v & 1) ? R : 0));
    uint8_t* path = rec + 32 * (size_t)B;
    for (int u = t; u < log_R + log_cnt; u += blockDim.x) {
        const uint4* src;
        if (u < log_R) {
            src = reinterpret_cast<const uint4*>(base + off_dig0 + 32 * (p * 2 * R + layer_off(R, u) + ((jj >> u) ^ 1)));
        } else {
            const int w = u - log_R;
            const size_t run = p * world + owner;
            src = reinterpret_cast<const uint4*>(top0 + 32 * (layer_off((size_t)cnt, w) + ((run >> w) ^ 1)));
        }
        uint4* dst = reinterpret_cast<uint4*>(path + 32 * (size_t)u);
        dst[0] = src[0];
        dst[1] = src[1];
    }
}

}  // namespace

namespace mlbs {

int batch_init(BatchCore* sh) {
    const size_t B = sh->B;
    sh->R0 = sh->world == 1 ? sh->n : sh->R;
    sh->segs0 = sh->world == 1 ? 1 : sh->world / 2;
    sh->cnt0 = sh->world == 1 ? 1 : sh->world * sh->world / 2;
    sh->ev.resize(sh->local.size());
    int st = ML_OK;
    for (size_t i = 0; i < sh->local.size() && st == ML_OK; i++) {
        PeerRank& r = sh->local[i];
        cudaSetDevice(r.device);
        BatchCore::Events& e = sh->ev[i];
        for (cudaEvent_t* x : {&e.done[0], &e.done[1], &e.free[0], &e.free[1], &e.join})
            if (cudaEventCreateWithFlags(x, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); st = ML_ERR_CUDA; }
        // code pointers of every layer-0 segment: segment p of code c at layer0 + c * NL + p * 2 R0
        std::vector<const fe*> ptrs((size_t)sh->segs0 * B);
        for (int p = 0; p < sh->segs0; p++)
            for (size_t c = 0; c < B; c++) ptrs[(size_t)p * B + c] = at(r, sh->lay.layer[0]) + c * sh->NL + (size_t)p * 2 * sh->R0;
        if (st == ML_OK && cudaMemcpy(r.arena + sh->lay.segptrs, ptrs.data(), ptrs.size() * sizeof(void*), cudaMemcpyHostToDevice) != cudaSuccess) {
            cudaGetLastError();
            st = ML_ERR_CUDA;
        }
    }
    return st;
}

BatchCore::~BatchCore() {
    DeviceGuard guard;
    for (size_t i = 0; i < ev.size(); i++) {
        cudaSetDevice(local[i].device);
        Events& e = ev[i];
        for (cudaEvent_t x : {e.done[0], e.done[1], e.free[0], e.free[1], e.join})
            if (x) cudaEventDestroy(x);
    }
}

int batch_encode_exchange(BatchCore* sh, size_t li, const std::function<int(size_t j, fe* y, cudaStream_t s)>& encode) {
    PeerRank& r = sh->local[li];
    cudaStream_t s = r.st.main, side = r.st.side;
    const Layout& a = sh->lay;
    const size_t NL = sh->NL;
    BatchCore::Events& e = sh->ev[li];
    for (size_t j = 0; j < sh->B; j++) {
        fe* y = at(r, a.ycode) + (j & 1) * NL;
        MLB_CUDA(cudaStreamWaitEvent(s, e.free[j & 1], 0));  // the exchange of polynomial j-2 has read this buffer
        MLB_TRY(encode(j, y, s));
        MLB_CUDA(cudaEventRecord(e.done[j & 1], s));
        MLB_CUDA(cudaStreamWaitEvent(side, e.done[j & 1], 0));
        MLB_TRY(exchange_launch(sh, r, y, a.recv + j * NL * 16, side));
        MLB_CUDA(cudaEventRecord(e.free[j & 1], side));
    }
    MLB_CUDA(cudaEventRecord(e.join, side));
    MLB_CUDA(cudaStreamWaitEvent(s, e.join, 0));
    return peer_signal(sh->grp, r, PX, -1, s);
}

int batch_commit(BatchCore* sh, PeerRank& r, bool combine, bool mobius) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    const Layout& a = sh->lay;
    const size_t B = sh->B, NL = sh->NL, R0 = sh->R0;
    if (sh->world > 1) {
        const int log_N = (int)sh->n_vars + ML_LOG_BLOWUP;
        const RootTables* rt;
        MLB_TRY(get_root_tables(r.ctx, log_N, s, &rt));  // never a lazy build behind a spinning wait
        MLB_TRY(peer_wait(sh->grp, r, PX, -1, s));
        if (combine)
            for (size_t j = 0; j < B; j++)
                MLB_TRY(combine_launch(sh->L, at(r, a.recv) + j * NL, sh->R, r.rank, log_N, rt, at(r, a.layer[0]) + j * NL, s, mobius));
    }
    const fe* const* ptrs = reinterpret_cast<const fe* const*>(r.arena + a.segptrs);
    for (int p = 0; p < sh->segs0; p++) MLB_TRY(merkle_batched_rs_launch(ptrs + (size_t)p * B, B, 2 * R0, r.arena + a.dig[0] + 32 * (size_t)p * 2 * R0, s));
    return post_launch(sh, r, r.arena + a.dig[0], R0, sh->segs0, -1, a.mail[0], mail_partials(a, 0), PB);
}

const uint8_t* batch_root(const BatchCore* sh, const PeerRank& r) {
    return r.arena + sh->lay.top[0] + 32 * merkle_layer_offset((size_t)sh->cnt0, ilog2((size_t)sh->cnt0));
}

int batch_fold0_launch(BatchCore* sh, PeerRank& r, const fe* r_dev, fe* out, cudaStream_t s) {
    const int log_N = (int)sh->n_vars + ML_LOG_BLOWUP;
    const RootTables* rt;
    MLB_TRY(get_root_tables(r.ctx, log_N, s, &rt));
    const Layout& a = sh->lay;
    bpcs_shard_fold_kernel<<<peer_grid((size_t)sh->segs0 * sh->R0), 256, 0, s>>>(at(r, a.layer[0]), (int)sh->B, sh->NL, (size_t)sh->segs0, sh->R0, sh->NL,
                                                                                r.rank, log_N, at(r, a.rho), r_dev, rt->lo, rt->hi, out);
    MLB_KERNEL_CHECK();
    return ML_OK;
}

int assemble_bfri(BatchCore* sh, PeerRank& r0, const ml_fri* f, ml_transcript* t, ml_bfri_proof* p, const uint8_t* roots_lo) {
    cudaStream_t s = r0.st.main;
    if (f->layers.empty()) { set_error("open_query_at: no folded layer (domain too small)"); return ML_ERR_OUT_OF_RANGE; }  // n_vars = 1
    const int L = sh->L, Ls = L > 1 ? L : 1;  // layers held outside the tail's FriProverData
    const size_t B = sh->B, n = sh->n;
    std::vector<size_t> idx;
    derive_indices(t, 2 * n, idx);
    const size_t nq = idx.size(), stride0 = 32 * B + 32 * 64;
    std::vector<unsigned long long> idx64(idx.begin(), idx.end());
    std::vector<uint8_t> host0(nq * stride0);
    {
        Scratch didx(s), dout(s);
        MLB_TRY(didx.alloc(nq * 8));
        MLB_TRY(dout.alloc(host0.size()));
        MLB_TRY(h2d(didx.p, idx64.data(), nq * 8, s));
        bpcs_shard_open0_kernel<<<(unsigned)nq, 64, 0, s>>>(didx.as<unsigned long long>(), sh->grp.peers(), sh->lay.layer[0], sh->lay.dig[0],
                                                          r0.arena + sh->lay.top[0], n, sh->NL, sh->R0, (int)B, sh->world, sh->cnt0, stride0,
                                                          dout.as<uint8_t>());
        MLB_KERNEL_CHECK();
        MLB_TRY(d2h_sync(host0.data(), dout.p, host0.size(), s));
    }
    std::vector<uint8_t> host;
    int stride = 0;
    MLB_TRY(open_sharded(sh, r0, idx, 1, host, &stride));
    std::vector<size_t> sub(nq);
    for (size_t q = 0; q < nq; q++) sub[q] = idx[q] % (n >> Ls);
    std::vector<QueryH> qs;
    MLB_TRY(fri_open_queries(f, sub, qs, s));
    p->queries.assign(nq, BQueryH());
    const int depth0 = (int)ilog2(n);
    for (size_t q = 0; q < nq; q++) {
        PathH& bp = p->queries[q].batch_path;
        const uint8_t* rec0 = host0.data() + q * stride0;
        bp.value.assign(rec0, rec0 + 32 * B);
        bp.digests.assign(rec0 + 32 * B, rec0 + 32 * B + 32 * (size_t)depth0);
        fill_dirs(bp, idx[q], depth0);
        std::vector<PathH>& paths = p->queries[q].query.paths;
        for (int j = 1; j < L; j++) {
            const uint8_t* rec = host.data() + (q * L + j) * (size_t)stride;
            const int depth = (int)ilog2(n >> j);
            PathH ph;
            ph.value.assign(rec, rec + 32);
            ph.digests.assign(rec + 32, rec + 32 + 32 * (size_t)depth);
            fill_dirs(ph, idx[q] % (n >> j), depth);
            paths.push_back(std::move(ph));
        }
        for (auto& ph : qs[q].paths) paths.push_back(std::move(ph));
    }
    MLB_TRY(d2h_sync(p->batch_commitment, batch_root(sh, r0), 32, s));
    p->commitments.assign(roots_lo + 32, roots_lo + 32 * (size_t)Ls);  // layers 1 .. L-1 (round 0 absorbed no layer root)
    for (const auto& layer : f->layers) p->commitments.insert(p->commitments.end(), layer.tree->root, layer.tree->root + 32);
    p->last_elem = f->last;
    t->sha.digest(p->last_random);
    return ML_OK;
}

}  // namespace mlbs

struct ml_bpcs_shard : BatchCore {};

namespace {

const char* WHO = "ml_bpcs_shard";

// S0 of one rank: transcript and claim, B encodes, each exchanged while the next one runs
int bstage_encode(ml_bpcs_shard* sh, size_t li, const void* const* evals, const uint8_t* tr_state, const uint8_t* outputs) {
    PeerRank& r = sh->local[li];
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    const Layout& a = sh->lay;
    const size_t B = sh->B, NL = sh->NL;
    MLB_TRY(h2d(r.arena + a.tr, tr_state, sizeof(DevTranscript), s));
    MLB_TRY(h2d(r.arena + a.outs, outputs, B * 16, s));
    MLB_TRY(h2d(r.arena + a.eptrs, evals, B * sizeof(void*), s));
    MLB_CUDA(cudaMemsetAsync(sh->grp.status(r), 0, 16, s));
    if (sh->world == 1) {
        for (size_t j = 0; j < B; j++) MLB_TRY(encode_into(r.ctx, (const fe*)evals[j], sh->nloc, at(r, a.layer[0]) + j * NL, s));
        return ML_OK;
    }
    return batch_encode_exchange(sh, li, [&](size_t j, fe* y, cudaStream_t st) { return encode_into(r.ctx, (const fe*)evals[j], sh->nloc, y, st); });
}

// S2 + S3 of one rank: batch root, rho and claim; fingerprinted tables -> owners (flag PT); eq table
int bstage_tables(ml_bpcs_shard* sh, PeerRank& r, const std::vector<hfe>& pts) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    const Layout& a = sh->lay;
    MLB_TRY(top_launch(sh, r, PB, 0, sh->cnt0));
    bpcs_shard_root_kernel<<<1, 32, 0, s>>>(batch_root(sh, r), (DevTranscript*)(r.arena + a.tr), at(r, a.outs), (int)sh->B, at(r, a.rho), at(r, a.prev));
    MLB_KERNEL_CHECK();
    fe* fp = sh->world == 1 ? at(r, a.tail_m) : at(r, a.ycode);  // the encode buffers are free once S0 is done
    MLB_TRY(fingerprint_rows_launch((const fe* const*)(r.arena + a.eptrs), sh->B, sh->nloc, 0, fp, s, at(r, a.rho)));
    if (sh->world == 1) return local_eq_table(r.ctx, pts, (int)sh->n_vars, sh->L, r.rank, at(r, a.tail_d), s);
    MLB_TRY(tables_launch(sh, r, fp, a.m, s));
    MLB_TRY(local_eq_table(r.ctx, pts, (int)sh->n_vars, sh->L, r.rank, at(r, a.d), s));
    return peer_signal(sh->grp, r, PT, -1, s);
}

// round 0, phase A: wait for the tables, partial sums -> all (flag PR_0)
int bstage_post0(ml_bpcs_shard* sh, PeerRank& r, int* nb) {
    MLB_CUDA(cudaSetDevice(r.device));
    const Layout& a = sh->lay;
    MLB_TRY(peer_wait(sh->grp, r, PT, -1, r.st.main));
    MLB_TRY(sumcheck_sums_partials_launch(at(r, a.m), at(r, a.d), sh->nloc, at(r, a.part), nb, r.st.main));
    return post_launch(sh, r, nullptr, sh->R, 0, *nb, a.mail[0], mail_partials(a, 0), PR0);
}
// round 0, phase B: round polynomial and r_0 (no root: the batch root was absorbed in S2)
int bstage_round0(ml_bpcs_shard* sh, PeerRank& r) {
    MLB_CUDA(cudaSetDevice(r.device));
    MLB_TRY(peer_wait(sh->grp, r, PR0, -1, r.st.main));
    return finish_launch(sh, r, 0, nullptr);
}
// round 0, phase C: fingerprint + first fold of the codes, fold of the tables
int bstage_fold0(ml_bpcs_shard* sh, PeerRank& r, int* nb) {
    MLB_CUDA(cudaSetDevice(r.device));
    MLB_TRY(batch_fold0_launch(sh, r, at(r, sh->lay.r), fold_target(sh, r, 0), r.st.main));
    return fold_tables(sh, r, 0, nb);
}

// rank 0: the rest of the fold chain (at G = 1 from the batched first fold), the openings, the final transcript to everybody
int bprove_tail(ml_bpcs_shard* sh, PeerRank& r0, const std::vector<hfe>& pts, const uint8_t* outputs, ml_transcript* t, ml_bpcs_proof** out) {
    ml_fri* f = new ml_fri();
    struct FriGuard { ml_fri* p; ~FriGuard() { free_fri(p); } } fri_guard{f};
    ml_bpcs_proof* p = new ml_bpcs_proof();
    std::unique_ptr<ml_bpcs_proof> guard(p);
    p->sumcheck.resize(2 * sh->n_vars);
    ChainHooks hooks;
    if (sh->L == 0)
        hooks.first_fold = [&](const fe* r_dev, fe** next, bool* owns) {
            *owns = false;  // the tail code buffer of the arena
            *next = at(r0, sh->lay.tail_code);
            return batch_fold0_launch(sh, r0, r_dev, *next, r0.st.main);
        };
    uint8_t roots_lo[MAX_L * 32] = {0};
    MLB_TRY(tail_chain(sh, r0, f, hooks, p->sumcheck.data(), roots_lo, t, 4));
    MLB_TRY(assemble_bfri(sh, r0, f, t, &p->fri, roots_lo));
    if (&r0 == &sh->local[0]) sh->mark_phase(6);
    p->inputs = pts;
    p->outputs.resize(sh->B);
    for (size_t j = 0; j < sh->B; j++) p->outputs[j] = hfe_load(outputs + 16 * j);
    MLB_TRY(tail_release(sh, r0, t));  // also releases the other ranks' buffers for the next call
    *out = guard.release();
    return ML_OK;
}

}  // namespace

extern "C" {

void ml_bpcs_shard_free(ml_bpcs_shard* sh) { delete sh; }

int ml_bpcs_shard_create(int world, int n_local, const int* local_ranks, const int* local_devices, size_t n_polys, size_t n_vars, ml_bpcs_shard** out) {
    MLB_TRY(peer_check_world("ml_bpcs_shard_create", world, n_local));
    const int L = (int)ilog2((size_t)world);
    if (n_polys < 1 || n_polys > ((size_t)1 << 20)) { set_error("ml_bpcs_shard_create: n_polys = %zu, need 1 <= n_polys <= 2^20", n_polys); return ML_ERR_SIZE; }
    if (n_vars < 1 || n_vars < (size_t)(2 * L) || n_vars >= 40) {
        set_error("ml_bpcs_shard_create: n_vars = %zu, need max(1, 2*log2(world)) = %d <= n_vars < 40", n_vars, L ? 2 * L : 1);
        return ML_ERR_SIZE;
    }
    DeviceGuard guard;
    ml_bpcs_shard* sh = new ml_bpcs_shard();
    sh->who = WHO;
    int st = shard_init(sh, world, n_local, local_ranks, local_devices, n_vars, n_polys);
    if (st == ML_OK) st = batch_init(sh);
    if (st != ML_OK) { delete sh; return st; }
    *out = sh;
    return ML_OK;
}

int ml_bpcs_shard_export(ml_bpcs_shard* sh, uint8_t* records_out) { return sh->export_records(records_out); }
int ml_bpcs_shard_connect(ml_bpcs_shard* sh, const uint8_t* records, size_t n_records) { return sh->connect(records, n_records); }
void* ml_bpcs_shard_stream(const ml_bpcs_shard* sh, int local_index) { return sh->stream(local_index); }
size_t ml_bpcs_shard_arena_bytes(const ml_bpcs_shard* sh) { return sh->lay.total; }

// INSTRUMENTATION (include/multilinear_b200_instr.h): device time between the phase marks of the last call on the first local
// rank's main stream, in ms: [S0 encodes + exchange, S1 combine + batch tree, S2/S3 root + tables, sharded rounds, tail chain,
// openings] (the last two on rank 0 only).  Returns the count.
int ml_bpcs_shard_phase_ms(const ml_bpcs_shard* sh, double* out, int cap) { return sh->phase_ms(out, cap); }

// BatchedPCSProof::prove (batched_pcs.rs:130-180).  Every process calls it with the same claim and its own transcript copy; the
// proof comes out on the process that hosts rank 0 (*out = NULL elsewhere); every transcript ends in the same state.
int ml_bpcs_shard_prove_dev(ml_bpcs_shard* sh, const uint8_t* inputs, size_t n_vars, const uint8_t* outputs, size_t n_polys,
                            const void* const* local_evals_dev, ml_transcript* t, ml_bpcs_proof** out) {
    MLB_TRY(sh->check_ready());
    if (n_vars != sh->n_vars || n_polys != sh->B) {
        set_error("ml_bpcs_shard_prove: the claim has %zu polynomials of %zu variables, the handle %zu of %zu", n_polys, n_vars, sh->B, sh->n_vars);
        return ML_ERR_SIZE;
    }
    DeviceGuard guard;
    *out = nullptr;
    sh->grp.epoch++;
    std::vector<hfe> pts(n_vars);
    for (size_t i = 0; i < n_vars; i++) pts[i] = hfe_load(inputs + 16 * i);
    t->sha.update(inputs, n_vars * 16);    // BatchedPCSProverData::init (:44-49); every rank continues from this state
    t->sha.update(outputs, n_polys * 16);
    uint8_t tr_state[sizeof(DevTranscript)];
    memcpy(tr_state, &t->sha, sizeof(DevTranscript));
    const size_t nl = sh->local.size();
    std::vector<int> nb(nl, 0);
    sh->n_marks = 0;
    sh->mark_phase(0);
    for (size_t i = 0; i < nl; i++) MLB_TRY(bstage_encode(sh, i, local_evals_dev + i * n_polys, tr_state, outputs));
    sh->mark_phase(1);
    for (size_t i = 0; i < nl; i++) MLB_TRY(batch_commit(sh, sh->local[i], true, true));
    sh->mark_phase(2);
    for (size_t i = 0; i < nl; i++) MLB_TRY(bstage_tables(sh, sh->local[i], pts));
    sh->mark_phase(3);
    if (sh->L > 0) {
        for (size_t i = 0; i < nl; i++) MLB_TRY(bstage_post0(sh, sh->local[i], &nb[i]));
        for (size_t i = 0; i < nl; i++) MLB_TRY(bstage_round0(sh, sh->local[i]));
        for (size_t i = 0; i < nl; i++) MLB_TRY(bstage_fold0(sh, sh->local[i], &nb[i]));
        for (int k = 1; k < sh->L; k++) {
            for (size_t i = 0; i < nl; i++) MLB_TRY(stage_post(sh, sh->local[i], k, nb[i]));
            for (size_t i = 0; i < nl; i++) MLB_TRY(stage_round(sh, sh->local[i], k));
            for (size_t i = 0; i < nl; i++) MLB_TRY(stage_fold(sh, sh->local[i], k, &nb[i]));
        }
    }
    return end_call(sh, t, out, ml_bpcs_proof_free, [&](PeerRank& r0) { return bprove_tail(sh, r0, pts, outputs, t, out); });
}

// host evaluations (n_polys arrays of n) and a handle that hosts every rank: the drop-in for batched_pcs.rs:130
int ml_bpcs_shard_prove(ml_bpcs_shard* sh, const uint8_t* inputs, size_t n_vars, const uint8_t* outputs, size_t n_polys, const uint8_t* const* evals,
                        size_t n, ml_transcript* t, ml_bpcs_proof** out) {
    if (n_vars != sh->n_vars || n != sh->n || n_polys != sh->B) {
        set_error("ml_bpcs_shard_prove: need 2^n_vars == evals[j].len() == the handle's size and n_polys == the handle's");
        return ML_ERR_SIZE;
    }
    const size_t bytes = sh->nloc * 16;
    return sh->host_call("ml_bpcs_shard_prove", sh->B, bytes, [&](int rank, size_t j) { return evals[j] + (size_t)rank * bytes; },
                         [&](const void* const* dev) { return ml_bpcs_shard_prove_dev(sh, inputs, n_vars, outputs, n_polys, dev, t, out); });
}

}  // extern "C"
