// BatchedPCSProof::prove sharded over GPUs (BASELINE config 5; src/fri/batched_pcs.rs:130-180, src/fri/batched_fri.rs:41-225).
//
// The batch re-partitions from "by polynomial" (Moebius + RS-encode NTT per polynomial, batched_pcs.rs:144-149) to "by leaf range"
// (the batched Merkle leaf i hashes the ReedSolomonPairs of ALL codes at i, merkle_tree/mod.rs:110-116).  Every rank owns
//   * the polynomials j with j mod G == rank               (encode)
//   * leaf rows [rank*rows, (rank+1)*rows), rows = n/G     (hash, fingerprint, first fold, openings)
// and one peer-visible ARENA in HBM (peer.h: cudaMalloc, mapped into the other ranks through CUDA IPC or plain peer access):
//   mailbox (flags, subtree roots, challenge, final transcript) | pairs[B][rows][32] | digests of the row subtree |
//   stage[G][n/G] (fingerprint partial sums) | matrix[n] | next[n]   (the last two are used on rank 0)
// All data-path exchange is a kernel STORING into a peer's arena over NVLink, followed by a flag store (release, system scope);
// consumers wait on their own flags with a tiny spin kernel (acquire, system scope, bounded by a timeout).  No NCCL, no host
// barrier, no collective: the phases below are enqueued back to back on each rank's stream.
//
//   S0  encode local polynomials; pack pass stores pair (code[i], code[i+N/2]) of polynomial j into pairs[j][i mod rows] of rank
//       i/rows (two encode streams + a store stream, so the NVLink stores hide behind the next NTT); flag P1 -> all
//   S1  wait P1; hash the rows' batched leaves and the subtree above them (layers retained); root -> roots[rank] of all + flag P2
//   S2  wait P2; every rank hashes the top log2(G) levels, absorbs the batch root, draws the fingerprint challenge rho
//       (batched_fri.rs:80-86) — identical on all ranks; Horner partial sums of the local evaluation tables in rho^G, scaled by
//       rho^(G-1-rank), stored slice-wise into the stage areas of the slice owners; flag P3 -> all
//   S3  wait P3; add the G staged slices, store the result into rank 0's sumcheck matrix (batched_pcs.rs:55-63); flag P4 -> rank 0
//   S4  rank 0: wait P4; sumcheck round 0 (sums, round polynomial, challenge r0); r0 -> all + flag P5
//   S5  wait P5; fingerprint + first fold of the own rows from the pairs buffer (batched_fri.rs:124-150), stored into rank 0's
//       `next`; flag P6 -> rank 0
//   S6  rank 0: wait P6; the remaining single-code chain (fold_chain_dev), query indices, openings gathered from the owners'
//       arenas by peer loads (batch_open, batched_fri.rs:207-225), final transcript -> all + flag P7; other ranks wait P7.
//
// One handle hosts the ranks of ONE process: one rank (one process per GPU, arenas connected through IPC records the caller
// all-gathers with whatever transport it has) or all G of them (a single-process caller such as the Rust crate; devices may
// repeat, which the tests use to run G virtual ranks on one GPU).  Ranks that share a device share its streams and the host
// enqueues phase by phase over the local ranks, so on a shared device every wait is already satisfied when it is enqueued:
// kernels that wait on each other never run as separate launches on one GPU.
#include <algorithm>
#include <cstdlib>
#include <map>

#include "peer.h"
#include "prover_internal.h"
#include "sha256.cuh"

namespace mlb {
static __device__ __noinline__ void shard_compress(uint32_t st[8], uint32_t w[16]) { sha_compress(st, w); }
}  // namespace mlb
#define MLB_DT_COMPRESS(h, w) shard_compress(h, w)
#include "transcript.cuh"

using namespace mlb;
using namespace mlbp;

namespace {

enum Phase { P1 = 0, P2, P3, P4, P5, P6, P7, N_PHASES };
static const int MAXR = PEER_MAXR;

// ---- arena layout (byte offsets; every section 256-byte aligned)
struct Layout {
    size_t flags, roots, r0, final_tr, status, top, fr, prev, tr, tr_in, root_out, outputs, pairs, digests, stage, matrix, next, total;
};
static size_t align_up(size_t x) { return peer_align(x); }
static Layout make_layout(size_t B, size_t n, size_t G) {
    Layout L;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes); return r; };
    L.flags = take((size_t)N_PHASES * MAXR * 8);
    L.roots = take((size_t)MAXR * 32);
    L.r0 = take(32);
    L.final_tr = take(sizeof(DevTranscript));
    L.status = take(16);
    L.top = take((size_t)2 * MAXR * 32);
    L.fr = take(16);
    L.prev = take(16);
    L.tr = take(sizeof(DevTranscript));
    L.tr_in = take(sizeof(DevTranscript));
    L.root_out = take(32);
    L.outputs = take(B * 16);
    const size_t rows = n / G;
    L.pairs = take(B * rows * 32);
    L.digests = take(2 * rows * 32);
    L.stage = take(n * 16);
    L.matrix = take(n * 16);
    L.next = take(n * 16);
    L.total = o;
    return L;
}

// ------------------------------------------------------------------ S0: pack pass with the exchange fused in
// pair i of polynomial `poly` goes to rank dest = i / rows at pairs[poly][i % rows]; four pairs (128 bytes) in flight per thread
__global__ void __launch_bounds__(256) shard_pack_kernel(const fe* __restrict__ code, size_t half, size_t rows, size_t poly, PeerPtrs peers,
                                                         size_t off_pairs) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < half; i += 4 * stride) {
        uint4 x[4], y[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            x[u] = __ldg(reinterpret_cast<const uint4*>(code + i + u * stride));
            y[u] = __ldg(reinterpret_cast<const uint4*>(code + i + u * stride + half));
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const size_t k = i + u * stride, dest = k / rows, r = k - dest * rows;
            uint4* o = reinterpret_cast<uint4*>(peers.base[dest] + off_pairs) + 2 * (poly * rows + r);
            o[0] = x[u];
            o[1] = y[u];
        }
    }
    for (; i < half; i += stride) {
        const size_t dest = i / rows, r = i - dest * rows;
        uint4* o = reinterpret_cast<uint4*>(peers.base[dest] + off_pairs) + 2 * (poly * rows + r);
        o[0] = __ldg(reinterpret_cast<const uint4*>(code + i));
        o[1] = __ldg(reinterpret_cast<const uint4*>(code + i + half));
    }
}

// ------------------------------------------------------------------ S2: top of the batch tree + transcript, one warp
// waits for every rank's subtree root, hashes the top log2(G) levels (all retained in `top`, Merkle layout with G leaves), absorbs
// the batch root, draws rho = fingerprint_r and absorbs it (batched_fri.rs:80-86); prev = fingerprint(rho, outputs)
// (batched_pcs.rs:92-94).  Deterministic, so every rank reaches the same rho without an exchange.
__global__ void __launch_bounds__(32) shard_root_kernel(const unsigned long long* flags_p2, int world, unsigned long long epoch,
                                                        unsigned long long timeout_ns, int* status, const uint8_t* __restrict__ roots,
                                                        uint8_t* __restrict__ top, const DevTranscript* tr_in, DevTranscript* tr_out,
                                                        const fe* __restrict__ outputs, int n_outputs, fe* fr_out, fe* prev_out,
                                                        uint8_t* root_out, int with_transcript) {
    wait_flags(flags_p2, world, -1, epoch, timeout_ns, status);
    __syncwarp();
    const int t = threadIdx.x;
    for (int i = t; i < world * 8; i += 32) reinterpret_cast<uint32_t*>(top)[i] = reinterpret_cast<const uint32_t*>(roots)[i];
    __syncwarp();
    int layer = 0;
    for (int cnt = world; cnt > 1; cnt >>= 1, layer++) {
        uint8_t* cur = top + 32 * (2 * world - ((2 * world) >> layer));
        uint8_t* nxt = top + 32 * (2 * world - ((2 * world) >> (layer + 1)));
        if (t < (cnt >> 1)) {
            uint32_t l[8], r[8], o[8];
            sha_load_digest(cur + 64 * t, l);
            sha_load_digest(cur + 64 * t + 32, r);
            uint32_t w[16];
#pragma unroll
            for (int k = 0; k < 8; k++) { w[k] = l[k]; w[8 + k] = r[k]; }
            sha_iv(o);
            shard_compress(o, w);
            uint32_t pad[16] = {0x80000000u, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 512u};
            shard_compress(o, pad);
            sha_store_digest(nxt + 32 * t, o);
        }
        __syncwarp();
    }
    if (t != 0) return;
    const uint8_t* root = top + 32 * (2 * world - ((2 * world) >> layer));
    for (int i = 0; i < 32; i++) root_out[i] = root[i];
    if (!with_transcript) return;
    DevTranscript tr = *tr_in;
    fe rho;
    const fe acc = dt_batch_root(&tr, root, outputs, n_outputs, &rho);
    fe_store(fr_out, rho);
    fe_store(prev_out, acc);
    *tr_out = tr;
}

// ------------------------------------------------------------------ S2/S3: fingerprinted evaluation table (batched_pcs.rs:55-63)
// matrix[i] = sum_j evals_j[i] * rho^(B-1-j).  Rank g holds j = g + l*G: Horner over l in rho^G, times rho^(G-1-g); position i is
// stored into the stage area of its slice owner i / slice, at stage[g][i % slice].
__global__ void __launch_bounds__(256) shard_fp_partial_kernel(const fe* const* __restrict__ evals, int n_local, size_t n, const fe* __restrict__ fr,
                                                               int rank, int world, PeerPtrs peers, size_t off_stage, size_t slice) {
    __shared__ fe sh[2];
    if (threadIdx.x == 0) {
        const fe rho = fe_load(fr);
        sh[0] = fe_pow_u64(rho, (unsigned long long)world);
        sh[1] = fe_pow_u64(rho, (unsigned long long)(world - 1 - rank));
    }
    __syncthreads();
    const fe rho_g = sh[0], scale = sh[1];
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        fe acc = fe_load_nc(evals[0] + i);
        for (int l = 1; l < n_local; l++) acc = fe_add(fe_mul(acc, rho_g), fe_load_nc(evals[l] + i));
        if (world - 1 - rank) acc = fe_mul(acc, scale);
        const size_t dest = i / slice, r = i - dest * slice;
        fe_store(reinterpret_cast<fe*>(peers.base[dest] + off_stage) + (size_t)rank * slice + r, acc);
    }
}
__global__ void __launch_bounds__(256) shard_fp_reduce_kernel(const fe* __restrict__ stage, int world, size_t slice, fe* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < slice; i += stride) {
        fe acc = fe_load(stage + i);
        for (int g = 1; g < world; g++) acc = fe_add(acc, fe_load(stage + (size_t)g * slice + i));
        fe_store(out + i, acc);
    }
}

// ------------------------------------------------------------------ S5: fingerprint + first fold of the own rows (batched_fri.rs:124-150)
__device__ __forceinline__ fe shard_root_pow(const fe* __restrict__ lo, const fe* __restrict__ hi, size_t e) {
    fe w = fe_load_nc(lo + (e & (((size_t)1 << LO_BITS) - 1)));
    if (e >> LO_BITS) w = fe_mul(w, fe_load_nc(hi + (e >> LO_BITS)));
    return w;
}
__global__ void __launch_bounds__(256) shard_first_fold_kernel(const uint8_t* __restrict__ pairs, int n_codes, size_t rows, size_t row_base,
                                                               const fe* __restrict__ fr, const fe* __restrict__ r_dev, int log_n0,
                                                               const fe* __restrict__ lo, const fe* __restrict__ hi, fe* __restrict__ next_out) {
    const fe rho = fe_load(fr), r_half = fe_load(r_dev + 1);
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t n0 = (size_t)1 << log_n0;
    for (; i < rows; i += stride) {
        fe a = fe_zero(), b = fe_zero();
        for (int j = 0; j < n_codes; j++) {
            const fe* p = reinterpret_cast<const fe*>(pairs + ((size_t)j * rows + i) * 32);
            a = fe_add(fe_mul(a, rho), fe_load_nc(p));
            b = fe_add(fe_mul(b, rho), fe_load_nc(p + 1));
        }
        const size_t gi = row_base + i;
        fe even = fe_half(fe_add(a, b));
        fe d = fe_sub(a, b);
        if (gi != 0) d = fe_mul(d, shard_root_pow(lo, hi, n0 - gi));  // gen_pows[len - i] (:141-145); i = 0 special-cased (:133-139)
        fe_store(next_out + i, fe_add(even, fe_mul(r_half, d)));
    }
}

// ------------------------------------------------------------------ S6: batch_open across ranks (batched_fri.rs:207-225)
// block q: all B pairs at leaf idx[q] from the owner's pairs buffer, the path's lower log2(rows) siblings from the owner's
// subtree digests (peer loads), the upper log2(G) siblings from the local top tree
__global__ void __launch_bounds__(64) shard_gather_kernel(const unsigned long long* __restrict__ indices, PeerPtrs peers, size_t off_pairs,
                                                          size_t off_digests, const uint8_t* __restrict__ top, int world, size_t rows,
                                                          int n_codes, int depth, uint8_t* __restrict__ vals_out, uint8_t* __restrict__ path_out) {
    const size_t q = blockIdx.x;
    const unsigned long long idx = indices[q];
    const size_t owner = idx / rows, local = idx - owner * rows;
    const uint8_t* pairs = peers.base[owner] + off_pairs;
    const uint8_t* digs = peers.base[owner] + off_digests;
    for (int j = threadIdx.x; j < n_codes; j += blockDim.x) {
        const uint4* src = reinterpret_cast<const uint4*>(pairs + ((size_t)j * rows + local) * 32);
        uint4* dst = reinterpret_cast<uint4*>(vals_out + (q * n_codes + j) * 32);
        dst[0] = src[0];
        dst[1] = src[1];
    }
    int sub_depth = 0;
    while (((size_t)1 << sub_depth) < rows) sub_depth++;
    const int l = threadIdx.x;
    if (l < depth) {
        const uint4* src;
        if (l < sub_depth) {
            const size_t sib = (local >> l) ^ 1;
            src = reinterpret_cast<const uint4*>(digs + 32 * ((2 * rows - ((2 * rows) >> l)) + sib));
        } else {
            const int t = l - sub_depth;
            const size_t sib = (owner >> t) ^ 1;
            src = reinterpret_cast<const uint4*>(top + 32 * ((2 * (size_t)world - ((2 * (size_t)world) >> t)) + sib));
        }
        uint4* dst = reinterpret_cast<uint4*>(path_out + (q * depth + l) * 32);
        dst[0] = src[0];
        dst[1] = src[1];
    }
}

// ------------------------------------------------------------------ host side
struct ShardRank : PeerRank {
    fe* code[2] = {nullptr, nullptr};
    cudaEvent_t ev_done[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr}, ev_fork = nullptr, ev_enc2 = nullptr, ev_side = nullptr;
    const fe** evals_ptrs_dev = nullptr;  // n_local_polys device pointers
    uint8_t* pinned = nullptr;            // host staging: transcript state | outputs | evals pointers
};

}  // namespace

struct ml_shard {
    int world = 1;
    size_t B = 0, n_vars = 0, n = 0, rows = 0, slice = 0, polys_per_rank = 0;
    Layout lay;
    std::vector<ShardRank> local;
    PeerGroup grp;  // arenas of all ranks, flags, epoch, timeout (peer.h)
    // device-time marks of the last call on the first local rank's main stream (include/multilinear_b200_instr.h)
    static const int N_MARKS = 10;
    cudaEvent_t mark[N_MARKS] = {nullptr};
    int n_marks = 0;
    unsigned pack_ctas = 32;
};

namespace {

PeerPtrs peers_of(const ml_shard* sh) { return sh->grp.peers(); }
unsigned long long* flags_at(const ml_shard* sh, const ShardRank& r, int phase) { return sh->grp.flags(r, phase); }
int* status_at(const ml_shard* sh, const ShardRank& r) { return sh->grp.status(r); }
int signal(const ml_shard* sh, const ShardRank& r, int phase, int only, cudaStream_t s) { return peer_signal(sh->grp, r, phase, only, s); }
int wait(const ml_shard* sh, const ShardRank& r, int phase, int only_from, cudaStream_t s) { return peer_wait(sh->grp, r, phase, only_from, s); }
int push(const ml_shard* sh, const ShardRank& r, const void* src_dev, int nbytes, size_t dst_off, int phase, int only, cudaStream_t s) {
    return peer_push(sh->grp, r, src_dev, nbytes, dst_off, phase, only, s);
}
unsigned grid_for(size_t n) { return peer_grid(n); }

void free_rank(ShardRank& r) {
    cudaSetDevice(r.device);
    cudaDeviceSynchronize();
    for (int b = 0; b < 2; b++) {
        if (r.code[b]) cudaFree(r.code[b]);
        if (r.ev_done[b]) cudaEventDestroy(r.ev_done[b]);
        if (r.ev_free[b]) cudaEventDestroy(r.ev_free[b]);
    }
    if (r.ev_fork) cudaEventDestroy(r.ev_fork);
    if (r.ev_enc2) cudaEventDestroy(r.ev_enc2);
    if (r.ev_side) cudaEventDestroy(r.ev_side);
    if (r.evals_ptrs_dev) cudaFree((void*)r.evals_ptrs_dev);
    if (r.pinned) cudaFreeHost(r.pinned);
    peer_rank_free(r);
}

// ---- S0: encode + pack of one local rank (enqueue only)
int stage_encode_pack(ml_shard* sh, ShardRank& r, const void* const* evals /* this rank's polynomials */) {
    MLB_CUDA(cudaSetDevice(r.device));
    const size_t n = sh->n, N = 2 * n;
    cudaStream_t main = r.st.main, es[2] = {r.st.main, r.st.enc2}, side = r.st.side;
    MLB_CUDA(cudaEventRecord(r.ev_fork, main));
    MLB_CUDA(cudaStreamWaitEvent(r.st.enc2, r.ev_fork, 0));
    MLB_CUDA(cudaStreamWaitEvent(side, r.ev_fork, 0));
    const PeerPtrs peers = peers_of(sh);
    size_t blocks = (n + 255) / 256;
    if (blocks > sh->pack_ctas) blocks = sh->pack_ctas;
    for (size_t l = 0; l < sh->polys_per_rank; l++) {
        const int b = (int)(l & 1);
        if (l >= 2) MLB_CUDA(cudaStreamWaitEvent(es[b], r.ev_free[b], 0));  // the store pass has finished reading code buffer b
        MLB_TRY(encode_into(r.ctx, (const fe*)evals[l], n, r.code[b], es[b]));
        MLB_CUDA(cudaEventRecord(r.ev_done[b], es[b]));
        MLB_CUDA(cudaStreamWaitEvent(side, r.ev_done[b], 0));
        // the store pass runs on a small grid: it is NVLink-latency bound and must leave the SMs to the next polynomial's NTT
        shard_pack_kernel<<<(unsigned)blocks, 256, 0, side>>>(r.code[b], N / 2, sh->rows, (size_t)r.rank + l * sh->world, peers, sh->lay.pairs);
        MLB_KERNEL_CHECK();
        MLB_CUDA(cudaEventRecord(r.ev_free[b], side));
    }
    MLB_CUDA(cudaEventRecord(r.ev_enc2, r.st.enc2));
    MLB_CUDA(cudaStreamWaitEvent(main, r.ev_enc2, 0));
    MLB_CUDA(cudaEventRecord(r.ev_side, side));
    MLB_CUDA(cudaStreamWaitEvent(main, r.ev_side, 0));
    return signal(sh, r, P1, -1, main);
}
// ---- S1: leaf range subtree, root to everybody
int stage_subtree(ml_shard* sh, ShardRank& r) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    MLB_TRY(wait(sh, r, P1, -1, s));
    uint8_t* dig = r.arena + sh->lay.digests;
    MLB_TRY(merkle_batched_pairs_strided_launch(r.arena + sh->lay.pairs, sh->B, sh->rows, dig, s));
    const uint8_t* root = dig + 32 * merkle_layer_offset(sh->rows, ilog2(sh->rows));
    return push(sh, r, root, 32, sh->lay.roots + 32 * (size_t)r.rank, P2, -1, s);
}
// ---- S2a: batch root (+ transcript, rho, claimed sum)
int stage_root(ml_shard* sh, ShardRank& r, bool with_transcript) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    shard_root_kernel<<<1, 32, 0, s>>>(flags_at(sh, r, P2), sh->world, sh->grp.epoch, sh->grp.timeout_ns, status_at(sh, r), r.arena + sh->lay.roots,
                                       r.arena + sh->lay.top, (const DevTranscript*)(r.arena + sh->lay.tr_in), (DevTranscript*)(r.arena + sh->lay.tr),
                                       (const fe*)(r.arena + sh->lay.outputs), (int)sh->B, (fe*)(r.arena + sh->lay.fr), (fe*)(r.arena + sh->lay.prev),
                                       r.arena + sh->lay.root_out, with_transcript ? 1 : 0);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
// ---- S2b: fingerprint partial sums into the slice owners' stage areas
int stage_fp_partial(ml_shard* sh, ShardRank& r) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    shard_fp_partial_kernel<<<grid_for(sh->n), 256, 0, s>>>(r.evals_ptrs_dev, (int)sh->polys_per_rank, sh->n, (const fe*)(r.arena + sh->lay.fr), r.rank,
                                                            sh->world, peers_of(sh), sh->lay.stage, sh->slice);
    MLB_KERNEL_CHECK();
    return signal(sh, r, P3, -1, s);
}
// ---- S3: reduce the own slice into rank 0's matrix
int stage_fp_reduce(ml_shard* sh, ShardRank& r) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    MLB_TRY(wait(sh, r, P3, -1, s));
    fe* out = reinterpret_cast<fe*>(sh->grp.base[0] + sh->lay.matrix) + (size_t)r.rank * sh->slice;
    shard_fp_reduce_kernel<<<grid_for(sh->slice), 256, 0, s>>>((const fe*)(r.arena + sh->lay.stage), sh->world, sh->slice, out);
    MLB_KERNEL_CHECK();
    return signal(sh, r, P4, 0, s);
}
// ---- S5: first fold of the own rows into rank 0's `next`
int stage_first_fold(ml_shard* sh, ShardRank& r) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    const int log_n0 = (int)sh->n_vars + ML_LOG_BLOWUP;
    const RootTables* rt;
    MLB_TRY(get_root_tables(r.ctx, log_n0, s, &rt));  // exists since the encode; never a lazy build behind a spinning wait
    MLB_TRY(wait(sh, r, P5, 0, s));
    fe* out = reinterpret_cast<fe*>(sh->grp.base[0] + sh->lay.next) + (size_t)r.rank * sh->rows;
    shard_first_fold_kernel<<<grid_for(sh->rows), 256, 0, s>>>(r.arena + sh->lay.pairs, (int)sh->B, sh->rows, (size_t)r.rank * sh->rows,
                                                              (const fe*)(r.arena + sh->lay.fr), (const fe*)(r.arena + sh->lay.r0), log_n0, rt->lo,
                                                              rt->hi, out);
    MLB_KERNEL_CHECK();
    return signal(sh, r, P6, 0, s);
}

// phase boundary on the first local rank's main stream
void mark_phase(ml_shard* sh, int idx) {
    if (idx >= ml_shard::N_MARKS || sh->local.empty()) return;
    ShardRank& r = sh->local[0];
    cudaSetDevice(r.device);
    if (!sh->mark[idx] && cudaEventCreate(&sh->mark[idx]) != cudaSuccess) { cudaGetLastError(); return; }
    cudaEventRecord(sh->mark[idx], r.st.main);
    if (idx + 1 > sh->n_marks) sh->n_marks = idx + 1;
}
ShardRank* rank0_of(ml_shard* sh) {
    for (auto& r : sh->local)
        if (r.rank == 0) return &r;
    return nullptr;
}

int check_ready(ml_shard* sh) { return peer_check_ready(sh->grp, "ml_shard"); }
// upload the per-call small inputs of a rank through its pinned staging block (asynchronous, stream ordered)
int upload_inputs(ml_shard* sh, ShardRank& r, const HostSha256* tr, const uint8_t* outputs, const void* const* evals) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    MLB_CUDA(cudaStreamSynchronize(s));  // the staging block of the previous call is free (calls on one handle are sequential anyway)
    uint8_t* h = r.pinned;
    const size_t o_tr = 0, o_out = 128, o_ptr = 128 + align_up(sh->B * 16);
    if (tr) {
        memcpy(h + o_tr, tr, sizeof(DevTranscript));
        MLB_CUDA(cudaMemcpyAsync(r.arena + sh->lay.tr_in, h + o_tr, sizeof(DevTranscript), cudaMemcpyHostToDevice, s));
    }
    if (outputs) {
        memcpy(h + o_out, outputs, sh->B * 16);
        MLB_CUDA(cudaMemcpyAsync(r.arena + sh->lay.outputs, h + o_out, sh->B * 16, cudaMemcpyHostToDevice, s));
    }
    memcpy(h + o_ptr, evals, sh->polys_per_rank * sizeof(void*));
    MLB_CUDA(cudaMemcpyAsync((void*)r.evals_ptrs_dev, h + o_ptr, sh->polys_per_rank * sizeof(void*), cudaMemcpyHostToDevice, s));
    MLB_CUDA(cudaMemsetAsync(status_at(sh, r), 0, 16, s));
    return ML_OK;
}
int read_status(ml_shard* sh, ShardRank& r) { return peer_read_status(sh->grp, r, "ml_shard"); }

// batch layer openings + the rest of the proof on rank 0 (batched_fri.rs:207-225, 296-308)
int shard_assemble(ml_shard* sh, ShardRank& r0, ml_fri* fri, ml_transcript* t, ml_bfri_proof* p, const uint8_t batch_root[32]) {
    cudaStream_t s = r0.st.main;
    const size_t N = 2 * sh->n, L = sh->n, B = sh->B;
    if (fri->layers.empty()) { set_error("open_query_at: no folded layer (domain too small)"); return ML_ERR_OUT_OF_RANGE; }
    std::vector<size_t> idx;
    derive_indices(t, N, idx);
    const size_t nq = idx.size();
    const int depth = (int)ilog2(L);
    std::vector<unsigned long long> idx64(idx.begin(), idx.end());
    Scratch didx(s), dvals(s), dpaths(s);
    MLB_TRY(didx.alloc(nq * 8));
    MLB_TRY(dvals.alloc(nq * B * 32));
    MLB_TRY(dpaths.alloc(nq * 32 * (size_t)(depth ? depth : 1)));
    MLB_TRY(h2d(didx.p, idx64.data(), nq * 8, s));
    shard_gather_kernel<<<(unsigned)nq, 64, 0, s>>>(didx.as<unsigned long long>(), peers_of(sh), sh->lay.pairs, sh->lay.digests, r0.arena + sh->lay.top,
                                                    sh->world, sh->rows, (int)B, depth, dvals.as<uint8_t>(), dpaths.as<uint8_t>());
    MLB_KERNEL_CHECK();
    std::vector<uint8_t> hv(nq * B * 32), hp(nq * 32 * (size_t)depth);
    MLB_CUDA(cudaMemcpyAsync(hv.data(), dvals.p, hv.size(), cudaMemcpyDeviceToHost, s));
    MLB_TRY(d2h_sync(hp.data(), dpaths.p, hp.size(), s));
    std::vector<size_t> sub(nq);
    for (size_t q = 0; q < nq; q++) sub[q] = idx[q] % (L / 2);  // :217-218
    std::vector<QueryH> qs;
    MLB_TRY(fri_open_queries(fri, sub, qs, s));
    p->queries.resize(nq);
    for (size_t q = 0; q < nq; q++) {
        PathH& bp = p->queries[q].batch_path;
        bp.value.assign(hv.begin() + q * B * 32, hv.begin() + (q + 1) * B * 32);
        bp.digests.assign(hp.begin() + q * 32 * (size_t)depth, hp.begin() + (q + 1) * 32 * (size_t)depth);
        fill_dirs(bp, idx[q], depth);
        p->queries[q].query = std::move(qs[q]);
    }
    memcpy(p->batch_commitment, batch_root, 32);
    p->commitments.resize(32 * fri->layers.size());
    for (size_t j = 0; j < fri->layers.size(); j++) memcpy(&p->commitments[32 * j], fri->layers[j].tree->root, 32);
    p->last_elem = fri->last;
    t->sha.digest(p->last_random);
    return ML_OK;
}

}  // namespace

extern "C" {

int ml_shard_create(int world, int n_local, const int* local_ranks, const int* local_devices, size_t n_polys, size_t n_vars, ml_shard** out) {
    MLB_TRY(peer_check_world("ml_shard_create", world, n_local));
    if (n_vars < 1 || n_vars >= 40) { set_error("ml_shard_create: n_vars out of range"); return ML_ERR_SIZE; }
    const size_t n = (size_t)1 << n_vars;
    if (n_polys == 0 || n_polys % (size_t)world || n % (size_t)world || n / (size_t)world < 2) {
        set_error("ml_shard_create: polynomials and leaves must split evenly over the ranks (>= 2 leaves per rank)");
        return ML_ERR_SIZE;
    }
    DeviceGuard guard;
    ml_shard* sh = new ml_shard();
    sh->world = world; sh->B = n_polys; sh->n_vars = n_vars; sh->n = n;
    sh->rows = n / world; sh->slice = n / world; sh->polys_per_rank = n_polys / world;
    sh->lay = make_layout(n_polys, n, world);
    sh->grp.world = world;
    sh->grp.arena_bytes = sh->lay.total;
    sh->grp.off_flags = sh->lay.flags;
    sh->grp.off_status = sh->lay.status;
    if (const char* e = getenv("MLB_SHARD_TIMEOUT_S")) sh->grp.timeout_ns = (unsigned long long)(atof(e) * 1e9);
    if (const char* e = getenv("MLB_SHARD_PACK_CTAS")) sh->pack_ctas = (unsigned)atoi(e);
    int st = ML_OK;
    for (int i = 0; i < n_local && st == ML_OK; i++) {
        ShardRank r;
        r.rank = local_ranks[i];
        r.device = local_devices[i];
        st = peer_rank_init(sh->grp, r, "ml_shard_create", sh->lay.pairs);
        if (st != ML_OK && st != ML_ERR_ALLOC) break;
        bool ok = st == ML_OK && cudaMalloc((void**)&r.code[0], 2 * n * 16) == cudaSuccess && cudaMalloc((void**)&r.code[1], 2 * n * 16) == cudaSuccess &&
                  cudaMalloc((void**)&r.evals_ptrs_dev, sh->polys_per_rank * sizeof(void*)) == cudaSuccess &&
                  cudaMallocHost((void**)&r.pinned, 128 + align_up(n_polys * 16) + sh->polys_per_rank * sizeof(void*)) == cudaSuccess;
        for (int b = 0; b < 2 && ok; b++)
            ok = cudaEventCreateWithFlags(&r.ev_done[b], cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&r.ev_free[b], cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&r.ev_fork, cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&r.ev_enc2, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&r.ev_side, cudaEventDisableTiming) == cudaSuccess;
        sh->local.push_back(r);
        if (!ok) { cudaGetLastError(); set_error("ml_shard_create: allocation of %zu bytes on device %d failed", sh->lay.total, r.device); st = ML_ERR_ALLOC; }
    }
    if (st == ML_OK && n_local == world) {
        std::vector<PeerRank*> ranks;
        for (auto& r : sh->local) ranks.push_back(&r);
        st = peer_link_local(sh->grp, ranks, "ml_shard_create");
    }
    if (st != ML_OK) { ml_shard_free(sh); return st; }
    *out = sh;
    return ML_OK;
}

// INSTRUMENTATION (include/multilinear_b200_instr.h): device time between the phase marks of the last call on the first local
// rank's main stream, in ms: commit: [S0 encode+pack, S1 subtree, S2 root]; prove: [S0, S1, S2 root+rho, S2 fingerprint partials,
// S3 reduce, S4 wait for the matrix (rank 0), chain incl. S5 first fold (rank 0), openings + proof (rank 0)].  Returns the count.
int ml_shard_phase_ms(const ml_shard* sh, double* out, int cap) {
    int n = 0;
    for (int i = 0; i + 1 < sh->n_marks && n < cap; i++) {
        float ms = 0;
        if (!sh->mark[i] || !sh->mark[i + 1] || cudaEventElapsedTime(&ms, sh->mark[i], sh->mark[i + 1]) != cudaSuccess) { cudaGetLastError(); ms = -1.f; }
        out[n++] = ms;
    }
    return n;
}

void ml_shard_free(ml_shard* sh) {
    if (!sh) return;
    DeviceGuard guard;
    for (int i = 0; i < ml_shard::N_MARKS; i++)
        if (sh->mark[i]) cudaEventDestroy(sh->mark[i]);
    for (auto& r : sh->local) free_rank(r);
    peer_group_release(sh->grp, sh->local.empty() ? guard.prev : sh->local[0].device);
    delete sh;
}

/* one record per local rank: int32 rank | int32 reserved | 64-byte CUDA IPC handle of the arena */
size_t ml_shard_record_bytes(void) { return PEER_RECORD_BYTES; }
int ml_shard_num_local(const ml_shard* sh) { return (int)sh->local.size(); }
int ml_shard_export(ml_shard* sh, uint8_t* records_out) {
    std::vector<PeerRank*> ranks;
    for (auto& r : sh->local) ranks.push_back(&r);
    return peer_export(ranks, records_out);
}
int ml_shard_connect(ml_shard* sh, const uint8_t* records, size_t n_records) {
    if (sh->local.size() != 1) { set_error("ml_shard_connect: only for handles that host one rank"); return ML_ERR_ARG; }
    return peer_connect(sh->grp, sh->local[0], records, n_records, "ml_shard_connect");
}
void* ml_shard_stream(const ml_shard* sh, int local_index) {
    if (local_index < 0 || (size_t)local_index >= sh->local.size()) return nullptr;
    return (void*)sh->local[local_index].st.main;
}
size_t ml_shard_arena_bytes(const ml_shard* sh) { return sh->lay.total; }

// Merkle::batch_commit of the encoded batch (batched_fri.rs:62-77 after batched_pcs.rs:144-149): phases S0-S2a.
// local_evals_dev: for every local rank in handle order, its polynomials in increasing global index (rank, rank+G, ...).
int ml_shard_batch_commit_dev(ml_shard* sh, const void* const* local_evals_dev, uint8_t root_out[32]) {
    MLB_TRY(check_ready(sh));
    DeviceGuard guard;
    sh->grp.epoch++;
    const size_t ppr = sh->polys_per_rank;
    for (size_t i = 0; i < sh->local.size(); i++) MLB_TRY(upload_inputs(sh, sh->local[i], nullptr, nullptr, local_evals_dev + i * ppr));
    sh->n_marks = 0;
    mark_phase(sh, 0);
    for (size_t i = 0; i < sh->local.size(); i++) { MLB_TRY(stage_encode_pack(sh, sh->local[i], local_evals_dev + i * ppr)); if (i == 0) mark_phase(sh, 1); }
    for (size_t i = 0; i < sh->local.size(); i++) { MLB_TRY(stage_subtree(sh, sh->local[i])); if (i == 0) mark_phase(sh, 2); }
    for (size_t i = 0; i < sh->local.size(); i++) { MLB_TRY(stage_root(sh, sh->local[i], false)); if (i == 0) mark_phase(sh, 3); }
    int st = ML_OK;
    for (auto& r : sh->local) {
        MLB_CUDA(cudaSetDevice(r.device));
        int s1 = d2h_sync(root_out, r.arena + sh->lay.root_out, 32, r.st.main);
        if (s1 == ML_OK) s1 = read_status(sh, r);
        if (s1 != ML_OK) st = s1;
    }
    return st;
}

// BatchedPCSProof::prove (batched_pcs.rs:130-180).  Every process calls it with the same claim and its own transcript copy; the
// proof comes out on the process that hosts rank 0 (*out = NULL elsewhere); every transcript ends in the same state.
int ml_shard_batched_pcs_prove_dev(ml_shard* sh, const uint8_t* inputs, size_t n_vars, const uint8_t* outputs, size_t n_polys,
                                   const void* const* local_evals_dev, ml_transcript* t, ml_bpcs_proof** out) {
    MLB_TRY(check_ready(sh));
    if (n_vars != sh->n_vars || n_polys != sh->B) { set_error("ml_shard_batched_pcs_prove: claim does not match the handle's shape"); return ML_ERR_SIZE; }
    DeviceGuard guard;
    *out = nullptr;
    sh->grp.epoch++;
    const size_t ppr = sh->polys_per_rank, n = sh->n, domain = n << ML_LOG_BLOWUP;
    // BatchedPCSProverData::init (:37-77): the claim enters the transcript first
    t->sha.update(inputs, n_vars * 16);    // :44-46
    t->sha.update(outputs, n_polys * 16);  // :47-49
    ShardRank* r0 = rank0_of(sh);
    ml_sumcheck* sc = nullptr;
    std::vector<hfe> pts(n_vars), outs(n_polys);
    for (size_t i = 0; i < n_vars; i++) pts[i] = hfe_load(inputs + 16 * i);
    for (size_t i = 0; i < n_polys; i++) outs[i] = hfe_load(outputs + 16 * i);
    for (size_t i = 0; i < sh->local.size(); i++) MLB_TRY(upload_inputs(sh, sh->local[i], &t->sha, outputs, local_evals_dev + i * ppr));
    if (r0) {  // the eq table does not depend on anything (:66-67): build it while the stream is idle
        MLB_CUDA(cudaSetDevice(r0->device));
        sc = new ml_sumcheck();
        sc->height = n;
        sc->stream = r0->st.main;
        sc->matrix = reinterpret_cast<fe*>(r0->arena + sh->lay.matrix);
        sc->owns_matrix = false;
        int st = pmalloc((void**)&sc->delta, n * 16, r0->st.main);
        if (st == ML_OK) st = eq_table_launch(r0->ctx, pts.data(), n_vars, sc->delta, r0->st.main);
        if (st != ML_OK) { free_sumcheck(sc); return st; }
    }
    struct ScGuard { ml_sumcheck* p; ~ScGuard() { free_sumcheck(p); } } sc_guard{sc};

    sh->n_marks = 0;
    mark_phase(sh, 0);
    for (size_t i = 0; i < sh->local.size(); i++) { MLB_TRY(stage_encode_pack(sh, sh->local[i], local_evals_dev + i * ppr)); if (i == 0) mark_phase(sh, 1); }  // S0
    for (size_t i = 0; i < sh->local.size(); i++) { MLB_TRY(stage_subtree(sh, sh->local[i])); if (i == 0) mark_phase(sh, 2); }                                  // S1
    for (size_t i = 0; i < sh->local.size(); i++) {                                                                                                              // S2
        MLB_TRY(stage_root(sh, sh->local[i], true));
        if (i == 0) mark_phase(sh, 3);
        MLB_TRY(stage_fp_partial(sh, sh->local[i]));
        if (i == 0) mark_phase(sh, 4);
    }
    for (size_t i = 0; i < sh->local.size(); i++) { MLB_TRY(stage_fp_reduce(sh, sh->local[i])); if (i == 0) mark_phase(sh, 5); }                               // S3

    int st = ML_OK;
    if (r0) {
        MLB_CUDA(cudaSetDevice(r0->device));
        cudaStream_t s = r0->st.main;
        MLB_TRY(wait(sh, *r0, P4, -1, s));  // S4: the sumcheck matrix is complete
        if (r0 == &sh->local[0]) mark_phase(sh, 6);
        ml_fri* fri = new ml_fri();
        fri->log_n0 = (int)ilog2(domain);
        fri->stream = s;
        ChainHooks hooks;
        hooks.tr_dev = (const DevTranscript*)(r0->arena + sh->lay.tr);
        hooks.prev_dev = (const fe*)(r0->arena + sh->lay.prev);
        hooks.first_fold = [&](const fe* r_dev, fe** next, bool* owns) -> int {
            MLB_TRY(push(sh, *r0, r_dev, 32, sh->lay.r0, P5, -1, s));                     // r0 -> all
            for (auto& r : sh->local) MLB_TRY(stage_first_fold(sh, r));                     // S5 of every local rank
            MLB_CUDA(cudaSetDevice(r0->device));
            MLB_TRY(wait(sh, *r0, P6, -1, s));                                              // S6: `next` is complete
            *next = reinterpret_cast<fe*>(r0->arena + sh->lay.next);
            *owns = false;
            return ML_OK;
        };
        ml_bpcs_proof* p = new ml_bpcs_proof();
        const size_t num_steps = ilog2(domain) - ML_LOG_BLOWUP;  // :90
        p->sumcheck.resize(2 * num_steps);
        st = fold_chain_dev(r0->ctx, fri, &hooks, sc, 0, p->sumcheck.data(), 0, false, t, s);  // :100-123
        if (r0 == &sh->local[0]) mark_phase(sh, 7);
        uint8_t batch_root[32];
        if (st == ML_OK) st = d2h_sync(batch_root, r0->arena + sh->lay.root_out, 32, s);
        if (st == ML_OK) st = read_status(sh, *r0);
        if (st == ML_OK) st = shard_assemble(sh, *r0, fri, t, &p->fri, batch_root);              // :155-173
        if (r0 == &sh->local[0]) mark_phase(sh, 8);
        free_fri(fri);
        if (st == ML_OK) {  // final transcript to everybody; also releases the other ranks' buffers for the next call
            Scratch trd(s);
            st = trd.alloc(128);
            if (st == ML_OK) st = h2d(trd.p, &t->sha, sizeof(DevTranscript), s);
            if (st == ML_OK) st = push(sh, *r0, trd.p, (int)(sizeof(DevTranscript) + 15) / 16 * 16, sh->lay.final_tr, P7, -1, s);
            if (st == ML_OK) st = stream_wait_blocking(s);
        }
        if (st != ML_OK) { delete p; return st; }
        p->inputs = pts;
        p->outputs = outs;
        *out = p;
    } else {
        for (auto& r : sh->local) MLB_TRY(stage_first_fold(sh, r));  // S5
    }
    // ranks other than 0: wait for the end of the proof (their buffers are read by rank 0's openings until then)
    for (auto& r : sh->local) {
        if (r.rank == 0) continue;
        MLB_CUDA(cudaSetDevice(r.device));
        MLB_TRY(wait(sh, r, P7, 0, r.st.main));
        int s1 = read_status(sh, r);
        if (s1 != ML_OK) { st = s1; continue; }
        if (!r0) {  // another process holds rank 0: adopt its final transcript
            HostSha256 fin;
            MLB_TRY(d2h_sync(&fin, r.arena + sh->lay.final_tr, sizeof(DevTranscript), r.st.main));
            t->sha = fin;
        }
    }
    return st;
}

// host-pointer convenience for a single-process handle: evals[j] are the n_polys evaluation tables on the host
int ml_shard_batched_pcs_prove(ml_shard* sh, const uint8_t* inputs, size_t n_vars, const uint8_t* outputs, size_t n_polys,
                               const uint8_t* const* evals, ml_transcript* t, ml_bpcs_proof** out) {
    if ((int)sh->local.size() != sh->world) { set_error("ml_shard_batched_pcs_prove: host-pointer entry needs a handle that hosts every rank"); return ML_ERR_ARG; }
    if (n_polys != sh->B || n_vars != sh->n_vars) { set_error("ml_shard_batched_pcs_prove: claim does not match the handle's shape"); return ML_ERR_SIZE; }
    DeviceGuard guard;
    const size_t ppr = sh->polys_per_rank;
    std::vector<void*> dev(n_polys, nullptr);
    int st = ML_OK;
    for (size_t i = 0; i < sh->local.size() && st == ML_OK; i++) {
        ShardRank& r = sh->local[i];
        if (cudaSetDevice(r.device) != cudaSuccess) { st = ML_ERR_CUDA; break; }
        for (size_t l = 0; l < ppr && st == ML_OK; l++) {
            void*& d = dev[i * ppr + l];
            st = pmalloc(&d, sh->n * 16, r.st.main);
            if (st == ML_OK) st = h2d(d, evals[(size_t)r.rank + l * sh->world], sh->n * 16, r.st.main);
        }
        if (st == ML_OK && cudaStreamSynchronize(r.st.main) != cudaSuccess) st = ML_ERR_CUDA;
    }
    if (st == ML_OK) st = ml_shard_batched_pcs_prove_dev(sh, inputs, n_vars, outputs, n_polys, dev.data(), t, out);
    for (size_t i = 0; i < sh->local.size(); i++) {
        cudaSetDevice(sh->local[i].device);
        cudaStreamSynchronize(sh->local[i].st.main);
        for (size_t l = 0; l < ppr; l++) pfree(dev[i * ppr + l], sh->local[i].st.main);
    }
    return st;
}

}  // extern "C"
