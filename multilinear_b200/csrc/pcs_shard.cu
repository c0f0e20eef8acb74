// One PCSProof::prove (src/fri/multilinear_pcs.rs:90-136) sharded over G ranks, one GPU each; the proof is byte-identical to
// ml_pcs_prove's.  Notation: L = log2 G, n = 2^v evaluations, N = 2n code length, R = N / G^2, NL = N / G, w = w_N.
//
//   S0  rank b encodes its block evals[b*n/G, (b+1)*n/G) alone (encode_into: Moebius over the low v-L variables, bit reversal,
//       RS encode of length NL).  The block holds NTT input residue class rev_L(b) mod G.  It stores slice [rR, (r+1)R) of its
//       code into rank r's `recv`, and its evaluations into the owners' sumcheck tables, which are CYCLIC: rank g owns table
//       entries i = m*G + g.  The local eq table is eq(inputs[0 .. v-L)) times prod_{b<L} (bit_b(g) ? p : 1-p), p = inputs[v-1-b].
//       Flag PX -> all.
//   S1  wait PX; combine: rank r owns code columns k2 in [rR, (r+1)R).  For each, y[b] = code_b[k2]; Moebius over the rank bits;
//       X[k2 + NL*k1] = sum_b w_G^(rev(b)*k1) * w^(rev(b)*k2) * y[b] for k1 < G (twiddle, then a G-point DFT in registers).
//       Layer 0 then holds G runs of R elements per rank.
//   Rounds k = 0 .. L-1: layer k has G/2^k runs per rank, stored as G/2^(k+1) SEGMENTS [run p | run p + G/2^(k+1)] of 2R
//       elements: a segment is an RS code whose pairs (j, j+R) are exactly leaves p*NL + rR + j of the global layer, so the
//       global tree has the segments' subtrees as its bottom log2(R) levels (run q = p*G + r).  Every pair (i, i + h/2) of the
//       cyclic sumcheck tables is local while h >= 2G.
//       A   subtree of every segment; the run roots and the rank's two sumcheck partial sums -> every rank; flag PR_k -> all
//       B   wait PR_k; hash the top of the layer-k tree (G^2/2^(k+1) run roots); chain_sumcheck_finish_kernel absorbs the root,
//           the round polynomial, draws r_k and updates the claim: deterministic, identical on every rank
//       C   fold the tables; FRI fold of every segment with the GLOBAL leaf index for the twiddle, written in the segment
//           layout of layer k+1.  After round L-1 layer L is one run per rank: stored into rank 0's `tail_code` at rR, and the
//           tables (height n/G^2) strided into rank 0's `tail_m` / `tail_d` at m*G + g; flag PG -> rank 0
//   Tail (rank 0): wait PG; fold_chain_dev from k = L with layer L committed but not absorbed; openings: layers < L gathered from
//       the owners' arenas by peer loads (upper path from rank 0's copy of the layer's top tree), layers >= L by
//       fri_open_queries; the final transcript -> all + flag PF.  Every process's transcript ends in rank 0's state.
//   G = 1 runs the same code without the exchange: the encode and the tables go straight into the tail buffers.
#include <cstdlib>
#include <memory>

#include "pcs_shard.h"
#include "reduce.cuh"
#include "sha256.cuh"

using namespace mlb;
using namespace mlbp;
using namespace mlbs;

namespace {

// ------------------------------------------------------------------ S0: exchange of the local code, cyclic tables
// code slice [dest*R, (dest+1)*R) -> rank dest's recv[rank*R ..]
__global__ void __launch_bounds__(256) pcs_shard_exchange_kernel(const fe* __restrict__ code, size_t NL, size_t R, int rank, PeerPtrs peers, size_t off_recv) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < NL; k += stride) {
        const size_t dest = k / R, j = k - dest * R;
        reinterpret_cast<uint4*>(peers.base[dest] + off_recv)[(size_t)rank * R + j] = __ldg(reinterpret_cast<const uint4*>(code + k));
    }
}
// block entry o (global b*nloc + o) -> table of rank o mod G (REV: rank rev_L(o mod G)) at (b*nloc + o) / G; stores are
// contiguous per destination
template <bool REV>
__global__ void __launch_bounds__(256) pcs_shard_tables_kernel(const fe* __restrict__ evals, size_t nloc, int L, int rank, PeerPtrs peers, size_t off_m) {
    const size_t per = nloc >> L, stride = (size_t)gridDim.x * blockDim.x;
    for (size_t x = (size_t)blockIdx.x * blockDim.x + threadIdx.x; x < nloc; x += stride) {
        const size_t cls = x / per, ml = x - cls * per;
        const size_t dest = REV ? (__brev((unsigned)cls) >> (32 - L)) : cls;
        reinterpret_cast<uint4*>(peers.base[dest] + off_m)[(size_t)rank * per + ml] = __ldg(reinterpret_cast<const uint4*>(evals + (ml << L) + cls));
    }
}
__global__ void __launch_bounds__(256) pcs_shard_scale_kernel(fe* __restrict__ d, size_t n, fe s) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) fe_store(d + i, fe_mul(fe_load(d + i), s));
}

// ------------------------------------------------------------------ S1: Moebius over the rank bits + twiddle + G-point DFT
// (MOBIUS = false: the local codes encode coefficients, the FRI prover's S1 is twiddle + DFT only)
template <int LG, bool MOBIUS>
__global__ void __launch_bounds__(256) pcs_shard_combine_kernel(const fe* __restrict__ recv, size_t R, int rank, int log_N, const fe* __restrict__ lo,
                                                                const fe* __restrict__ hi, fe* __restrict__ layer0) {
    constexpr int G = 1 << LG;
    __shared__ fe tw[G / 2];  // w_G^t = w^(N t / G)
    if (threadIdx.x < G / 2) tw[threadIdx.x] = root_pow(lo, hi, ((size_t)threadIdx.x << log_N) >> LG);
    __syncthreads();
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < R; j += stride) {
        fe a[G];
#pragma unroll
        for (int b = 0; b < G; b++) a[b] = fe_load_nc(recv + (size_t)b * R + j);
        if (MOBIUS) {
#pragma unroll
            for (int m = 1; m < G; m <<= 1)  // to_coefficient over the rank bits (polynomials.rs:150-163)
#pragma unroll
                for (int b = 0; b < G; b++)
                    if (b & m) a[b] = fe_sub(a[b], a[b ^ m]);
        }
        // a[b] *= w^(rev(b) * k2): input j1 = rev(b) of the DFT, already in the bit-reversed order the butterflies below take
        const size_t k2 = (size_t)rank * R + j;
        const fe wk = root_pow(lo, hi, k2);
        fe p = wk;  // w^(k2 * j1) for j1 = 1, 2, ...
#pragma unroll
        for (int j1 = 1; j1 < G; j1++) {
            int b = 0;
#pragma unroll
            for (int t = 0; t < LG; t++) b |= ((j1 >> t) & 1) << (LG - 1 - t);
            a[b] = fe_mul(a[b], p);
            if (j1 + 1 < G) p = fe_mul(p, wk);
        }
#pragma unroll
        for (int len = 2; len <= G; len <<= 1)
#pragma unroll
            for (int i = 0; i < G; i += len)
#pragma unroll
                for (int t = 0; t < len / 2; t++) {
                    const fe v = t == 0 ? a[i + t + len / 2] : fe_mul(a[i + t + len / 2], tw[t * (G / len)]);
                    const fe u = a[i + t];
                    a[i + t] = fe_add(u, v);
                    a[i + t + len / 2] = fe_sub(u, v);
                }
#pragma unroll
        for (int k1 = 0; k1 < G; k1++) fe_store(layer0 + run_pos(G, k1, j, R), a[k1]);
    }
}

// ------------------------------------------------------------------ rounds
// A: this rank's partial sums (CTA partials -> one pair; none if nb < 0) and run roots -> every rank's mailbox, then the flag there
__global__ void __launch_bounds__(256) pcs_shard_post_kernel(const fe* __restrict__ part, int nb, const uint8_t* __restrict__ dig, size_t R, int segs,
                                                             int rank, int world, PeerPtrs peers, size_t off_roots, size_t off_partials, size_t off_flag,
                                                             unsigned long long epoch) {
    __shared__ fe scratch[32];
    __shared__ fe sums[2];
    fe a1 = fe_zero(), a2 = fe_zero();
    for (int b = threadIdx.x; b < nb; b += blockDim.x) { a1 = fe_add(a1, part[2 * b]); a2 = fe_add(a2, part[2 * b + 1]); }
    const fe e1 = block_sum(a1, scratch);
    const fe e2 = block_sum(a2, scratch);
    if (threadIdx.x == 0) { sums[0] = e1; sums[1] = e2; }
    __syncthreads();
    const int g = threadIdx.x;
    if (g >= world) return;
    uint8_t* dst = peers.base[g];
    const size_t top = layer_off(R, ilog2_dev(R));
    for (int p = 0; p < segs; p++) {
        const uint4* src = reinterpret_cast<const uint4*>(dig + 32 * ((size_t)p * 2 * R + top));
        uint4* d4 = reinterpret_cast<uint4*>(dst + off_roots + 32 * ((size_t)p * world + rank));
        d4[0] = src[0];
        d4[1] = src[1];
    }
    if (nb >= 0) {
        fe_store(reinterpret_cast<fe*>(dst + off_partials) + 2 * rank, sums[0]);
        fe_store(reinterpret_cast<fe*>(dst + off_partials) + 2 * rank + 1, sums[1]);
    }
    __threadfence_system();
    flag_store_release(reinterpret_cast<unsigned long long*>(dst + off_flag) + rank, epoch);
}
// B: one warp waits for every rank's post, then hashes the top of the layer tree (cnt run roots; all levels kept in `top`)
__global__ void __launch_bounds__(32) pcs_shard_top_kernel(const unsigned long long* flags, int world, unsigned long long epoch, unsigned long long timeout_ns,
                                                           int* status, const uint8_t* __restrict__ roots, int cnt, uint8_t* __restrict__ top) {
    wait_flags(flags, world, -1, epoch, timeout_ns, status);
    __syncwarp();
    const int t = threadIdx.x;
    for (int i = t; i < cnt * 8; i += 32) reinterpret_cast<uint32_t*>(top)[i] = reinterpret_cast<const uint32_t*>(roots)[i];
    __syncwarp();
    int layer = 0;
    for (int c = cnt; c > 1; c >>= 1, layer++) {
        const uint8_t* cur = top + 32 * layer_off(cnt, layer);
        uint8_t* nxt = top + 32 * layer_off(cnt, layer + 1);
        for (int i = t; i < (c >> 1); i += 32) {
            uint32_t l[8], r[8], o[8], w[16];
            sha_load_digest(cur + 64 * i, l);
            sha_load_digest(cur + 64 * i + 32, r);
#pragma unroll
            for (int k = 0; k < 8; k++) { w[k] = l[k]; w[8 + k] = r[k]; }
            sha_iv(o);
            sha_compress(o, w);
            sha_compress_pad512(o);
            sha_store_digest(nxt + 32 * i, o);
        }
        __syncwarp();
    }
}
// C: FRI fold (fri/mod.rs:90-114) of every segment of layer k; leaf index gi = p*NL + rank*R + j is global for the twiddle
// w^(-gi * 2^k).  Output run p goes to its place in layer k+1 (`out`, which may be rank 0's tail buffer at rank*R).
__global__ void __launch_bounds__(256) pcs_shard_fold_kernel(const fe* __restrict__ cur, size_t segs, size_t R, size_t NL, int rank, int k, int log_N,
                                                             const fe* __restrict__ r_dev, const fe* __restrict__ lo, const fe* __restrict__ hi,
                                                             fe* __restrict__ out) {
    const fe rh = fe_load(r_dev + 1);
    const size_t total = segs * R, N = (size_t)1 << log_N, stride = (size_t)gridDim.x * blockDim.x;
    for (size_t x = (size_t)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += stride) {
        const size_t p = x / R, j = x - p * R;
        const fe a = fe_load_nc(cur + p * 2 * R + j), b = fe_load_nc(cur + p * 2 * R + j + R);
        const size_t gi = p * NL + (size_t)rank * R + j;
        fe d = fe_sub(a, b);
        if (gi != 0) d = fe_mul(d, root_pow(lo, hi, N - (gi << k)));
        fe_store(out + run_pos(segs, p, j, R), fe_add(fe_half(fe_add(a, b)), fe_mul(rh, d)));
    }
}
// local tables (height h) -> rank 0's tail tables at m*G + rank
__global__ void __launch_bounds__(256) pcs_shard_gather_tables_kernel(const fe* __restrict__ m, const fe* __restrict__ d, size_t h, int rank, int world,
                                                                      fe* __restrict__ tm, fe* __restrict__ td) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < h; i += stride) {
        reinterpret_cast<uint4*>(tm)[i * world + rank] = __ldg(reinterpret_cast<const uint4*>(m + i));
        reinterpret_cast<uint4*>(td)[i * world + rank] = __ldg(reinterpret_cast<const uint4*>(d + i));
    }
}

// ------------------------------------------------------------------ openings of the sharded layers (open_query_at, :154-174)
struct OpenArgs {
    size_t off_layer[MAX_L], off_dig[MAX_L];
    const uint8_t* top[MAX_L];  // rank 0's copies of the top trees
    size_t n, NL, R;
    int L, j0, world, log_R, stride;  // layers j0 .. L-1; stride: bytes per (query, layer) record = 32 value + 32 * 64 path
};
// block (q, j): pair and path of leaf idx[q] mod (n >> j) in layer j, from the owner's arena
__global__ void __launch_bounds__(64) pcs_shard_open_kernel(const unsigned long long* __restrict__ idx, PeerPtrs peers, OpenArgs a, uint8_t* __restrict__ out) {
    const int q = blockIdx.x, j = blockIdx.y + a.j0, t = threadIdx.x;
    const size_t i = idx[q] % (a.n >> j);
    const size_t p = i / a.NL, k2 = i - p * a.NL, owner = k2 / a.R, jj = k2 - owner * a.R;
    const int cnt = (a.world * a.world) >> (j + 1), log_cnt = ilog2_dev((size_t)cnt);
    uint8_t* rec = out + ((size_t)q * a.L + j) * a.stride;
    const uint8_t* base = peers.base[owner];
    if (t < 2) {
        const fe* seg = reinterpret_cast<const fe*>(base + a.off_layer[j]) + p * 2 * a.R;
        *reinterpret_cast<uint4*>(rec + 16 * t) = *reinterpret_cast<const uint4*>(seg + jj + (t ? a.R : 0));
    }
    if (t < a.log_R + log_cnt) {
        const uint4* src;
        if (t < a.log_R) {
            const uint8_t* dig = base + a.off_dig[j] + 32 * (p * 2 * a.R);
            src = reinterpret_cast<const uint4*>(dig + 32 * (layer_off(a.R, t) + ((jj >> t) ^ 1)));
        } else {
            const int u = t - a.log_R;
            const size_t run = p * a.world + owner;
            src = reinterpret_cast<const uint4*>(a.top[j] + 32 * (layer_off((size_t)cnt, u) + ((run >> u) ^ 1)));
        }
        uint4* dst = reinterpret_cast<uint4*>(rec + 32 + 32 * (size_t)t);
        dst[0] = src[0];
        dst[1] = src[1];
    }
}

}  // namespace

struct ml_pcs_shard : ShardCore {};

namespace mlbs {

Layout make_layout(size_t n, int G, size_t B, bool fri) {
    const int L = (int)ilog2((size_t)G);
    const size_t NL = 2 * n / G, R = NL / G, nloc = n / G;
    const bool sharded = G > 1, batched = B > 0;
    Layout a;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o = peer_align(o + bytes); return r; };
    a.flags = take((size_t)N_PHASES * MAXR * 8);
    a.status = take(16);
    a.tr = take(sizeof(DevTranscript));
    a.prev = take(16);
    a.r = take(32);
    a.sc = take((size_t)MAX_L * 32);
    a.roots_out = take((size_t)MAX_L * 32);
    a.final_tr = take(sizeof(DevTranscript));
    for (int k = 0; k < MAX_L; k++) a.mail[k] = take(MAIL_ROOTS * 32 + (size_t)MAXR * 32);  // run roots | partial pairs
    for (int k = 0; k < MAX_L; k++) a.top[k] = take(2 * MAIL_ROOTS * 32);
    a.part = take(fri ? 0 : (size_t)(2 * sumcheck_max_blocks() + 2) * 16);
    a.rho = take(batched ? 16 : 0);
    a.outs = take(fri ? 0 : B * 16);
    a.eptrs = take(fri ? 0 : B * 8);
    a.segptrs = take((sharded ? (size_t)G / 2 : 1) * B * 8);
    // batched: two encode buffers (the encode of polynomial j+1 overlaps the exchange of j) and one recv slice per polynomial
    a.ycode = take(sharded ? (batched ? 2 : 1) * NL * 16 : 0);
    a.recv = take(sharded ? (batched ? B : 1) * NL * 16 : 0);
    a.coef = take(sharded && fri && !batched ? nloc * 16 : 0);
    for (int k = 0; k < MAX_L; k++) {
        const bool held = k < L || (k == 0 && batched);
        a.layer[k] = take(held ? (k == 0 && batched ? B : 1) * ((size_t)G >> k) * R * 16 : 0);
        a.dig[k] = take(held ? ((size_t)G >> k) * R * 32 : 0);
    }
    if (sharded && fri && batched) a.coef = a.layer[0];  // B slices of nloc: read by the encodes, before any combine writes layer 0
    a.m = take(sharded && !fri ? nloc * 16 : 0);
    a.d = take(sharded && !fri ? nloc * 16 : 0);
    a.tail_code = take(NL * 16);
    a.tail_m = take(fri ? 0 : nloc * 16);
    a.tail_d = take(fri ? 0 : nloc * 16);
    a.total = o;
    return a;
}

void mark_phase(ShardCore* sh, int idx) {
    if (idx >= ShardCore::N_MARKS || sh->local.empty()) return;
    PeerRank& r = sh->local[0];
    cudaSetDevice(r.device);
    if (!sh->mark[idx] && cudaEventCreate(&sh->mark[idx]) != cudaSuccess) { cudaGetLastError(); return; }
    cudaEventRecord(sh->mark[idx], r.st.main);
    if (idx + 1 > sh->n_marks) sh->n_marks = idx + 1;
}
PeerRank* rank0_of(ShardCore* sh) {
    for (auto& r : sh->local)
        if (r.rank == 0) return &r;
    return nullptr;
}

int shard_init(ShardCore* sh, int world, int n_local, const int* local_ranks, const int* local_devices, size_t n_vars, size_t B, const char* who,
               bool fri) {
    const int L = (int)ilog2((size_t)world);
    sh->world = world; sh->L = L; sh->n_vars = n_vars; sh->n = (size_t)1 << n_vars; sh->B = B;
    sh->NL = 2 * sh->n / world; sh->R = sh->NL / world; sh->nloc = sh->n / world;
    sh->lay = make_layout(sh->n, world, B, fri);
    sh->grp.world = world;
    sh->grp.arena_bytes = sh->lay.total;
    sh->grp.off_flags = sh->lay.flags;
    sh->grp.off_status = sh->lay.status;
    if (const char* e = getenv("MLB_SHARD_TIMEOUT_S")) sh->grp.timeout_ns = (unsigned long long)(atof(e) * 1e9);
    int st = ML_OK;
    for (int i = 0; i < n_local && st == ML_OK; i++) {
        PeerRank r;
        r.rank = local_ranks[i];
        r.device = local_devices[i];
        st = peer_rank_init(sh->grp, r, who, sh->lay.ycode);
        if (st == ML_OK || st == ML_ERR_ALLOC) sh->local.push_back(r);
    }
    if (st == ML_OK && n_local == world) {
        std::vector<PeerRank*> ranks;
        for (auto& r : sh->local) ranks.push_back(&r);
        st = peer_link_local(sh->grp, ranks, who);
    }
    return st;
}

void shard_free(ShardCore* sh) {
    DeviceGuard guard;
    for (int i = 0; i < ShardCore::N_MARKS; i++)
        if (sh->mark[i]) cudaEventDestroy(sh->mark[i]);
    for (auto& r : sh->local) {
        cudaSetDevice(r.device);
        cudaDeviceSynchronize();
        peer_rank_free(r);
    }
    peer_group_release(sh->grp, sh->local.empty() ? guard.prev : sh->local[0].device);
}

int shard_export(ShardCore* sh, uint8_t* records_out) {
    std::vector<PeerRank*> ranks;
    for (auto& r : sh->local) ranks.push_back(&r);
    return peer_export(ranks, records_out);
}
int shard_connect(ShardCore* sh, const uint8_t* records, size_t n_records, const char* who) {
    if (sh->local.size() != 1) { set_error("%s: only for handles that host one rank", who); return ML_ERR_ARG; }
    return peer_connect(sh->grp, sh->local[0], records, n_records, who);
}
void* shard_stream(const ShardCore* sh, int local_index) {
    if (local_index < 0 || (size_t)local_index >= sh->local.size()) return nullptr;
    return (void*)sh->local[local_index].st.main;
}
int shard_phase_ms(const ShardCore* sh, double* out, int cap) {
    int n = 0;
    for (int i = 0; i + 1 < sh->n_marks && n < cap; i++) {
        float ms = 0;
        if (!sh->mark[i] || !sh->mark[i + 1] || cudaEventElapsedTime(&ms, sh->mark[i], sh->mark[i + 1]) != cudaSuccess) { cudaGetLastError(); ms = -1.f; }
        out[n++] = ms;
    }
    return n;
}

int exchange_launch(ShardCore* sh, PeerRank& r, const fe* ycode, size_t off_recv, cudaStream_t s) {
    pcs_shard_exchange_kernel<<<peer_grid(sh->NL), 256, 0, s>>>(ycode, sh->NL, sh->R, r.rank, sh->grp.peers(), off_recv);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
int tables_launch(ShardCore* sh, PeerRank& r, const fe* src, size_t off_m, cudaStream_t s, bool rev_dest) {
    if (rev_dest) pcs_shard_tables_kernel<true><<<peer_grid(sh->nloc), 256, 0, s>>>(src, sh->nloc, sh->L, r.rank, sh->grp.peers(), off_m);
    else pcs_shard_tables_kernel<false><<<peer_grid(sh->nloc), 256, 0, s>>>(src, sh->nloc, sh->L, r.rank, sh->grp.peers(), off_m);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
int local_eq_table(Ctx* ctx, const std::vector<hfe>& pts, int v, int L, int rank, fe* d, cudaStream_t s) {
    MLB_TRY(eq_table_launch(ctx, pts.data(), (size_t)(v - L), d, s));
    if (L == 0) return ML_OK;
    hfe scale = 1;
    for (int b = 0; b < L; b++) {
        const hfe p = pts[(size_t)(v - 1 - b)];
        scale = hfe_mul(scale, ((rank >> b) & 1) ? p : hfe_sub(1, p));
    }
    const size_t nloc = (size_t)1 << (v - L);
    pcs_shard_scale_kernel<<<peer_grid(nloc), 256, 0, s>>>(d, nloc, to_dev_fe_h(scale));
    MLB_KERNEL_CHECK();
    return ML_OK;
}

template <bool MOBIUS>
int combine_launch_t(int L, const fe* recv, size_t R, int rank, int log_N, const RootTables* rt, fe* layer0, cudaStream_t s) {
    const unsigned grid = peer_grid(R);
    switch (L) {
        case 1: pcs_shard_combine_kernel<1, MOBIUS><<<grid, 256, 0, s>>>(recv, R, rank, log_N, rt->lo, rt->hi, layer0); break;
        case 2: pcs_shard_combine_kernel<2, MOBIUS><<<grid, 256, 0, s>>>(recv, R, rank, log_N, rt->lo, rt->hi, layer0); break;
        case 3: pcs_shard_combine_kernel<3, MOBIUS><<<grid, 256, 0, s>>>(recv, R, rank, log_N, rt->lo, rt->hi, layer0); break;
        case 4: pcs_shard_combine_kernel<4, MOBIUS><<<grid, 256, 0, s>>>(recv, R, rank, log_N, rt->lo, rt->hi, layer0); break;
        default: set_error("ml_pcs_shard: log2(world) = %d out of range", L); return ML_ERR_ARG;
    }
    MLB_KERNEL_CHECK();
    return ML_OK;
}
int combine_launch(int L, const fe* recv, size_t R, int rank, int log_N, const RootTables* rt, fe* layer0, cudaStream_t s, bool mobius) {
    return mobius ? combine_launch_t<true>(L, recv, R, rank, log_N, rt, layer0, s) : combine_launch_t<false>(L, recv, R, rank, log_N, rt, layer0, s);
}

int post_launch(ShardCore* sh, PeerRank& r, const uint8_t* dig, size_t R, int segs, int nb, size_t off_roots, size_t off_partials, int phase) {
    pcs_shard_post_kernel<<<1, 256, 0, r.st.main>>>(at(r, sh->lay.part), nb, dig, R, segs, r.rank, sh->world, sh->grp.peers(), off_roots, off_partials,
                                                    sh->lay.flags + (size_t)phase * MAXR * 8, sh->grp.epoch);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
int top_launch(ShardCore* sh, PeerRank& r, int phase, int k, int cnt) {
    pcs_shard_top_kernel<<<1, 32, 0, r.st.main>>>(sh->grp.flags(r, phase), sh->world, sh->grp.epoch, sh->grp.timeout_ns, sh->grp.status(r),
                                                  r.arena + sh->lay.mail[k], cnt, r.arena + sh->lay.top[k]);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
int finish_launch(ShardCore* sh, PeerRank& r, int k, const uint8_t* root) {
    const Layout& a = sh->lay;
    return chain_sumcheck_finish_launch(at(r, mail_partials(a, k)), sh->world, at(r, a.prev), (DevTranscript*)(r.arena + a.tr), root, root ? 32 : 0,
                                        root ? r.arena + a.roots_out + 32 * k : nullptr, at(r, a.sc) + 2 * k, at(r, a.r), r.st.main);
}

// S0 of one rank: claim state, encode, exchange, tables
int stage_encode(ShardCore* sh, PeerRank& r, const fe* evals, const uint8_t* claim_state, const std::vector<hfe>& pts) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    const Layout& a = sh->lay;
    MLB_TRY(h2d(r.arena + a.tr, claim_state, sizeof(DevTranscript), s));
    MLB_TRY(h2d(r.arena + a.prev, claim_state + sizeof(DevTranscript), 16, s));
    MLB_CUDA(cudaMemsetAsync(sh->grp.status(r), 0, 16, s));
    if (sh->world == 1) {
        MLB_TRY(encode_into(r.ctx, evals, sh->nloc, at(r, a.tail_code), s));
        MLB_CUDA(cudaMemcpyAsync(at(r, a.tail_m), evals, sh->nloc * 16, cudaMemcpyDeviceToDevice, s));
        return local_eq_table(r.ctx, pts, (int)sh->n_vars, sh->L, r.rank, at(r, a.tail_d), s);
    }
    MLB_TRY(encode_into(r.ctx, evals, sh->nloc, at(r, a.ycode), s));
    MLB_TRY(exchange_launch(sh, r, at(r, a.ycode), a.recv, s));
    MLB_TRY(tables_launch(sh, r, evals, a.m, s));
    MLB_TRY(local_eq_table(r.ctx, pts, (int)sh->n_vars, sh->L, r.rank, at(r, a.d), s));
    return peer_signal(sh->grp, r, PX, -1, s);
}

// S1 of one rank: wait for the slices, combine into layer 0, round-0 partial sums
int stage_combine(ShardCore* sh, PeerRank& r, int* nb) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    const Layout& a = sh->lay;
    const int log_N = (int)sh->n_vars + ML_LOG_BLOWUP;
    const RootTables* rt;
    MLB_TRY(get_root_tables(r.ctx, log_N, s, &rt));  // never a lazy build behind a spinning wait
    MLB_TRY(peer_wait(sh->grp, r, PX, -1, s));
    MLB_TRY(combine_launch(sh->L, at(r, a.recv), sh->R, r.rank, log_N, rt, at(r, a.layer[0]), s));
    return sumcheck_sums_partials_launch(at(r, a.m), at(r, a.d), sh->nloc, at(r, a.part), nb, s);
}

// round k, phase A: segment subtrees, post roots + partial sums
int stage_post(ShardCore* sh, PeerRank& r, int k, int nb) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    const Layout& a = sh->lay;
    const size_t segs = (size_t)sh->world >> (k + 1), R = sh->R;
    for (size_t p = 0; p < segs; p++) MLB_TRY(merkle_rs_launch(at(r, a.layer[k]) + p * 2 * R, 2 * R, r.arena + a.dig[k] + 32 * p * 2 * R, s));
    return post_launch(sh, r, r.arena + a.dig[k], R, (int)segs, nb, a.mail[k], mail_partials(a, k), PR0 + k);
}
// round k, phase B: top of the layer tree, round polynomial, challenge (same on every rank)
int stage_round(ShardCore* sh, PeerRank& r, int k) {
    MLB_CUDA(cudaSetDevice(r.device));
    const int cnt = (sh->world * sh->world) >> (k + 1);
    MLB_TRY(top_launch(sh, r, PR0 + k, k, cnt));
    return finish_launch(sh, r, k, r.arena + sh->lay.top[k] + 32 * merkle_layer_offset((size_t)cnt, ilog2((size_t)cnt)));
}
fe* fold_target(ShardCore* sh, PeerRank& r, int k) {
    if (k + 1 == sh->L) return reinterpret_cast<fe*>(sh->grp.base[0] + sh->lay.tail_code) + (size_t)r.rank * sh->R;
    return at(r, sh->lay.layer[k + 1]);
}
int fold_tables(ShardCore* sh, PeerRank& r, int k, int* nb) {
    cudaStream_t s = r.st.main;
    const Layout& a = sh->lay;
    const size_t h = sh->nloc >> k;
    if (k + 1 < sh->L) return sumcheck_fold_sums_launch(at(r, a.m), at(r, a.d), h, at(r, a.r), at(r, a.part), nb, s);  // h >= 4 here
    MLB_TRY(sumcheck_fold_launch(at(r, a.m), at(r, a.d), h, 0, at(r, a.r), s));
    pcs_shard_gather_tables_kernel<<<peer_grid(h / 2), 256, 0, s>>>(at(r, a.m), at(r, a.d), h / 2, r.rank, sh->world,
                                                                   reinterpret_cast<fe*>(sh->grp.base[0] + a.tail_m), reinterpret_cast<fe*>(sh->grp.base[0] + a.tail_d));
    MLB_KERNEL_CHECK();
    return peer_signal(sh->grp, r, PG, 0, s);
}
// round k, phase C: fold tables and code; after the last sharded round, hand layer L and the tables to rank 0
int stage_fold(ShardCore* sh, PeerRank& r, int k, int* nb) {
    MLB_TRY(fold_code(sh, r, k));
    return fold_tables(sh, r, k, nb);
}
int fold_code(ShardCore* sh, PeerRank& r, int k) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    const Layout& a = sh->lay;
    const int log_N = (int)sh->n_vars + ML_LOG_BLOWUP;
    const RootTables* rt;
    MLB_TRY(get_root_tables(r.ctx, log_N, s, &rt));
    const size_t segs = (size_t)sh->world >> (k + 1);
    pcs_shard_fold_kernel<<<peer_grid(segs * sh->R), 256, 0, s>>>(at(r, a.layer[k]), segs, sh->R, sh->NL, r.rank, k, log_N, at(r, a.r), rt->lo, rt->hi,
                                                                  fold_target(sh, r, k));
    MLB_KERNEL_CHECK();
    return ML_OK;
}

int open_sharded(ShardCore* sh, PeerRank& r0, const std::vector<size_t>& idx, int j0, std::vector<uint8_t>& host, int* stride) {
    cudaStream_t s = r0.st.main;
    const int L = sh->L;
    const size_t nq = idx.size();
    OpenArgs oa;
    memset(&oa, 0, sizeof oa);
    oa.stride = *stride = 32 + 32 * 64;
    if (j0 >= L) return ML_OK;
    for (int j = 0; j < L; j++) { oa.off_layer[j] = sh->lay.layer[j]; oa.off_dig[j] = sh->lay.dig[j]; oa.top[j] = r0.arena + sh->lay.top[j]; }
    oa.n = sh->n; oa.NL = sh->NL; oa.R = sh->R; oa.L = L; oa.j0 = j0; oa.world = sh->world; oa.log_R = (int)ilog2(sh->R);
    std::vector<unsigned long long> idx64(idx.begin(), idx.end());
    Scratch didx(s), dout(s);
    MLB_TRY(didx.alloc(nq * 8));
    MLB_TRY(dout.alloc(nq * L * (size_t)oa.stride));
    MLB_TRY(h2d(didx.p, idx64.data(), nq * 8, s));
    pcs_shard_open_kernel<<<dim3((unsigned)nq, (unsigned)(L - j0)), 64, 0, s>>>(didx.as<unsigned long long>(), sh->grp.peers(), oa, dout.as<uint8_t>());
    MLB_KERNEL_CHECK();
    host.resize(nq * L * (size_t)oa.stride);
    return d2h_sync(host.data(), dout.p, host.size(), s);
}

int tail_chain(ShardCore* sh, PeerRank& r0, ml_fri* f, const ChainHooks& hooks, hfe* sumcheck, uint8_t* roots_lo, ml_transcript* t, int mark_base) {
    MLB_CUDA(cudaSetDevice(r0.device));
    cudaStream_t s = r0.st.main;
    const Layout& a = sh->lay;
    const int L = sh->L;
    if (L > 0) MLB_TRY(peer_wait(sh->grp, r0, PG, -1, s));
    if (&r0 == &sh->local[0]) mark_phase(sh, mark_base);
    f->log_n0 = (int)sh->n_vars + ML_LOG_BLOWUP;
    f->stream = s;
    if (!hooks.first_fold) MLB_TRY(fri_push_layer(f, at(r0, a.tail_code), sh->NL, false, s, true));  // layer L, committed, root not absorbed yet
    ml_sumcheck sc;  // tables in the arena: not freed by the chain
    sc.matrix = at(r0, a.tail_m);
    sc.delta = at(r0, a.tail_d);
    sc.owns_matrix = false;
    sc.height = sh->nloc;
    sc.stream = s;
    ChainHooks h = hooks;
    h.tr_dev = (const DevTranscript*)(r0.arena + a.tr);
    h.prev_dev = at(r0, a.prev);
    MLB_TRY(fold_chain_dev(r0.ctx, f, &h, sumcheck ? &sc : nullptr, 0, sumcheck ? sumcheck + 2 * L : nullptr, (size_t)L, !hooks.first_fold, t, s));
    if (&r0 == &sh->local[0]) mark_phase(sh, mark_base + 1);
    if (L > 0) {  // sumcheck (c1, c2) and layer roots of the sharded rounds
        uint8_t lo[MAX_L * 32];
        if (sumcheck) MLB_CUDA(cudaMemcpyAsync(lo, r0.arena + a.sc, (size_t)L * 32, cudaMemcpyDeviceToHost, s));
        MLB_TRY(d2h_sync(roots_lo, r0.arena + a.roots_out, (size_t)L * 32, s));
        if (sumcheck)
            for (int i = 0; i < 2 * L; i++) sumcheck[i] = hfe_load(lo + 16 * i);
    }
    return peer_read_status(sh->grp, r0, sh->who);
}

int tail_release(ShardCore* sh, PeerRank& r0, ml_transcript* t) {
    if (sh->world == 1) return ML_OK;
    cudaStream_t s = r0.st.main;
    Scratch trd(s);
    MLB_TRY(trd.alloc(128));
    MLB_TRY(h2d(trd.p, &t->sha, sizeof(DevTranscript), s));
    MLB_TRY(peer_push(sh->grp, r0, trd.p, (int)(sizeof(DevTranscript) + 15) / 16 * 16, sh->lay.final_tr, PF, -1, s));
    return stream_wait_blocking(s);
}
int tail_fail(ShardCore* sh, PeerRank& r0, int st) {
    if (sh->world == 1) return ML_OK;
    cudaStream_t s = r0.st.main;
    const int word[4] = {st, 0, 0, 0};
    Scratch d(s);
    MLB_TRY(d.alloc(16));
    MLB_TRY(h2d(d.p, word, 16, s));
    MLB_TRY(peer_push(sh->grp, r0, d.p, 16, sh->lay.status, PF, -1, s));
    return stream_wait_blocking(s);
}

// ranks other than 0: wait for the end of the proof (their buffers are read by rank 0's openings until then)
int finish_ranks(ShardCore* sh, ml_transcript* t, int st) {
    for (auto& r : sh->local) {
        if (r.rank == 0) continue;
        MLB_CUDA(cudaSetDevice(r.device));
        MLB_TRY(peer_wait(sh->grp, r, PF, 0, r.st.main));
        int s1 = peer_read_status(sh->grp, r, sh->who);
        if (s1 != ML_OK) { st = s1; continue; }
        if (!rank0_of(sh)) {  // another process holds rank 0: adopt its final transcript
            HostSha256 fin;
            MLB_TRY(d2h_sync(&fin, r.arena + sh->lay.final_tr, sizeof(DevTranscript), r.st.main));
            t->sha = fin;
        }
    }
    return st;
}

int assemble_fri(ShardCore* sh, PeerRank& r0, const ml_fri* f, ml_transcript* t, ml_fri_proof* p, const uint8_t* roots_lo) {
    cudaStream_t s = r0.st.main;
    const int L = sh->L;
    std::vector<size_t> idx;
    derive_indices(t, 2 * sh->n, idx);
    const size_t nq = idx.size();
    std::vector<uint8_t> host;
    int stride = 0;
    MLB_TRY(open_sharded(sh, r0, idx, 0, host, &stride));
    std::vector<size_t> sub(nq);
    for (size_t q = 0; q < nq; q++) sub[q] = idx[q] % (sh->n >> L);
    std::vector<QueryH> qs;
    MLB_TRY(fri_open_queries(f, sub, qs, s));
    p->queries.assign(nq, QueryH());
    for (size_t q = 0; q < nq; q++) {
        std::vector<PathH>& paths = p->queries[q].paths;
        paths.resize(L);
        for (int j = 0; j < L; j++) {
            const uint8_t* rec = host.data() + (q * L + j) * (size_t)stride;
            const int depth = (int)ilog2(sh->n >> j);
            paths[j].value.assign(rec, rec + 32);
            paths[j].digests.assign(rec + 32, rec + 32 + 32 * (size_t)depth);
            fill_dirs(paths[j], idx[q] % (sh->n >> j), depth);
        }
        for (auto& ph : qs[q].paths) paths.push_back(std::move(ph));
    }
    p->commitments.assign(roots_lo, roots_lo + 32 * (size_t)L);
    for (const auto& layer : f->layers) p->commitments.insert(p->commitments.end(), layer.tree->root, layer.tree->root + 32);
    p->last_elem = f->last;
    t->sha.digest(p->last_random);
    return ML_OK;
}

}  // namespace mlbs

namespace {

const char* WHO = "ml_pcs_shard";

// rank 0: the rest of the fold chain from layer L, the openings (:113-129), the final transcript to everybody
int prove_tail(ml_pcs_shard* sh, PeerRank& r0, const uint8_t* inputs, const uint8_t* output, ml_transcript* t, ml_pcs_proof** out) {
    ml_fri* f = new ml_fri();
    struct FriGuard { ml_fri* p; ~FriGuard() { free_fri(p); } } fri_guard{f};
    ml_pcs_proof* p = new ml_pcs_proof();
    std::unique_ptr<ml_pcs_proof> guard(p);
    p->sumcheck.resize(2 * sh->n_vars);
    uint8_t roots_lo[MAX_L * 32];
    MLB_TRY(tail_chain(sh, r0, f, ChainHooks(), p->sumcheck.data(), roots_lo, t, 3));
    MLB_TRY(assemble_fri(sh, r0, f, t, &p->fri, roots_lo));
    if (&r0 == &sh->local[0]) mark_phase(sh, 5);
    p->inputs.resize(sh->n_vars);
    for (size_t i = 0; i < sh->n_vars; i++) p->inputs[i] = hfe_load(inputs + 16 * i);
    p->output = hfe_load(output);
    MLB_TRY(tail_release(sh, r0, t));  // also releases the other ranks' buffers for the next call
    *out = guard.release();
    return ML_OK;
}

}  // namespace

extern "C" {

int ml_pcs_shard_create(int world, int n_local, const int* local_ranks, const int* local_devices, size_t n_vars, ml_pcs_shard** out) {
    MLB_TRY(peer_check_world("ml_pcs_shard_create", world, n_local));
    const int L = (int)ilog2((size_t)world);
    if (n_vars < 1 || n_vars < (size_t)(2 * L) || n_vars >= 40) {
        set_error("ml_pcs_shard_create: n_vars = %zu, need max(1, 2*log2(world)) = %d <= n_vars < 40", n_vars, L ? 2 * L : 1);
        return ML_ERR_SIZE;
    }
    DeviceGuard guard;
    ml_pcs_shard* sh = new ml_pcs_shard();
    int st = shard_init(sh, world, n_local, local_ranks, local_devices, n_vars, 0, "ml_pcs_shard_create");
    if (st != ML_OK) { ml_pcs_shard_free(sh); return st; }
    *out = sh;
    return ML_OK;
}

void ml_pcs_shard_free(ml_pcs_shard* sh) {
    if (!sh) return;
    shard_free(sh);
    delete sh;
}

int ml_pcs_shard_export(ml_pcs_shard* sh, uint8_t* records_out) { return shard_export(sh, records_out); }
int ml_pcs_shard_connect(ml_pcs_shard* sh, const uint8_t* records, size_t n_records) { return shard_connect(sh, records, n_records, "ml_pcs_shard_connect"); }
void* ml_pcs_shard_stream(const ml_pcs_shard* sh, int local_index) { return shard_stream(sh, local_index); }
size_t ml_pcs_shard_arena_bytes(const ml_pcs_shard* sh) { return sh->lay.total; }

// INSTRUMENTATION (include/multilinear_b200_instr.h): device time between the phase marks of the last call on the first local
// rank's main stream, in ms: [S0 encode + exchange + tables, S1 combine, sharded rounds, tail chain, openings] (the last two
// on rank 0 only).  Returns the count.
int ml_pcs_shard_phase_ms(const ml_pcs_shard* sh, double* out, int cap) { return shard_phase_ms(sh, out, cap); }

// PCSProof::prove (multilinear_pcs.rs:90-136).  Every process calls it with the same claim and its own transcript copy; the proof
// comes out on the process that hosts rank 0 (*out = NULL elsewhere); every transcript ends in the same state.
int ml_pcs_shard_prove_dev(ml_pcs_shard* sh, const uint8_t* inputs, size_t n_vars, const uint8_t output[16], const void* const* local_evals_dev,
                           ml_transcript* t, ml_pcs_proof** out) {
    MLB_TRY(peer_check_ready(sh->grp, WHO));
    if (n_vars != sh->n_vars) { set_error("ml_pcs_shard_prove: the claim has %zu variables, the handle %zu", n_vars, sh->n_vars); return ML_ERR_SIZE; }
    DeviceGuard guard;
    *out = nullptr;
    sh->grp.epoch++;
    std::vector<hfe> pts(n_vars);
    for (size_t i = 0; i < n_vars; i++) pts[i] = hfe_load(inputs + 16 * i);
    uint8_t claim_state[sizeof(DevTranscript) + 16];  // the device transcript and the running claim start as tr | output
    memcpy(claim_state, &t->sha, sizeof(DevTranscript));
    memcpy(claim_state + sizeof(DevTranscript), output, 16);
    const size_t nl = sh->local.size();
    std::vector<int> nb(nl, 0);
    sh->n_marks = 0;
    mark_phase(sh, 0);
    for (size_t i = 0; i < nl; i++) MLB_TRY(stage_encode(sh, sh->local[i], (const fe*)local_evals_dev[i], claim_state, pts));
    mark_phase(sh, 1);
    if (sh->L > 0) {
        for (size_t i = 0; i < nl; i++) MLB_TRY(stage_combine(sh, sh->local[i], &nb[i]));
        mark_phase(sh, 2);
        for (int k = 0; k < sh->L; k++) {
            for (size_t i = 0; i < nl; i++) MLB_TRY(stage_post(sh, sh->local[i], k, nb[i]));
            for (size_t i = 0; i < nl; i++) MLB_TRY(stage_round(sh, sh->local[i], k));
            for (size_t i = 0; i < nl; i++) MLB_TRY(stage_fold(sh, sh->local[i], k, &nb[i]));
        }
    } else {
        mark_phase(sh, 2);
    }
    int st = ML_OK;
    if (PeerRank* r0 = rank0_of(sh)) st = prove_tail(sh, *r0, inputs, output, t, out);
    st = finish_ranks(sh, t, st);
    if (st != ML_OK && *out) { ml_pcs_proof_free(*out); *out = nullptr; }
    return st;
}

// host evaluations (all n) and a handle that hosts every rank: the drop-in for multilinear_pcs.rs:90
int ml_pcs_shard_prove(ml_pcs_shard* sh, const uint8_t* inputs, size_t n_vars, const uint8_t output[16], const uint8_t* evals, size_t n,
                       ml_transcript* t, ml_pcs_proof** out) {
    if ((int)sh->local.size() != sh->world) { set_error("ml_pcs_shard_prove: host-pointer entry needs a handle that hosts every rank"); return ML_ERR_ARG; }
    if (n_vars != sh->n_vars || n != sh->n) { set_error("ml_pcs_shard_prove: need 2^n_vars == evals.len() == the handle's size"); return ML_ERR_SIZE; }
    DeviceGuard guard;
    std::vector<void*> dev(sh->local.size(), nullptr);
    int st = ML_OK;
    for (size_t i = 0; i < sh->local.size() && st == ML_OK; i++) {
        PeerRank& r = sh->local[i];
        if (cudaSetDevice(r.device) != cudaSuccess) { st = ML_ERR_CUDA; break; }
        st = pmalloc(&dev[i], sh->nloc * 16, r.st.main);
        if (st == ML_OK) st = h2d(dev[i], evals + (size_t)r.rank * sh->nloc * 16, sh->nloc * 16, r.st.main);
        if (st == ML_OK && cudaStreamSynchronize(r.st.main) != cudaSuccess) st = ML_ERR_CUDA;
    }
    if (st == ML_OK) st = ml_pcs_shard_prove_dev(sh, inputs, n_vars, output, dev.data(), t, out);
    for (size_t i = 0; i < sh->local.size(); i++) {
        cudaSetDevice(sh->local[i].device);
        cudaStreamSynchronize(sh->local[i].st.main);
        pfree(dev[i], sh->local[i].st.main);
    }
    return st;
}

}  // extern "C"
