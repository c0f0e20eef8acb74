// Sync-free fold chain: device-resident transcript steps and the fused tail kernel.
//
// Reference control flow (src/fri/mod.rs:136-145, src/fri/multilinear_pcs.rs:58-73): per round the prover
//   [sumcheck: two partial sums -> round polynomial -> absorb c1,c2] -> r = next_challenge() -> fold tables and code
//   with r -> Merkle-commit the folded code -> absorb its root.
// Every step depends on the previous one through the transcript.  With the transcript on the host that is one
// device->host round trip per round (24 at 2^24).  Here:
//   * large rounds: the same kernels as before, but the challenge is produced by a one-thread kernel that advances
//     the transcript in HBM and leaves r (and r/2) in device memory for the fold kernels — nothing returns to the host;
//   * once the code fits one CTA (<= 4096 elements) a single kernel runs ALL remaining rounds: sumcheck sums,
//     transcript, table fold, FRI fold, leaf hashes, tree levels, in shared/L2 with __syncthreads between phases.
//     This replaces ~60 latency-bound launches (ncu: 20-220 us each, profiles/r1_launches_bench_v0.csv).
#include "field.cuh"
#include "internal.h"
#include "reduce.cuh"
#include "sha256.cuh"

namespace mlb {
// single expansions of the compression function for the whole translation unit (leaf, node and transcript hashing)
static __device__ __noinline__ void chain_compress(uint32_t st[8], uint32_t w[16]) { sha_compress(st, w); }
static __device__ __noinline__ void chain_compress_pad512(uint32_t st[8]) { sha_compress_pad512(st); }
}  // namespace mlb
#define MLB_DT_COMPRESS(h, w) chain_compress(h, w)
#include "transcript.cuh"

namespace mlb {

__device__ __forceinline__ void chain_leaf(uint4 x, uint4 y, uint32_t out[8]) {
    uint32_t w[16];
    sha_words_from_le(x, w);
    sha_words_from_le(y, w + 4);
    w[8] = 0x80000000u; w[9] = 0; w[10] = 0; w[11] = 0; w[12] = 0; w[13] = 0; w[14] = 0; w[15] = 256u;
    sha_iv(out);
    chain_compress(out, w);
}
__device__ __forceinline__ void chain_node(const uint32_t l[8], const uint32_t r[8], uint32_t out[8]) {
    uint32_t w[16];
#pragma unroll
    for (int k = 0; k < 8; k++) { w[k] = l[k]; w[8 + k] = r[k]; }
    sha_iv(out);
    chain_compress(out, w);
    chain_compress_pad512(out);
}
__device__ __forceinline__ uint8_t* chain_layer_ptr(uint8_t* digests, size_t n_leaves, int layer, size_t idx) {
    return digests + 32 * ((2 * n_leaves - ((2 * n_leaves) >> layer)) + idx);
}
__device__ __forceinline__ fe chain_root_pow(const fe* __restrict__ lo, const fe* __restrict__ hi, size_t e) {
    fe w = fe_load_nc(lo + (e & (((size_t)1 << LO_BITS) - 1)));
    if (e >> LO_BITS) w = fe_mul(w, fe_load_nc(hi + (e >> LO_BITS)));
    return w;
}

// ------------------------------------------------------------------ transcript step kernels
// absorb `absorb_len` bytes at `absorb` (a Merkle root in HBM), copy them to `copy_out`, then r = next_challenge():
// r_out[0] = r, r_out[1] = r / 2
__global__ void chain_challenge_kernel(DevTranscript* tr, const uint8_t* absorb, int absorb_len, uint8_t* copy_out, fe* r_out,
                                       int want_challenge) {
    if (threadIdx.x != 0) return;
    DevTranscript t = *tr;
    if (absorb_len > 0) {
        dt_absorb(&t, absorb, absorb_len);
        if (copy_out)
            for (int i = 0; i < absorb_len; i++) copy_out[i] = absorb[i];
        *tr = t;
    }
    if (want_challenge) {
        fe r = dt_challenge(&t);
        fe_store(r_out, r);
        fe_store(r_out + 1, fe_half(r));
    }
}
// sumcheck round bookkeeping (src/constraint_system/sumcheck.rs:185-199) from the per-CTA partial sums:
//   e1, e2 -> e0 = prev - e1 -> (c1, c2) -> absorb -> r -> prev = p(r)
__global__ void __launch_bounds__(256) chain_sumcheck_finish_kernel(const fe* __restrict__ partials, int nb, fe* prev, DevTranscript* tr,
                                                                    const uint8_t* absorb, int absorb_len, uint8_t* copy_out,
                                                                    fe* sc_out, fe* r_out) {
    __shared__ fe scratch[32];
    fe a1 = fe_zero(), a2 = fe_zero();
    for (int b = threadIdx.x; b < nb; b += blockDim.x) {
        a1 = fe_add(a1, partials[2 * b]);
        a2 = fe_add(a2, partials[2 * b + 1]);
    }
    fe e1 = block_sum(a1, scratch);
    fe e2 = block_sum(a2, scratch);
    if (threadIdx.x != 0) return;
    DevTranscript t = *tr;
    if (absorb_len > 0) {
        dt_absorb(&t, absorb, absorb_len);
        if (copy_out)
            for (int i = 0; i < absorb_len; i++) copy_out[i] = absorb[i];
    }
    fe e0 = fe_sub(fe_load(prev), e1);
    fe c2 = fe_half(fe_add(fe_sub(e0, fe_add(e1, e1)), e2));  // (e0 - 2 e1 + e2) / 2
    fe c1 = fe_sub(fe_sub(e1, e0), c2);
    dt_absorb_fe(&t, c1);  // nonzero_coeffs = coeffs[1..] (sumcheck.rs:193-197, :263-267)
    dt_absorb_fe(&t, c2);
    fe r = dt_challenge(&t);
    fe_store(prev, fe_add(e0, fe_mul(r, fe_add(c1, fe_mul(r, c2)))));
    fe_store(sc_out, c1);
    fe_store(sc_out + 1, c2);
    fe_store(r_out, r);
    fe_store(r_out + 1, fe_half(r));
    *tr = t;
}

// FriProof::prove's query phase (src/fri/mod.rs:268-277) on one thread, from the transcript the fold chain left in HBM:
// 128 times idx = LE u64 of the digest's first 8 bytes mod N/2 (a mask: N/2 is a power of two), then absorb idx as 8 LE bytes;
// last_random = the digest after the last absorb.  The transcript's final state goes to tr_out.
__global__ void fri_query_indices_kernel(const DevTranscript* tr_in, DevTranscript* tr_out, int log_half, unsigned long long* indices,
                                         uint8_t* last_random) {
    if (threadIdx.x != 0) return;
    DevTranscript t = *tr_in;
    const unsigned long long mask = (1ull << log_half) - 1ull;
    uint32_t st[8];
    for (int q = 0; q < ML_NUM_QUERIES; q++) {
        dt_digest_words(&t, st);
        // digest bytes are the big-endian state words: bytes 0..7 read as LE u64 -> bswap(st[0]) | bswap(st[1]) << 32
        const unsigned long long idx = ((unsigned long long)sha_bswap(st[0]) | ((unsigned long long)sha_bswap(st[1]) << 32)) & mask;
        indices[q] = idx;
        uint8_t b[8];
#pragma unroll
        for (int i = 0; i < 8; i++) b[i] = (uint8_t)(idx >> (8 * i));
        dt_absorb(&t, b, 8);
    }
    dt_digest_words(&t, st);
    for (int i = 0; i < 8; i++) {
        last_random[4 * i] = (uint8_t)(st[i] >> 24); last_random[4 * i + 1] = (uint8_t)(st[i] >> 16);
        last_random[4 * i + 2] = (uint8_t)(st[i] >> 8); last_random[4 * i + 3] = (uint8_t)st[i];
    }
    *tr_out = t;
}
int fri_query_indices_launch(const DevTranscript* tr_in, DevTranscript* tr_out, int log_half, unsigned long long* indices, uint8_t* last_random,
                             cudaStream_t s) {
    ProfScope prof(PROF_TRANSCRIPT, 0.0, s);
    fri_query_indices_kernel<<<1, 32, 0, s>>>(tr_in, tr_out, log_half, indices, last_random);
    MLB_KERNEL_CHECK();
    return ML_OK;
}

// ------------------------------------------------------------------ fused tail
__global__ void __launch_bounds__(1024, 1) chain_tail_kernel(TailArgs a) {
    __shared__ DevTranscript tr;
    __shared__ fe sh_r[2];
    __shared__ fe sh_prev;
    __shared__ fe scratch[32];
    const int tid = threadIdx.x, nthreads = blockDim.x;
    if (tid == 0) {
        tr = *a.tr;
        if (a.m) sh_prev = fe_load(a.prev);
    }
    __syncthreads();
    size_t n = a.n0, h = a.height;
    int k = a.k0;
    const size_t n_domain = (size_t)1 << a.log_n0;
    const uint8_t* pending = a.absorb_first_root ? chain_layer_ptr(a.digests[0], n >> 1, (int)(63 - __clzll((unsigned long long)(n >> 1))), 0) : nullptr;
    uint8_t* pending_copy = a.absorb_first_root ? a.first_root_out : nullptr;
    const fe* cur = a.codes[0];
    for (int round = 0; n > 2; round++, k++) {
        const size_t half_n = n >> 1;
        // ---- A: (sumcheck sums ->) challenge
        if (a.m) {
            const size_t off = h >> 1;
            fe_acc s1, s2;
            acc_zero(s1);
            acc_zero(s2);
            for (size_t i = tid; i < off; i += nthreads) {
                fe m0 = fe_load(a.m + i), m1 = fe_load(a.m + i + off), d0 = fe_load(a.d + i), d1 = fe_load(a.d + i + off);
                acc_mul_add(s1, m1, d1);
                acc_mul_add(s2, fe_sub(fe_add(m1, m1), m0), fe_sub(fe_add(d1, d1), d0));
            }
            fe e1 = block_sum(acc_reduce(s1), scratch);
            fe e2 = block_sum(acc_reduce(s2), scratch);
            if (tid == 0) {
                if (pending) {
                    dt_absorb(&tr, pending, 32);
                    if (pending_copy) for (int i = 0; i < 32; i++) pending_copy[i] = pending[i];
                }
                fe e0 = fe_sub(sh_prev, e1);
                fe c2 = fe_half(fe_add(fe_sub(e0, fe_add(e1, e1)), e2));
                fe c1 = fe_sub(fe_sub(e1, e0), c2);
                dt_absorb_fe(&tr, c1);
                dt_absorb_fe(&tr, c2);
                fe r = dt_challenge(&tr);
                sh_prev = fe_add(e0, fe_mul(r, fe_add(c1, fe_mul(r, c2))));
                fe_store(a.sc_out + 2 * round, c1);
                fe_store(a.sc_out + 2 * round + 1, c2);
                sh_r[0] = r;
                sh_r[1] = fe_half(r);
            }
        } else if (tid == 0) {
            if (pending) {
                dt_absorb(&tr, pending, 32);
                if (pending_copy) for (int i = 0; i < 32; i++) pending_copy[i] = pending[i];
            }
            fe r = dt_challenge(&tr);
            sh_r[0] = r;
            sh_r[1] = fe_half(r);
        }
        __syncthreads();
        const fe r = sh_r[0], rh = sh_r[1];
        // ---- B: fold the sumcheck tables (sumcheck.rs:234-247)
        if (a.m) {
            const size_t off = h >> 1;
            for (size_t i = tid; i < off; i += nthreads) {
                fe m0 = fe_load(a.m + i), m1 = fe_load(a.m + i + off), d0 = fe_load(a.d + i), d1 = fe_load(a.d + i + off);
                fe_store(a.m + i, fe_add(m0, fe_mul(r, fe_sub(m1, m0))));
                fe_store(a.d + i, fe_add(d0, fe_mul(r, fe_sub(d1, d0))));
            }
            h = off;
        }
        // ---- C: FRI fold (fri/mod.rs:90-114)
        fe* next = half_n == 2 ? a.last_out : a.codes[round + 1];
        for (size_t i = tid; i < half_n; i += nthreads) {
            fe x = fe_load(cur + i), y = fe_load(cur + i + half_n);
            fe even = fe_half(fe_add(x, y));
            fe dd = fe_sub(x, y);
            if (i != 0) dd = fe_mul(dd, chain_root_pow(a.lo, a.hi, n_domain - (i << k)));
            fe_store(next + i, fe_add(even, fe_mul(rh, dd)));
        }
        __syncthreads();
        if (half_n == 2) {  // fri/mod.rs:116-126
            if (tid == 0) {
                fe x0 = fe_load(next), x1 = fe_load(next + 1);
                if (!fe_eq(x0, x1)) *a.status = ML_ERR_NOT_RS_CODE;
                else dt_absorb_fe(&tr, x0);
            }
            pending = nullptr;
            break;
        }
        // ---- D: Merkle commit of the folded code (fri/mod.rs:128-133)
        const size_t L = half_n >> 1;
        uint8_t* dig = a.digests[round + 1];
        for (size_t i = tid; i < L; i += nthreads) {
            uint32_t o[8];
            chain_leaf(*reinterpret_cast<const uint4*>(next + i), *reinterpret_cast<const uint4*>(next + i + L), o);
            sha_store_digest(chain_layer_ptr(dig, L, 0, i), o);
        }
        __syncthreads();
        int layer = 0;
        for (size_t cnt = L; cnt > 1; cnt >>= 1, layer++) {
            for (size_t i = tid; i < (cnt >> 1); i += nthreads) {
                uint32_t l[8], rr[8], o[8];
                sha_load_digest(chain_layer_ptr(dig, L, layer, 2 * i), l);
                sha_load_digest(chain_layer_ptr(dig, L, layer, 2 * i + 1), rr);
                chain_node(l, rr, o);
                sha_store_digest(chain_layer_ptr(dig, L, layer + 1, i), o);
            }
            __syncthreads();
        }
        pending = chain_layer_ptr(dig, L, layer, 0);
        pending_copy = a.roots_out + 32 * round;
        cur = next;
        n = half_n;
    }
    if (tid == 0) {
        if (pending) {  // only when the loop never ran (n0 <= 2)
            dt_absorb(&tr, pending, 32);
            if (pending_copy) for (int i = 0; i < 32; i++) pending_copy[i] = pending[i];
        }
        *a.tr = tr;
        if (a.m) fe_store(a.prev, sh_prev);
    }
}

// last fold produced two elements: they must be equal (fri/mod.rs:116-126); absorb the last element
__global__ void chain_last_kernel(const fe* two, DevTranscript* tr, fe* last_out, int* status) {
    if (threadIdx.x != 0) return;
    fe x0 = fe_load(two), x1 = fe_load(two + 1);
    if (!fe_eq(x0, x1)) { *status = ML_ERR_NOT_RS_CODE; return; }
    DevTranscript t = *tr;
    dt_absorb_fe(&t, x0);
    *tr = t;
    fe_store(last_out, x0);
}
int chain_last_launch(const fe* two, DevTranscript* tr, fe* last_out, int* status, cudaStream_t s) {
    chain_last_kernel<<<1, 32, 0, s>>>(two, tr, last_out, status);
    MLB_KERNEL_CHECK();
    return ML_OK;
}

// sumcheck-only tail (compute_sumcheck_polynomials, sumcheck.rs:147-172): all remaining rounds of tables with
// height <= 4096 in one CTA; writes (c1, c2) and r per round
__global__ void __launch_bounds__(1024, 1) chain_sumcheck_tail_kernel(fe* m, fe* d, size_t height, fe* prev, DevTranscript* trp, fe* sc_out,
                                                                      fe* r_out) {
    __shared__ DevTranscript tr;
    __shared__ fe sh_r, sh_prev, scratch[32];
    const int tid = threadIdx.x, nthreads = blockDim.x;
    if (tid == 0) { tr = *trp; sh_prev = fe_load(prev); }
    __syncthreads();
    int round = 0;
    for (size_t h = height; h > 1; h >>= 1, round++) {
        const size_t off = h >> 1;
        fe_acc s1, s2;
        acc_zero(s1);
        acc_zero(s2);
        for (size_t i = tid; i < off; i += nthreads) {
            fe m0 = fe_load(m + i), m1 = fe_load(m + i + off), d0 = fe_load(d + i), d1 = fe_load(d + i + off);
            acc_mul_add(s1, m1, d1);
            acc_mul_add(s2, fe_sub(fe_add(m1, m1), m0), fe_sub(fe_add(d1, d1), d0));
        }
        fe e1 = block_sum(acc_reduce(s1), scratch);
        fe e2 = block_sum(acc_reduce(s2), scratch);
        if (tid == 0) {
            fe e0 = fe_sub(sh_prev, e1);
            fe c2 = fe_half(fe_add(fe_sub(e0, fe_add(e1, e1)), e2));
            fe c1 = fe_sub(fe_sub(e1, e0), c2);
            dt_absorb_fe(&tr, c1);
            dt_absorb_fe(&tr, c2);
            fe r = dt_challenge(&tr);
            sh_prev = fe_add(e0, fe_mul(r, fe_add(c1, fe_mul(r, c2))));
            fe_store(sc_out + 2 * round, c1);
            fe_store(sc_out + 2 * round + 1, c2);
            fe_store(r_out + round, r);
            sh_r = r;
        }
        __syncthreads();
        const fe r = sh_r;
        for (size_t i = tid; i < off; i += nthreads) {
            fe m0 = fe_load(m + i), m1 = fe_load(m + i + off), d0 = fe_load(d + i), d1 = fe_load(d + i + off);
            fe_store(m + i, fe_add(m0, fe_mul(r, fe_sub(m1, m0))));
            fe_store(d + i, fe_add(d0, fe_mul(r, fe_sub(d1, d0))));
        }
        __syncthreads();
    }
    if (tid == 0) { *trp = tr; fe_store(prev, sh_prev); }
}
int chain_sumcheck_tail_launch(fe* m, fe* d, size_t height, fe* prev, DevTranscript* tr, fe* sc_out, fe* r_out, cudaStream_t s) {
    ProfScope prof(PROF_TAIL, 0.0, s);
    chain_sumcheck_tail_kernel<<<1, 1024, 0, s>>>(m, d, height, prev, tr, sc_out, r_out);
    MLB_KERNEL_CHECK();
    return ML_OK;
}

// ------------------------------------------------------------------ width-w sumcheck rounds (sumcheck.rs:174-202) on the device
// Round bookkeeping by the first warp: evals[1..td] (already summed) -> evals[0] = prev - evals[1] (:188) -> coefficients through
// the precomputed Lagrange matrix over x = 0..td (interpolate, :189-192; lane i*n + j multiplies lag[i][j] * y[j], row sums by
// shuffles) -> lane 0: absorb coeffs[1..] (:193-197) -> r (:198) -> prev = p(r) (:199).  `lag_sh` and `ev` live in shared memory.
// Returns r (valid in lane 0); writes coef_out[0..td) and *prev_io from lane 0.
__device__ __forceinline__ fe wchain_round_warp(const fe* ev /* shared: td values, points 1..td */, int td, const fe* lag_sh /* shared (td+1)^2 */,
                                                fe* prev_io /* shared */, DevTranscript* t /* lane 0's */, fe* coef_out) {
    const int lane = threadIdx.x & 31, n = td + 1;
    const int i = lane / n, j = lane - i * n;
    fe term = fe_zero();
    if (lane < n * n) {
        const fe y = j == 0 ? fe_sub(*prev_io, ev[0]) : ev[j - 1];
        term = fe_mul(lag_sh[i * n + j], y);
    }
    // row sum over j: lanes i*n .. i*n + n - 1 (n <= 5)
    fe acc = term;
    for (int d = 1; d < n; d++) {
        fe o;
#pragma unroll
        for (int k = 0; k < 4; k++) o.v[k] = __shfl_down_sync(0xffffffffu, term.v[k], d);
        if (j + d < n) acc = fe_add(acc, o);
    }
    // coefficient c_i now sits in lane i*n; bring c_0..c_td to lane 0
    fe c[W_MAX_TD + 1];
#pragma unroll
    for (int q = 0; q <= W_MAX_TD; q++) {
        const int src = q <= td ? q * n : 0;
#pragma unroll
        for (int k = 0; k < 4; k++) c[q].v[k] = __shfl_sync(0xffffffffu, acc.v[k], src);
    }
    fe r = fe_zero();
    if (lane == 0) {
#pragma unroll
        for (int q = 1; q <= W_MAX_TD; q++)
            if (q <= td) { dt_absorb_fe(t, c[q]); fe_store(coef_out + (q - 1), c[q]); }
        r = dt_challenge(t);
        fe v = fe_zero();
#pragma unroll
        for (int q = W_MAX_TD; q >= 0; q--)
            if (q <= td) v = fe_add(fe_mul(v, r), c[q]);
        *prev_io = v;
    }
    return r;
}
__global__ void __launch_bounds__(256) wchain_finish_kernel(const fe* __restrict__ partials, int nb, int td, const fe* __restrict__ lag, fe* prev,
                                                            DevTranscript* tr, fe* coef_out, fe* r_store, fe* r_dev) {
    __shared__ fe scratch[32];
    __shared__ fe ev[W_MAX_TD], lag_sh[(W_MAX_TD + 1) * (W_MAX_TD + 1)], sh_prev;
    __shared__ DevTranscript sh_tr;
    const int n = td + 1;
    if (threadIdx.x >= 64 && threadIdx.x < 64 + n * n) lag_sh[threadIdx.x - 64] = fe_load(lag + (threadIdx.x - 64));
    if (threadIdx.x == 128) sh_prev = fe_load(prev);
    if (threadIdx.x >= 160 && threadIdx.x < 160 + (int)(sizeof(DevTranscript) / 4))
        reinterpret_cast<uint32_t*>(&sh_tr)[threadIdx.x - 160] = reinterpret_cast<const uint32_t*>(tr)[threadIdx.x - 160];
    for (int k = 0; k < td; k++) {
        fe a = fe_zero();
        for (int b = threadIdx.x; b < nb; b += blockDim.x) a = fe_add(a, partials[(size_t)b * td + k]);
        a = block_sum(a, scratch);
        if (threadIdx.x == 0) ev[k] = a;
    }
    __syncthreads();
    if (threadIdx.x >= 32) return;
    DevTranscript t;
    if (threadIdx.x == 0) t = sh_tr;
    const fe r = wchain_round_warp(ev, td, lag_sh, &sh_prev, &t, coef_out);
    if (threadIdx.x != 0) return;
    fe_store(prev, sh_prev);
    fe_store(r_store, r);
    fe_store(r_dev, r);
    *tr = t;
}
// every remaining round of small width-w tables in one CTA: points 1..td in one pass per round (row_{r+1} = row_r + (x1 - x0)),
// round bookkeeping on the first warp, fold, repeat.  WMAX bounds the row arrays (4 keeps them in registers for narrow traces).
template <int WMAX>
__global__ void __launch_bounds__(512, 1) wchain_tail_kernel(fe* m, fe* d, size_t height, int width, WTerms terms, int td, const fe* __restrict__ lag,
                                                             fe* prev, DevTranscript* trp, fe* coef_out, fe* rs_out) {
    __shared__ DevTranscript tr;
    __shared__ fe sh_r, sh_prev, scratch[32], ev[W_MAX_TD], lag_sh[(W_MAX_TD + 1) * (W_MAX_TD + 1)];
    __shared__ fe t_coef[W_MAX_TERMS];
    __shared__ uint32_t t_len[W_MAX_TERMS], t_off[W_MAX_TERMS], t_cols[W_MAX_COLS];
    const int tid = threadIdx.x, nthreads = blockDim.x;
    for (int t = tid; t < terms.n_terms; t += nthreads) { t_coef[t] = terms.coef[t]; t_len[t] = terms.len[t]; t_off[t] = terms.off[t]; }
    for (int c = tid; c < terms.n_cols; c += nthreads) t_cols[c] = terms.cols[c];
    if (tid < (td + 1) * (td + 1)) lag_sh[tid] = fe_load(lag + tid);
    if (tid == 0) { tr = *trp; sh_prev = fe_load(prev); }
    __syncthreads();
    int round = 0;
    for (size_t h = height; h > 1; h >>= 1, round++) {
        const size_t off = h >> 1;
        fe_acc a[W_MAX_TD];
#pragma unroll
        for (int k = 0; k < W_MAX_TD; k++) acc_zero(a[k]);
        for (size_t i = tid; i < off; i += nthreads) {
            fe row[WMAX], diff[WMAX];
#pragma unroll
            for (int j = 0; j < WMAX; j++) {
                if (j < width) {
                    fe x0 = fe_load(m + i * width + j), x1 = fe_load(m + (i + off) * width + j);
                    row[j] = x1;
                    diff[j] = fe_sub(x1, x0);
                }
            }
            fe d0 = fe_load(d + i), dd = fe_load(d + i + off);
            const fe ddiff = fe_sub(dd, d0);
#pragma unroll
            for (int k = 0; k < W_MAX_TD; k++) {
                if (k < td) {
                    fe comp = fe_zero();
                    for (int t = 0; t < terms.n_terms; t++) {
                        fe p = t_coef[t];
                        for (uint32_t c = 0; c < t_len[t]; c++) {
                            const uint32_t col = t_cols[t_off[t] + c];
                            fe x = row[0];
#pragma unroll
                            for (int j = 1; j < WMAX; j++) x = col == (uint32_t)j ? row[j] : x;  // select chain: keeps `row` in registers
                            p = fe_mul(p, x);
                        }
                        comp = fe_add(comp, p);
                    }
                    acc_mul_add(a[k], comp, dd);
                    if (k + 1 < td) {
#pragma unroll
                        for (int j = 0; j < WMAX; j++)
                            if (j < width) row[j] = fe_add(row[j], diff[j]);
                        dd = fe_add(dd, ddiff);
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < W_MAX_TD; k++) {
            if (k < td) {
                fe sk = block_sum(acc_reduce(a[k]), scratch);
                if (tid == 0) ev[k] = sk;
            }
        }
        __syncthreads();
        if (tid < 32) {
            const fe r = wchain_round_warp(ev, td, lag_sh, &sh_prev, &tr, coef_out + (size_t)round * td);
            if (tid == 0) { sh_r = r; fe_store(rs_out + round, r); }
        }
        __syncthreads();
        const fe r = sh_r;
        // fold (:234-247): rows i < off of the matrix and of delta
        const size_t total = off * (size_t)(width + 1);
        for (size_t e = tid; e < total; e += nthreads) {
            fe* base;
            size_t idx, hi;
            if (e < off * (size_t)width) { base = m; idx = e; hi = e + off * (size_t)width; }
            else { base = d; idx = e - off * (size_t)width; hi = idx + off; }
            fe x0 = fe_load(base + idx), x1 = fe_load(base + hi);
            fe_store(base + idx, fe_add(x0, fe_mul(r, fe_sub(x1, x0))));
        }
        __syncthreads();
    }
    if (tid == 0) { *trp = tr; fe_store(prev, sh_prev); }
}
int wchain_finish_launch(const fe* partials, int nb, int td, const fe* lag, fe* prev, DevTranscript* tr, fe* coef_out, fe* r_store, fe* r_dev,
                         cudaStream_t s) {
    ProfScope prof(PROF_TRANSCRIPT, 0.0, s);
    wchain_finish_kernel<<<1, 256, 0, s>>>(partials, nb, td, lag, prev, tr, coef_out, r_store, r_dev);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
int wchain_tail_launch(fe* m, fe* d, size_t height, int width, const WTerms& t, int td, const fe* lag, fe* prev, DevTranscript* tr, fe* coef_out,
                       fe* rs_out, cudaStream_t s) {
    ProfScope prof(PROF_TAIL, 0.0, s);
    if (width <= 4) wchain_tail_kernel<4><<<1, 512, 0, s>>>(m, d, height, width, t, td, lag, prev, tr, coef_out, rs_out);
    else wchain_tail_kernel<W_MAX_WIDTH><<<1, 512, 0, s>>>(m, d, height, width, t, td, lag, prev, tr, coef_out, rs_out);
    MLB_KERNEL_CHECK();
    return ML_OK;
}

int chain_challenge_launch(DevTranscript* tr, const uint8_t* absorb, int absorb_len, uint8_t* copy_out, fe* r_out, bool want_challenge,
                           cudaStream_t s) {
    ProfScope prof(PROF_TRANSCRIPT, 0.0, s);
    chain_challenge_kernel<<<1, 32, 0, s>>>(tr, absorb, absorb_len, copy_out, r_out, want_challenge ? 1 : 0);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
int chain_sumcheck_finish_launch(const fe* partials, int nb, fe* prev, DevTranscript* tr, const uint8_t* absorb, int absorb_len,
                                 uint8_t* copy_out, fe* sc_out, fe* r_out, cudaStream_t s) {
    ProfScope prof(PROF_TRANSCRIPT, 0.0, s);
    chain_sumcheck_finish_kernel<<<1, 256, 0, s>>>(partials, nb, prev, tr, absorb, absorb_len, copy_out, sc_out, r_out);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
int chain_tail_launch(const TailArgs& a, cudaStream_t s) {
    ProfScope prof(PROF_TAIL, 0.0, s);
    chain_tail_kernel<<<1, 1024, 0, s>>>(a);
    MLB_KERNEL_CHECK();
    return ML_OK;
}

}  // namespace mlb
