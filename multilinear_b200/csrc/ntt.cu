// NTT / INTT / Reed-Solomon encode over Field128 on sm_100a.
//
// Reference semantics (src/ntt/mod.rs:69-110, 132-173; src/fri/mod.rs:19-28): natural-order coefficients in,
// natural-order evaluations X[k] = sum_j x[j] * gen^(j*k) out.  The reference does bit-reverse + radix-2 DIT
// in place on one core; here the transform is a multi-pass ("four-step") decomposition sized for HBM + SMEM:
//
//   N = R_0 * R_1 * ... * R_{P-1},  each R_p <= 512 (P = 1 and R <= 4096 for small N)
//   pass p views the array as [A][R_p][B] (A = R_0..R_{p-1}, B = R_{p+1}..R_{P-1}) and one CTA owns a tile of
//   R_p x T elements (T contiguous columns, T*16 B >= 128 B coalesced runs, 64 KB of shared memory):
//     1. tile -> shared memory (the RS encoder reads only the n live coefficients; the zero half is implicit)
//     2. R_p-point DIF over the strided index, three radix-2 stages per round in registers, twiddles w_R^e from a
//        shared-memory copy of the small-root table (no multiplies spent on twiddle generation)
//     3. store un-bit-reversed, fused with the inter-pass twiddle w_N^(k*b*A) (two-level table, one extra multiply);
//        the last pass instead writes natural order k = k_0 + R_0*k_1 + ... in T-element runs.
//   The bit-reversal permutations of the reference never touch HBM; index math is checked by tools/ntt_model.py.
#include <cstdlib>
#include "field.cuh"
#include "internal.h"

namespace mlb {

static const int NTT_THREADS = 256;
static const int TILE_LOG = 12;  // 4096 elements = 64 KB per CTA

struct PassArgs {
    const fe* in;
    fe* out;
    const fe* small;  // w_4096^(+-i), i < 2048
    const fe* lo;     // inter-pass twiddle tables of the domain (lo may be the 1/N-scaled copy)
    const fe* hi;
    const fe* wtab;   // optional precomputed inter-pass twiddle matrix [k*B + b] (saves the table-combine multiply)
    fe scale;         // single-pass inverse: 1/N
    int log_n, log_r, log_t, log_a, log_b;
    int last, inverse, zero_padded, scaled_lo, has_scale;
    int bitrev_in;    // pass 0 of a zero-padded transform: input element j is read from in[rev_{log_n-1}(j)]
    int n_passes;
    int radix_log[4];
};

// LAST: this round contains the final stages of the tile, where l == 0 for every item, so the twiddle exponent
// depends on the unrolled j only and the trivial multiplies (w^0) vanish at compile time.  Other rounds multiply
// unconditionally (tw[0] = 1): a data-dependent skip would put every butterfly in its own basic block and stop
// the scheduler from interleaving the twelve independent multiply chains of an item.
template <int NS, bool LAST>
__device__ __forceinline__ void dif_round(fe* data, const fe* tw, int pitch, int log_r, int log_t, int q, int tid) {
    // stages q .. q+NS-1 of the R-point DIF; an item is the 2^NS elements m = blk*(R>>q) + j*(R>>(q+NS)) + l of column t
    const int log_lr = LAST ? 0 : log_r - q - NS;  // l range = R >> (q+NS)
    const int items = 1 << (log_r + log_t - NS);
    for (int w = tid; w < items; w += NTT_THREADS) {
        const int t = w & ((1 << log_t) - 1);
        const int rest = w >> log_t;
        const int l = LAST ? 0 : (rest & ((1 << log_lr) - 1));
        const int blk = rest >> log_lr;
        const int m0 = (blk << (log_r - q)) + l;
        fe x[1 << NS];
#pragma unroll
        for (int j = 0; j < (1 << NS); j++) x[j] = data[(m0 + (j << log_lr)) * pitch + t];
#pragma unroll
        for (int u = 0; u < NS; u++) {
            const int span = 1 << (NS - 1 - u);
#pragma unroll
            for (int j = 0; j < (1 << NS); j++) {
                if (j & span) continue;
                fe a = x[j], b = x[j + span];
                x[j] = fe_add(a, b);
                fe d = fe_sub(a, b);
                if (LAST) {
                    if ((j & (span - 1)) != 0) d = fe_mul(d, tw[(j & (span - 1)) << (q + u)]);  // compile-time skip of w^0
                } else {
                    const int e = (((j & (span - 1)) << log_lr) + l) << (q + u);
                    d = fe_mul(d, tw[e]);
                }
                x[j + span] = d;
            }
        }
#pragma unroll
        for (int j = 0; j < (1 << NS); j++) data[(m0 + (j << log_lr)) * pitch + t] = x[j];
    }
}

__global__ void __launch_bounds__(NTT_THREADS, 3) ntt_pass_kernel(PassArgs p) {
    extern __shared__ uint4 smem_raw[];
    fe* data = reinterpret_cast<fe*>(smem_raw);
    const int R = 1 << p.log_r, T = 1 << p.log_t;
    // the row padding only matters where lanes run along m (the last pass's contiguous-row load)
    const int pitch = (p.last && T > 1) ? T + 1 : T;
    fe* tw = data + (size_t)R * pitch;
    const int tid = threadIdx.x;
    const size_t tile = blockIdx.x;

    for (int i = tid; i < (R >> 1); i += NTT_THREADS) tw[i] = fe_load_nc(p.small + ((size_t)i << (12 - p.log_r)));
    if (tid == 0 && R == 1) tw[0] = fe_one();

    // ---- tile coordinates
    size_t a = 0, bt = 0, ap = 0, k0_base = 0;
    const int log_rb = p.log_r + p.log_b;
    if (!p.last) {
        const int log_tiles_b = p.log_b - p.log_t;
        bt = tile & (((size_t)1 << log_tiles_b) - 1);
        a = tile >> log_tiles_b;
    } else if (p.n_passes > 1) {
        const int log_k0_tiles = p.radix_log[0] - p.log_t;
        k0_base = (tile & (((size_t)1 << log_k0_tiles) - 1)) << p.log_t;
        ap = tile >> log_k0_tiles;
    }
    const int log_a_rest = p.log_a - (p.n_passes > 1 ? p.radix_log[0] : 0);  // log2(A / R_0)

    // ---- load
    const int tile_elems = R * T;
    if (!p.last && p.bitrev_in) {
        // PCS encode (multilinear_pcs.rs:101-107): x[j] = c[rev_v(j)], j = m*B + b  ->  c[(rev(b) << (log_r-1)) | rev(m)].
        // For a fixed column b the R/2 live rows are one contiguous 4 KB block of c, so the permutation costs nothing in HBM.
        const int half_log = p.log_r - 1, half = R >> 1;
        for (int idx = tid; idx < half * T; idx += NTT_THREADS) {
            const int t = idx >> half_log, mp = idx & (half - 1);
            const size_t b = (bt << p.log_t) + t;
            const size_t rb = p.log_b ? (size_t)(__brevll((unsigned long long)b) >> (64 - p.log_b)) : 0;
            const int m = half_log ? (int)(__brev((unsigned)mp) >> (32 - half_log)) : 0;
            data[m * pitch + t] = fe_load_nc(p.in + (rb << half_log) + mp);
            data[(m + half) * pitch + t] = fe_zero();
        }
    } else if (!p.last) {
        const size_t base = (a << log_rb) + (bt << p.log_t);
#pragma unroll 8
        for (int idx = tid; idx < tile_elems; idx += NTT_THREADS) {
            const int t = idx & (T - 1), m = idx >> p.log_t;
            fe v;
            if (p.zero_padded && m >= (R >> 1)) v = fe_zero();
            else v = fe_load_nc(p.in + base + ((size_t)m << p.log_b) + t);
            data[m * pitch + t] = v;
        }
    } else {
#pragma unroll 8
        for (int idx = tid; idx < tile_elems; idx += NTT_THREADS) {
            const int m = idx & (R - 1), t = idx >> p.log_r;
            const size_t arow = (((k0_base + t) << log_a_rest) + ap);
            fe v;
            if (p.zero_padded && m >= (R >> 1)) v = fe_zero();  // only when the whole transform is one pass
            else v = fe_load_nc(p.in + (arow << p.log_r) + m);
            data[m * pitch + t] = v;
        }
    }
    __syncthreads();

    // ---- R-point DIF, three stages per round
    // the partial round (log_r mod 3 stages) goes first so that the last round is always a full radix-8 one
    for (int q = 0; q < p.log_r;) {
        const int rem = p.log_r - q;
        const int ns = rem % 3 ? rem % 3 : 3;
        const bool last = rem == ns;
        if (ns == 3) { if (last) dif_round<3, true>(data, tw, pitch, p.log_r, p.log_t, q, tid); else dif_round<3, false>(data, tw, pitch, p.log_r, p.log_t, q, tid); }
        else if (ns == 2) { if (last) dif_round<2, true>(data, tw, pitch, p.log_r, p.log_t, q, tid); else dif_round<2, false>(data, tw, pitch, p.log_r, p.log_t, q, tid); }
        else { if (last) dif_round<1, true>(data, tw, pitch, p.log_r, p.log_t, q, tid); else dif_round<1, false>(data, tw, pitch, p.log_r, p.log_t, q, tid); }
        q += ns;
        __syncthreads();
    }

    // ---- store (un-bit-reverse; inter-pass twiddle or natural-order scatter)
    if (!p.last) {
        const size_t base = (a << log_rb) + (bt << p.log_t);
        const size_t nmask = ((size_t)1 << p.log_n) - 1;
#pragma unroll 4
        for (int idx = tid; idx < tile_elems; idx += NTT_THREADS) {
            const int t = idx & (T - 1), pos = idx >> p.log_t;
            const size_t k = __brev((unsigned)pos) >> (32 - p.log_r);
            const size_t b = (bt << p.log_t) + t;
            fe v = data[pos * pitch + t];
            if (p.wtab) {
                v = fe_mul(v, fe_load_nc(p.wtab + (k << p.log_b) + b));
            } else {
                size_t e = (k * b) << p.log_a;
                if (p.inverse) e = (((size_t)1 << p.log_n) - e) & nmask;
                if (e != 0 || p.scaled_lo) {
                    fe w = fe_load_nc(p.lo + (e & (((size_t)1 << LO_BITS) - 1)));
                    if (e >> LO_BITS) w = fe_mul(w, fe_load_nc(p.hi + (e >> LO_BITS)));
                    v = fe_mul(v, w);
                }
            }
            fe_store(p.out + base + (k << p.log_b) + t, v);
        }
    } else {
        // a' digits k_1..k_{P-2} (k_1 most significant) -> mid = k_1 + R_1*k_2 + ...
        size_t mid = 0;
        {
            int shift_out = 0, rem = log_a_rest;
            for (int d = 1; d < p.n_passes - 1; d++) {
                rem -= p.radix_log[d];
                const size_t kd = (ap >> rem) & (((size_t)1 << p.radix_log[d]) - 1);
                mid |= kd << shift_out;
                shift_out += p.radix_log[d];
            }
        }
        const int log_r0 = p.n_passes > 1 ? p.radix_log[0] : 0;
#pragma unroll 4
        for (int idx = tid; idx < tile_elems; idx += NTT_THREADS) {
            const int t = idx & (T - 1), pos = idx >> p.log_t;
            const size_t k = p.log_r ? (__brev((unsigned)pos) >> (32 - p.log_r)) : 0;
            fe v = data[pos * pitch + t];
            if (p.has_scale) v = fe_mul(v, p.scale);
            fe_store(p.out + (k0_base + t) + (mid << log_r0) + (k << p.log_a), v);
        }
    }
}

// ------------------------------------------------------------------ root tables
__global__ void root_tables_kernel(fe* lo, fe* hi, fe* lo_ninv, fe gen, fe gen_hi, fe ninv, unsigned n_lo, unsigned n_hi) {
    unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_lo) {
        fe w = fe_pow_u64(gen, i);
        fe_store(lo + i, w);
        fe_store(lo_ninv + i, fe_mul(w, ninv));
    }
    if (i < n_hi) fe_store(hi + i, fe_pow_u64(gen_hi, i));
}
__global__ void small_roots_kernel(fe* fwd, fe* inv, fe w, fe winv) {
    unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 2048) {
        fe_store(fwd + i, fe_pow_u64(w, i));
        fe_store(inv + i, fe_pow_u64(winv, i));
    }
}
// inter-pass twiddle matrix: out[k*B + b] = w_N^(+-(k*b) << log_a) (lo may be the 1/N-scaled table)
__global__ void pass_table_kernel(fe* out, const fe* lo, const fe* hi, int log_n, int log_a, int log_b, int inverse, size_t count) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t nmask = ((size_t)1 << log_n) - 1;
    for (; i < count; i += stride) {
        const size_t k = i >> log_b, b = i & (((size_t)1 << log_b) - 1);
        size_t e = (k * b) << log_a;
        if (inverse) e = (((size_t)1 << log_n) - e) & nmask;
        fe w = fe_load_nc(lo + (e & (((size_t)1 << LO_BITS) - 1)));
        if (e >> LO_BITS) w = fe_mul(w, fe_load_nc(hi + (e >> LO_BITS)));
        fe_store(out + i, w);
    }
}

// pow_2_generator_powers (src/ntt/mod.rs:18-28): out[i] = hi[i >> LO_BITS] * lo[i & mask]
__global__ void powers_kernel(fe* out, const fe* lo, const fe* hi, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        fe w = fe_load_nc(lo + (i & (((size_t)1 << LO_BITS) - 1)));
        if (i >> LO_BITS) w = fe_mul(w, fe_load_nc(hi + (i >> LO_BITS)));
        fe_store(out + i, w);
    }
}

static fe to_dev_fe(hfe x) {
    fe r;
    r.v[0] = (uint32_t)x; r.v[1] = (uint32_t)(x >> 32); r.v[2] = (uint32_t)(x >> 64); r.v[3] = (uint32_t)(x >> 96);
    return r;
}

int get_root_tables(Ctx* ctx, int log_n, cudaStream_t s, const RootTables** out) {
    std::lock_guard<std::mutex> lock(ctx->roots_mu);
    if (!ctx->small_fwd) {
        hfe w;
        hfe_pow2_generator(12, &w);
        MLB_CUDA(cudaMalloc((void**)&ctx->small_fwd, 2048 * 16));
        MLB_CUDA(cudaMalloc((void**)&ctx->small_inv, 2048 * 16));
        small_roots_kernel<<<8, 256, 0, s>>>(ctx->small_fwd, ctx->small_inv, to_dev_fe(w), to_dev_fe(hfe_inv(w)));
        MLB_KERNEL_CHECK();
        MLB_CUDA(cudaStreamSynchronize(s));  // tables are shared by every stream afterwards
    }
    auto it = ctx->roots.find(log_n);
    if (it == ctx->roots.end()) {
        RootTables rt;
        rt.log_n = log_n;
        if (!hfe_pow2_generator((uint64_t)log_n, &rt.gen)) { set_error("no 2^%d-th root of unity", log_n); return ML_ERR_OUT_OF_RANGE; }
        const size_t n = (size_t)1 << log_n;
        const unsigned n_lo = (unsigned)(n < ((size_t)1 << LO_BITS) ? n : ((size_t)1 << LO_BITS));
        const unsigned n_hi = (unsigned)(n >> LO_BITS ? n >> LO_BITS : 1);
        if (cudaMalloc((void**)&rt.lo, (size_t)n_lo * 16) != cudaSuccess || cudaMalloc((void**)&rt.lo_ninv, (size_t)n_lo * 16) != cudaSuccess ||
            cudaMalloc((void**)&rt.hi, (size_t)n_hi * 16) != cudaSuccess) {
            cudaGetLastError();
            cudaFree(rt.lo); cudaFree(rt.lo_ninv); cudaFree(rt.hi);  // cudaFree(nullptr) is a no-op
            set_error("root tables for 2^%d: device allocation failed", log_n);
            return ML_ERR_ALLOC;
        }
        hfe gen_hi = hfe_pow(rt.gen, (hfe)1 << LO_BITS);
        hfe ninv = hfe_inv(hfe_new((hfe)n));
        unsigned m = n_lo > n_hi ? n_lo : n_hi;
        root_tables_kernel<<<(m + 255) / 256, 256, 0, s>>>(rt.lo, rt.hi, rt.lo_ninv, to_dev_fe(rt.gen), to_dev_fe(gen_hi), to_dev_fe(ninv), n_lo, n_hi);
        MLB_KERNEL_CHECK();
        MLB_CUDA(cudaStreamSynchronize(s));
        it = ctx->roots.emplace(log_n, rt).first;
    }
    *out = &it->second;
    return ML_OK;
}

// lazily built, cached per (size, direction, pass); skipped (nullptr) above 1 GiB per table
static int get_pass_table(Ctx* ctx, int log_n, bool inverse, int pass, int log_a, int log_r, int log_b, cudaStream_t s, const fe** out) {
    *out = nullptr;
    const size_t count = (size_t)1 << (log_r + log_b);
    if (count * 16 > ((size_t)1 << 30)) return ML_OK;
    // MLB_NTT_NO_WTAB: experiment switch — inter-pass twiddles from the two-level root tables (one more multiply per element and
    // pass, no N-entry matrix read from HBM); measured in profiles/r2_ntt_variants.txt
    static const bool no_wtab = getenv("MLB_NTT_NO_WTAB") != nullptr;
    if (no_wtab) return ML_OK;
    std::lock_guard<std::mutex> lock(ctx->roots_mu);
    RootTables& rt = ctx->roots[log_n];  // exists: get_root_tables ran first
    fe*& slot = rt.pass_tw[inverse ? 1 : 0][pass];
    if (!slot) {
        fe* tab;
        if (cudaMalloc((void**)&tab, count * 16) != cudaSuccess) { cudaGetLastError(); return ML_OK; }  // fall back to the two-level path
        size_t blocks = (count + 255) / 256;
        if (blocks > (size_t)ctx->sm_count * 16) blocks = (size_t)ctx->sm_count * 16;
        const fe* lo = (inverse && pass == 0) ? rt.lo_ninv : rt.lo;
        pass_table_kernel<<<(unsigned)blocks, 256, 0, s>>>(tab, lo, rt.hi, log_n, log_a, log_b, inverse ? 1 : 0, count);
        MLB_KERNEL_CHECK();
        MLB_CUDA(cudaStreamSynchronize(s));
        slot = tab;
    }
    *out = slot;
    return ML_OK;
}

int powers_launch(Ctx* ctx, int log_n, fe* out, cudaStream_t s) {
    const RootTables* rt;
    MLB_TRY(get_root_tables(ctx, log_n, s, &rt));
    const size_t n = (size_t)1 << log_n;
    size_t blocks = (n + 255) / 256;
    if (blocks > (size_t)ctx->sm_count * 16) blocks = (size_t)ctx->sm_count * 16;
    powers_kernel<<<(unsigned)blocks, 256, 0, s>>>(out, rt->lo, rt->hi, n);
    MLB_KERNEL_CHECK();
    return ML_OK;
}

// Natural-order NTT of size 2^log_n with the domain generator pow_2_generator(log_n) (or its inverse, with the
// 1/N scaling of intt).  rs_zero_padded: `in` holds N/2 coefficients, the upper half of the input is zero
// (reed_solomon's resize, src/fri/mod.rs:24).  in == out is allowed for P == 1 only when not zero padded.
int ntt_launch(Ctx* ctx, const fe* in, fe* out, int log_n, bool inverse, bool rs_zero_padded, cudaStream_t s, bool bitrev_in, fe* tmp_in) {
    if (bitrev_in && !(rs_zero_padded && !inverse && log_n > TILE_LOG)) { set_error("ntt: bit-reversed input needs a multi-pass RS encode"); return ML_ERR_ARG; }
    MLB_CUDA(cudaFuncSetAttribute(ntt_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
    const RootTables* rt;
    MLB_TRY(get_root_tables(ctx, log_n, s, &rt));
    if (log_n == 0) {
        if (in != out) MLB_CUDA(cudaMemcpyAsync(out, in, 16, cudaMemcpyDeviceToDevice, s));
        return ML_OK;
    }
    int n_passes = log_n <= TILE_LOG ? 1 : (log_n + 8) / 9;
    int radix_log[4] = {0, 0, 0, 0};
    if (n_passes > 4) { set_error("NTT size 2^%d not supported", log_n); return ML_ERR_ARG; }
    for (int p = 0; p < n_passes; p++) radix_log[p] = log_n / n_passes + (p < log_n % n_passes ? 1 : 0);

    // passes 0..P-2 are tile-in-place and run in a scratch buffer; the last pass scatters to natural order in `out`
    struct TmpGuard {  // stream-ordered scratch released on every exit path
        fe* p = nullptr;
        cudaStream_t s;
        explicit TmpGuard(cudaStream_t st) : s(st) {}
        ~TmpGuard() { if (p) cudaFreeAsync(p, s); }
    } tmp_guard(s);
    if (n_passes > 1 && !tmp_in) MLB_TRY(dev_alloc_async((void**)&tmp_guard.p, ((size_t)16) << log_n, s));
    fe* const tmp = tmp_in ? tmp_in : tmp_guard.p;

    const double nbytes = 16.0 * (double)((size_t)1 << log_n);
    ProfScope prof(PROF_NTT_PASS, rs_zero_padded ? 1.5 * nbytes : 2.0 * nbytes, s);  // read input once + write output once
    PassArgs a;
    memset(&a, 0, sizeof a);
    a.small = inverse ? ctx->small_inv : ctx->small_fwd;
    a.hi = rt->hi;
    a.log_n = log_n;
    a.inverse = inverse ? 1 : 0;
    a.n_passes = n_passes;
    for (int p = 0; p < 4; p++) a.radix_log[p] = radix_log[p];
    int log_a = 0;
    for (int p = 0; p < n_passes; p++) {
        a.last = p == n_passes - 1;
        a.in = p == 0 ? in : tmp;
        a.out = a.last ? out : tmp;
        a.log_r = radix_log[p];
        a.log_a = log_a;
        a.log_b = log_n - log_a - a.log_r;
        a.log_t = n_passes == 1 ? 0 : TILE_LOG - a.log_r;
        a.zero_padded = (rs_zero_padded && p == 0) ? 1 : 0;
        a.bitrev_in = (bitrev_in && p == 0) ? 1 : 0;
        a.scaled_lo = (inverse && p == 0 && n_passes > 1) ? 1 : 0;
        a.lo = a.scaled_lo ? rt->lo_ninv : rt->lo;
        a.wtab = nullptr;
        if (!a.last) MLB_TRY(get_pass_table(ctx, log_n, inverse, p, a.log_a, a.log_r, a.log_b, s, &a.wtab));
        a.has_scale = (inverse && n_passes == 1) ? 1 : 0;
        if (a.has_scale) a.scale = to_dev_fe(hfe_inv(hfe_new((hfe)1 << log_n)));
        const int R = 1 << a.log_r, T = 1 << a.log_t;
        const int pitch = (a.last && T > 1) ? T + 1 : T;
        const size_t smem = ((size_t)R * pitch + (R >> 1) + 1) * 16;
        const size_t tiles = ((size_t)1 << log_n) >> (a.log_r + a.log_t);
        ntt_pass_kernel<<<(unsigned)tiles, NTT_THREADS, smem, s>>>(a);
        MLB_KERNEL_CHECK();
        log_a += a.log_r;
    }
    return ML_OK;
}

// every table a forward transform of 2^log_n reads (root, small and inter-pass tables), built now so that later launches of
// that size only read them: a prove plan calls this at creation, and its enqueue path then never synchronises or allocates
int ntt_prepare(Ctx* ctx, int log_n, cudaStream_t s) {
    const RootTables* rt;
    MLB_TRY(get_root_tables(ctx, log_n, s, &rt));
    const int n_passes = log_n <= TILE_LOG ? 1 : (log_n + 8) / 9;
    if (n_passes > 4) { set_error("NTT size 2^%d not supported", log_n); return ML_ERR_ARG; }
    int log_a = 0;
    for (int p = 0; p + 1 < n_passes; p++) {
        const int log_r = log_n / n_passes + (p < log_n % n_passes ? 1 : 0);
        const fe* tab;
        MLB_TRY(get_pass_table(ctx, log_n, false, p, log_a, log_r, log_n - log_a - log_r, s, &tab));
        log_a += log_r;
    }
    return ML_OK;
}

// bit_reverse_permutation (src/ntt/mod.rs:113-123) on 16-byte elements; uses trailing_zeros(n) bits like the reference
__global__ void bit_reverse_kernel(const uint4* in, uint4* out, size_t n, int bits) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        // the reference swaps i <-> rev(i mod 2^bits) only for i < 2^bits; any tail beyond 2^bits stays put
        size_t j = (bits && (i >> bits) == 0) ? (size_t)(__brevll((unsigned long long)i) >> (64 - bits)) : i;
        out[i] = in[j];
    }
}
int bit_reverse_launch(const void* in, void* out, size_t n, size_t elem_bytes, cudaStream_t s) {
    if (elem_bytes != 16) { set_error("bit_reverse: device path handles 16-byte elements"); return ML_ERR_ARG; }
    if (n == 0) return ML_OK;
    int bits = __builtin_ctzll((unsigned long long)n);
    size_t blocks = (n + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    ProfScope prof(PROF_BITREV, 32.0 * (double)n, s);
    bit_reverse_kernel<<<(unsigned)blocks, 256, 0, s>>>((const uint4*)in, (uint4*)out, n, bits);
    MLB_KERNEL_CHECK();
    return ML_OK;
}

}  // namespace mlb
