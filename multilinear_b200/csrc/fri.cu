// FRI folding (src/fri/mod.rs:79-114, src/fri/batched_fri.rs:101-150) as streaming kernels.
//
// Reference, per output i < n/2:  a = cur[i], b = cur[i + n/2],
//     next[i] = ((a + b) + r * ((a - b) * w_N0^(-i * 2^k))) * 2^-1
// with the inverse twiddle read from a 512 MiB gen_pows table as gen_pows[N0 - i*2^k] (:106-110).
// Here the twiddle comes from the two-level root tables already resident for the NTT (one extra multiply,
// no large-table gather), the challenge is pre-halved on the host (r/2), and the halving of (a + b) is a
// shift: 3 multiplies, 48 bytes of HBM traffic per output.  The large rounds use fri_fold_chunk_kernel, which folds the
// high-table factor of the twiddle and r/2 into one constant per 4096-exponent chunk: 2 multiplies per output.
#include "field.cuh"
#include "internal.h"

namespace mlb {

__device__ __forceinline__ fe root_pow(const fe* __restrict__ lo, const fe* __restrict__ hi, size_t e) {
    fe w = fe_load_nc(lo + (e & (((size_t)1 << LO_BITS) - 1)));
    if (e >> LO_BITS) w = fe_mul(w, fe_load_nc(hi + (e >> LO_BITS)));
    return w;
}

// next[i] = half(a + b) + (r/2) * ((a - b) * w^-(i << k))
__global__ void __launch_bounds__(256) fri_fold_kernel(const fe* __restrict__ cur, size_t half_n, fe* __restrict__ next, fe r_half,
                                                       const fe* __restrict__ r_dev, int k, int log_n0, const fe* __restrict__ lo,
                                                       const fe* __restrict__ hi) {
    if (r_dev) r_half = fe_load(r_dev + 1);  // {r, r/2} left in HBM by the transcript kernel
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t n0 = (size_t)1 << log_n0;
    for (; i < half_n; i += stride) {
        fe a = fe_load_nc(cur + i), b = fe_load_nc(cur + i + half_n);
        fe even = fe_half(fe_add(a, b));
        fe d = fe_sub(a, b);
        if (i != 0) d = fe_mul(d, root_pow(lo, hi, n0 - (i << k)));  // i = 0: gen_pows[0] = 1 (:92-95)
        fe_store(next + i, fe_add(even, fe_mul(r_half, d)));
    }
}

// Two multiplies per output.  With j = i << k:  w^-j = w^-(4096 c) * w^-x,  c = j >> 12, x = j & 4095, and
//   w^-(4096 c) = hi[H - c] (c > 0),   w^-x = lo[4096 - x] * hi[H - 1] (x > 0),   H = N0 / 4096,
// so  (r/2) * w^-j = C[c] * lo[(4096 - x) & 4095]  with one constant C per chunk c (times hi[H-1] when x > 0).
// A CTA owns FOLD_SPAN consecutive outputs = 2^k chunks; its first 2^k threads build the chunk constants in shared
// memory (2 multiplies each), then every output costs  t = (a - b) * lo[..]  and  C * t.
static const int FOLD_SPAN = 4096;
static const int FOLD_MAX_K = 8;  // 2^k chunk constants per CTA <= blockDim
__global__ void __launch_bounds__(256) fri_fold_chunk_kernel(const fe* __restrict__ cur, size_t half_n, fe* __restrict__ next, fe r_half,
                                                             const fe* __restrict__ r_dev, int k, int log_n0, const fe* __restrict__ lo,
                                                             const fe* __restrict__ hi) {
    __shared__ fe c0[1 << FOLD_MAX_K], c1[1 << FOLD_MAX_K];
    if (r_dev) r_half = fe_load(r_dev + 1);
    const int tid = threadIdx.x;
    const size_t i0 = (size_t)blockIdx.x * FOLD_SPAN;
    const int log_chunk = LO_BITS - k;  // outputs per chunk
    const size_t c_first = i0 >> log_chunk;
    const size_t H = (size_t)1 << (log_n0 - LO_BITS);
    if (tid < (1 << k)) {
        const size_t c = c_first + tid;  // c < H / 2 because j < N0 / 2
        fe base = c ? fe_mul(r_half, fe_load_nc(hi + (H - c))) : r_half;
        c0[tid] = base;
        c1[tid] = fe_mul(base, fe_load_nc(hi + (H - 1)));
    }
    __syncthreads();
    // half_n is a multiple of FOLD_SPAN (checked at launch), so there is no bounds test and the loads of four iterations
    // (8 independent 16-byte loads per thread) can be issued back to back
#pragma unroll 4
    for (int u = 0; u < FOLD_SPAN / 256; u++) {
        const size_t i = i0 + tid + 256 * u;
        fe a = fe_load_nc(cur + i), b = fe_load_nc(cur + i + half_n);
        fe even = fe_half(fe_add(a, b));
        const unsigned x = (unsigned)((i << k) & (((size_t)1 << LO_BITS) - 1));
        const int ci = (int)((i >> log_chunk) - c_first);
        fe t = fe_mul(fe_sub(a, b), fe_load_nc(lo + ((((unsigned)1 << LO_BITS) - x) & (((unsigned)1 << LO_BITS) - 1))));  // lo[0] = 1 when x = 0
        fe c = x ? c1[ci] : c0[ci];
        fe_store(next + i, fe_add(even, fe_mul(c, t)));
    }
}

static fe to_dev_fe(hfe x) {
    fe r;
    r.v[0] = (uint32_t)x; r.v[1] = (uint32_t)(x >> 32); r.v[2] = (uint32_t)(x >> 64); r.v[3] = (uint32_t)(x >> 96);
    return r;
}
static inline unsigned grid_for(size_t n, size_t cap = 148 * 16) {
    size_t b = (n + 255) / 256;
    if (b > cap) b = cap;
    if (b == 0) b = 1;
    return (unsigned)b;
}

int fri_fold_launch(Ctx* ctx, const fe* cur, size_t n_cur, fe* next, hfe r, const fe* r_dev, size_t k, int log_n0, cudaStream_t s) {
    const RootTables* rt;
    MLB_TRY(get_root_tables(ctx, log_n0, s, &rt));
    const size_t half_n = n_cur / 2;
    ProfScope prof(PROF_FRI_FOLD, 24.0 * (double)n_cur, s);  // read n elements, write n/2
    if ((int)k <= FOLD_MAX_K && log_n0 > LO_BITS && half_n >= (size_t)FOLD_SPAN && half_n % FOLD_SPAN == 0 && (half_n << k) <= ((size_t)1 << (log_n0 - 1)))
        fri_fold_chunk_kernel<<<(unsigned)((half_n + FOLD_SPAN - 1) / FOLD_SPAN), 256, 0, s>>>(cur, half_n, next, to_dev_fe(hfe_half(r)), r_dev, (int)k,
                                                                                                 log_n0, rt->lo, rt->hi);
    else
        fri_fold_kernel<<<grid_for(half_n), 256, 0, s>>>(cur, half_n, next, to_dev_fe(hfe_half(r)), r_dev, (int)k, log_n0, rt->lo, rt->hi);
    MLB_KERNEL_CHECK();
    return ML_OK;
}

// batched first fold (batched_fri.rs:124-150): a, b are Horner fingerprints over the batch, acc = acc*rho + c_j
__global__ void __launch_bounds__(256) fri_batched_fold_kernel(const fe* const* __restrict__ codes, int n_codes, size_t half_n,
                                                               fe* __restrict__ next, fe rho, fe r_half, const fe* __restrict__ r_dev,
                                                               int log_n0, const fe* __restrict__ lo, const fe* __restrict__ hi) {
    if (r_dev) r_half = fe_load(r_dev + 1);
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t n0 = (size_t)1 << log_n0;
    for (; i < half_n; i += stride) {
        fe a = fe_zero(), b = fe_zero();
        for (int j = 0; j < n_codes; j++) {
            const fe* c = codes[j];
            a = fe_add(fe_mul(a, rho), fe_load_nc(c + i));
            b = fe_add(fe_mul(b, rho), fe_load_nc(c + i + half_n));
        }
        fe even = fe_half(fe_add(a, b));
        fe d = fe_sub(a, b);
        if (i != 0) d = fe_mul(d, root_pow(lo, hi, n0 - i));
        fe_store(next + i, fe_add(even, fe_mul(r_half, d)));
    }
}
int fri_batched_fold_launch(Ctx* ctx, const fe* const* codes, size_t n_codes, size_t n, fe* next, hfe fingerprint_r, hfe r,
                            const fe* r_dev, int log_n0, cudaStream_t s) {
    const RootTables* rt;
    MLB_TRY(get_root_tables(ctx, log_n0, s, &rt));
    const size_t half_n = n / 2;
    ProfScope prof(PROF_FRI_FOLD, 16.0 * (double)n * (double)n_codes + 8.0 * (double)n, s);
    fri_batched_fold_kernel<<<grid_for(half_n), 256, 0, s>>>(codes, (int)n_codes, half_n, next, to_dev_fe(fingerprint_r),
                                                              to_dev_fe(hfe_half(r)), r_dev, log_n0, rt->lo, rt->hi);
    MLB_KERNEL_CHECK();
    return ML_OK;
}

// fingerprinted evaluation table (batched_pcs.rs:55-63): out[i] = Horner_rho(polys[0][i], ..., polys[B-1][i])
__global__ void __launch_bounds__(256) fingerprint_rows_kernel(const fe* const* __restrict__ polys, int n_polys, size_t n, fe rho,
                                                               const fe* __restrict__ rho_dev, fe* __restrict__ out) {
    if (rho_dev) rho = fe_load(rho_dev);
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        fe a = fe_zero();
        for (int j = 0; j < n_polys; j++) a = fe_add(fe_mul(a, rho), fe_load_nc(polys[j] + i));
        fe_store(out + i, a);
    }
}
int fingerprint_rows_launch(const fe* const* polys, size_t n_polys, size_t n, hfe r, fe* out, cudaStream_t s, const fe* r_dev) {
    fingerprint_rows_kernel<<<grid_for(n), 256, 0, s>>>(polys, (int)n_polys, n, to_dev_fe(r), r_dev, out);
    MLB_KERNEL_CHECK();
    return ML_OK;
}

}  // namespace mlb
