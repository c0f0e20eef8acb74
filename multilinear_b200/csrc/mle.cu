// Multilinear-polynomial kernels (src/polynomials.rs:110-188, src/constraint_system/evaluation.rs:56-73,
// src/constraint_system/sumcheck.rs:133-138).
//
//  - Moebius transform evals <-> coeffs (:111-124, :150-163): c[j] -= c[j ^ 2^i] for every set bit i.  The reference
//    makes v full passes over memory; here bits are grouped so a 4096-element tile does up to 12 bit-levels in
//    shared memory per HBM round trip (2-3 passes at v = 24).
//  - eq table (Mask::evaluate over every index, O(n v) multiplies in the reference): built as the outer product
//    EH[idx >> lb] * EL[idx & mask] of two small tables, one multiply per entry.
//  - evaluate(args) (O(n v) in the reference): dot product of the table with the same separable weights, inner
//    sums accumulated unreduced.
#include "field.cuh"
#include "internal.h"
#include "reduce.cuh"

namespace mlb {

static const int MLE_THREADS = 256;

// Shared-memory slot of element m of a single-column tile (T = 1): 16-byte chunks XOR-swizzled inside each 128-byte line by the
// line index (the SWIZZLE_128B pattern).  The last round of such a tile walks m = 8*lane + j, i.e. all lanes of a quarter-warp in
// the same four banks (ncu: 28 M bank conflicts of 48 M wavefronts in the first pass); swizzled, the eight lanes land in eight
// different bank groups, while consecutive-m accesses stay conflict-free (a permutation inside one line).
__device__ __forceinline__ int mobius_swz(int m) { return m ^ ((m >> 3) & 7); }

template <int NS, bool SUB, int NT = MLE_THREADS, bool SWZ = false>
__device__ __forceinline__ void mobius_round(fe* data, int pitch, int log_r, int log_t, int q, int tid) {
    // bit-levels q .. q+NS-1 (counted from the top of the tile's R index), same item layout as the NTT rounds
    const int log_lr = log_r - q - NS;
    const int items = 1 << (log_r + log_t - NS);
    for (int w = tid; w < items; w += NT) {
        const int t = w & ((1 << log_t) - 1);
        const int rest = w >> log_t;
        const int l = rest & ((1 << log_lr) - 1);
        const int blk = rest >> log_lr;
        const int m0 = (blk << (log_r - q)) + l;
        fe x[1 << NS];
#pragma unroll
        for (int j = 0; j < (1 << NS); j++) x[j] = SWZ ? data[mobius_swz(m0 + (j << log_lr))] : data[(m0 + (j << log_lr)) * pitch + t];
#pragma unroll
        for (int u = 0; u < NS; u++) {
            const int span = 1 << (NS - 1 - u);
#pragma unroll
            for (int j = 0; j < (1 << NS); j++) {
                if (j & span) continue;
                x[j + span] = SUB ? fe_sub(x[j + span], x[j]) : fe_add(x[j + span], x[j]);
            }
        }
#pragma unroll
        for (int j = 0; j < (1 << NS); j++) {
            if (SWZ) data[mobius_swz(m0 + (j << log_lr))] = x[j];
            else data[(m0 + (j << log_lr)) * pitch + t] = x[j];
        }
    }
}

// tile = all 2^log_r values of index bits [bit_lo, bit_lo + log_r) x 2^log_t contiguous low indices
template <bool SUB, bool SWZ>
__global__ void __launch_bounds__(MLE_THREADS, 2) mobius_pass_kernel(const fe* __restrict__ in, fe* __restrict__ out, int log_r, int log_t,
                                                                     int bit_lo) {
    extern __shared__ uint4 smem_raw[];
    fe* data = reinterpret_cast<fe*>(smem_raw);
    const int R = 1 << log_r, T = 1 << log_t;
    const int pitch = T > 1 ? T + 1 : 1;
    const int tid = threadIdx.x;
    const size_t tile = blockIdx.x;
    // tile -> (hi part above the handled bits, low-run index)
    const int log_runs = bit_lo - log_t;  // number of T-runs below bit_lo
    const size_t run = tile & (((size_t)1 << log_runs) - 1);
    const size_t hi = tile >> log_runs;
    const size_t base = (hi << (bit_lo + log_r)) + (run << log_t);
    const int tile_elems = R * T;
    // unrolled so that 8 independent 16-byte loads per thread are in flight (2 CTAs/SM cannot hide HBM latency otherwise)
#pragma unroll 8
    for (int idx = tid; idx < tile_elems; idx += MLE_THREADS) {
        const int t = idx & (T - 1), m = idx >> log_t;
        data[SWZ ? mobius_swz(m) : m * pitch + t] = fe_load_nc(in + base + ((size_t)m << bit_lo) + t);
    }
    __syncthreads();
    // the order of bit-levels is irrelevant (the per-bit updates commute)
    for (int q = 0; q < log_r;) {
        const int ns = log_r - q >= 3 ? 3 : log_r - q;
        if (ns == 3) mobius_round<3, SUB, MLE_THREADS, SWZ>(data, pitch, log_r, log_t, q, tid);
        else if (ns == 2) mobius_round<2, SUB, MLE_THREADS, SWZ>(data, pitch, log_r, log_t, q, tid);
        else mobius_round<1, SUB, MLE_THREADS, SWZ>(data, pitch, log_r, log_t, q, tid);
        q += ns;
        __syncthreads();
    }
#pragma unroll 8
    for (int idx = tid; idx < tile_elems; idx += MLE_THREADS) {
        const int t = idx & (T - 1), m = idx >> log_t;
        fe_store(out + base + ((size_t)m << bit_lo) + t, data[SWZ ? mobius_swz(m) : m * pitch + t]);
    }
}

// Measured and dropped (profiles/r1_mobius_notes.txt): a persistent one-CTA-per-SM variant with a three-stage shared-memory ring
// fed by cp.async.bulk + mbarrier and drained by bulk stores.  It was correct but slower (0.514 ms vs 0.443 ms at 2^24): the
// column passes need one bulk copy per 256 B - 1 KB row run, issued by one warp while the others wait at the barrier, and the
// first pass was limited by shared-memory bank conflicts, not by load/compute/store serialisation.  The XOR swizzle above is
// what moved the number (0.443 -> 0.349 ms).
int mobius_launch(const fe* in, fe* out, size_t len, bool subtract, cudaStream_t s) {
    if (len == 0) return ML_OK;
    // the reference transforms only the first 2^trailing_zeros(len) entries (polynomials.rs:151-155)
    const int n = __builtin_ctzll((unsigned long long)len);
    const size_t span = (size_t)1 << n;
    if (in != out && len > span) MLB_CUDA(cudaMemcpyAsync(out + span, in + span, (len - span) * 16, cudaMemcpyDeviceToDevice, s));
    if (n == 0) {
        if (in != out) MLB_CUDA(cudaMemcpyAsync(out, in, 16, cudaMemcpyDeviceToDevice, s));
        return ML_OK;
    }
    MLB_CUDA(cudaFuncSetAttribute(mobius_pass_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
    MLB_CUDA(cudaFuncSetAttribute(mobius_pass_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
    MLB_CUDA(cudaFuncSetAttribute(mobius_pass_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
    MLB_CUDA(cudaFuncSetAttribute(mobius_pass_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
    ProfScope prof(PROF_MOBIUS, 32.0 * (double)span, s);
    int bit_lo = 0;
    const fe* src = in;
    // first pass: low min(n,12) bits, contiguous tiles; then groups of <= 8 bits with T = 4096 >> bits columns
    // later passes take 8 bits each (runs of >= 16 elements = 256 B per row).  Measured alternative: 10 bits with 64-byte runs
    // saves a pass at v = 22 but that pass runs at half the bandwidth, no net gain (tools/mobius_bench.py)
    int rem_passes = n > 12 ? (n - 12 + 7) / 8 : 0;
    int done_first = 0;
    while (bit_lo < n) {
        int log_r, log_t;
        if (!done_first) {
            log_r = n < 12 ? n : 12;
            log_t = 0;
            done_first = 1;
        } else {
            int rem = n - bit_lo;
            log_r = (rem + rem_passes - 1) / rem_passes;
            rem_passes--;
            log_t = 12 - log_r;
        }
        const int R = 1 << log_r, T = 1 << log_t;
        const int pitch = T > 1 ? T + 1 : 1;
        const size_t smem = (size_t)R * pitch * 16;
        const size_t tiles = span >> (log_r + log_t);
        if (log_t == 0 && log_r >= 6) {  // single-column tile: swizzled shared-memory layout
            if (subtract) mobius_pass_kernel<true, true><<<(unsigned)tiles, MLE_THREADS, smem, s>>>(src, out, log_r, log_t, bit_lo);
            else mobius_pass_kernel<false, true><<<(unsigned)tiles, MLE_THREADS, smem, s>>>(src, out, log_r, log_t, bit_lo);
        } else if (subtract) mobius_pass_kernel<true, false><<<(unsigned)tiles, MLE_THREADS, smem, s>>>(src, out, log_r, log_t, bit_lo);
        else mobius_pass_kernel<false, false><<<(unsigned)tiles, MLE_THREADS, smem, s>>>(src, out, log_r, log_t, bit_lo);
        MLB_KERNEL_CHECK();
        src = out;
        bit_lo += log_r;
    }
    return ML_OK;
}

// ---------------------------------------------------------------- separable weight tables
// mode 0: eq weights     w(idx) = prod_i (bit_i ? p_i : 1 - p_i)   (Mask::evaluate, evaluation.rs:56-73)
// mode 1: monomial       w(idx) = prod_i (bit_i ? p_i : 1)         (MultilinearPolynomial::evaluate, polynomials.rs:133-145)
// p_i for bit i of the *global* index is points[n_vars - 1 - i] (big-endian convention); this table covers
// bits [bit0, bit0 + nbits).
__global__ void weight_table_kernel(const fe* __restrict__ points, int n_vars, int bit0, int nbits, int mode, fe* __restrict__ out) {
    const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (1u << nbits)) return;
    fe acc = fe_one();
    for (int i = 0; i < nbits; i++) {
        fe p = fe_load_nc(points + (n_vars - 1 - (bit0 + i)));
        if ((idx >> i) & 1u) acc = fe_mul(acc, p);
        else if (mode == 0) acc = fe_mul(acc, fe_sub(fe_one(), p));
    }
    fe_store(out + idx, acc);
}
// mode 2: geometric  out[i] = x^(i << shift)
__global__ void power_table_kernel(fe x, int shift, unsigned count, fe* __restrict__ out) {
    const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= count) return;
    fe_store(out + idx, fe_pow_u64(x, (unsigned long long)idx << shift));
}
__global__ void __launch_bounds__(256) outer_product_kernel(const fe* __restrict__ wh, const fe* __restrict__ wl, int lb, size_t n,
                                                            fe* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) fe_store(out + i, fe_mul(fe_load_nc(wh + (i >> lb)), fe_load_nc(wl + (i & (((size_t)1 << lb) - 1)))));
}
// partials[blockIdx] = sum over this CTA's rows hi of WH[hi] * (sum_lo data[hi << lb | lo] * WL[lo]), positions >= len skipped
__global__ void __launch_bounds__(256) sepdot_kernel(const fe* __restrict__ data, size_t len, const fe* __restrict__ wh,
                                                     const fe* __restrict__ wl, int lb, size_t rows, fe* __restrict__ partials) {
    __shared__ fe scratch[32];
    fe total = fe_zero();
    for (size_t hi = blockIdx.x; hi < rows; hi += gridDim.x) {
        fe_acc a;
        acc_zero(a);
        const size_t base = hi << lb;
        for (size_t lo = threadIdx.x; lo < ((size_t)1 << lb); lo += blockDim.x) {
            if (base + lo < len) acc_mul_add(a, fe_load_nc(data + base + lo), fe_load_nc(wl + lo));
        }
        fe row = block_sum(acc_reduce(a), scratch);
        if (threadIdx.x == 0) total = fe_add(total, fe_mul(row, fe_load_nc(wh + hi)));
    }
    if (threadIdx.x == 0) fe_store(partials + blockIdx.x, total);
}
__global__ void __launch_bounds__(256) sum_partials_kernel(const fe* __restrict__ partials, int count, fe* __restrict__ out) {
    __shared__ fe scratch[32];
    fe a = fe_zero();
    for (int b = threadIdx.x; b < count; b += blockDim.x) a = fe_add(a, partials[b]);
    a = block_sum(a, scratch);
    if (threadIdx.x == 0) fe_store(out, a);
}

// builds WH (2^(nv-lb) entries) and WL (2^lb entries); points from the host (uploaded into the scratch) or already in HBM
// (points_dev).  The scratch is allocated (*scratch, the caller frees it) unless given in scratch_in.
static void weight_split(size_t n_vars, int* lb, int* hb) {
    *lb = (int)n_vars < 12 ? (int)n_vars : 12;
    *hb = (int)n_vars - *lb;
}
size_t eq_weights_elems(size_t n_vars) {
    int lb, hb;
    weight_split(n_vars, &lb, &hb);
    return n_vars + ((size_t)1 << lb) + ((size_t)1 << hb);
}
static int build_weights(const hfe* points, size_t n_vars, int mode, cudaStream_t s, fe** scratch, fe** wh, fe** wl, int* lb_out,
                         const fe* points_dev = nullptr, fe* scratch_in = nullptr) {
    const int nv = (int)n_vars;
    int lb, hb;
    weight_split(n_vars, &lb, &hb);
    *scratch = nullptr;
    fe* pts = scratch_in;
    if (!pts) {
        MLB_TRY(dev_alloc_async((void**)scratch, eq_weights_elems(n_vars) * 16, s));
        pts = *scratch;
    }
    *wl = pts + n_vars;
    *wh = *wl + ((size_t)1 << lb);
    if (points_dev) pts = (fe*)points_dev;
    else if (n_vars) MLB_CUDA(cudaMemcpyAsync(pts, points, n_vars * 16, cudaMemcpyHostToDevice, s));
    weight_table_kernel<<<((1u << lb) + 255) / 256, 256, 0, s>>>(pts, nv, 0, lb, mode, *wl);
    MLB_KERNEL_CHECK();
    weight_table_kernel<<<((1u << hb) + 255) / 256, 256, 0, s>>>(pts, nv, lb, hb, mode, *wh);
    MLB_KERNEL_CHECK();
    *lb_out = lb;
    return ML_OK;
}
static int sepdot(Ctx* ctx, const fe* data, size_t len, const fe* wh, const fe* wl, int lb, size_t rows, hfe* out, cudaStream_t s) {
    unsigned nb = (unsigned)(rows < (size_t)ctx->sm_count * 4 ? rows : (size_t)ctx->sm_count * 4);
    if (nb == 0) nb = 1;
    fe* partials;
    MLB_TRY(dev_alloc_async((void**)&partials, (size_t)(nb + 1) * 16, s));
    sepdot_kernel<<<nb, 256, 0, s>>>(data, len, wh, wl, lb, rows, partials);
    MLB_KERNEL_CHECK();
    sum_partials_kernel<<<1, 256, 0, s>>>(partials, (int)nb, partials + nb);
    MLB_KERNEL_CHECK();
    uint8_t tmp[16];
    MLB_CUDA(cudaMemcpyAsync(tmp, partials + nb, 16, cudaMemcpyDeviceToHost, s));
    MLB_CUDA(cudaStreamSynchronize(s));
    *out = hfe_load(tmp);
    MLB_TRY(dev_free_async(partials, s));
    return ML_OK;
}

static int mle_evaluate(Ctx* ctx, const fe* data, size_t len, const hfe* args, size_t n_args, int mode, hfe* out, cudaStream_t s) {
    // assert_eq!(1 << args.len(), len.next_power_of_two()) — polynomials.rs:127-131, :166-170
    size_t np2 = 1;
    while (np2 < len) np2 <<= 1;
    if (n_args >= 40 || ((size_t)1 << n_args) != np2) { set_error("Wrong number of arguments"); return ML_ERR_SIZE; }
    fe *scratch, *wh, *wl;
    int lb;
    MLB_TRY(build_weights(args, n_args, mode, s, &scratch, &wh, &wl, &lb));
    int st = sepdot(ctx, data, len, wh, wl, lb, (size_t)1 << (n_args - lb), out, s);
    MLB_TRY(dev_free_async(scratch, s));
    return st;
}
int mle_evals_evaluate_launch(Ctx* ctx, const fe* evals, size_t len, const hfe* args, size_t n_args, hfe* out, cudaStream_t s) {
    return mle_evaluate(ctx, evals, len, args, n_args, 0, out, s);
}
int mle_coeffs_evaluate_launch(Ctx* ctx, const fe* coeffs, size_t len, const hfe* args, size_t n_args, hfe* out, cudaStream_t s) {
    return mle_evaluate(ctx, coeffs, len, args, n_args, 1, out, s);
}
// delta table of SumcheckTables::build_tables_for_pcs (sumcheck.rs:133-138)
int eq_table_launch(Ctx* ctx, const hfe* inputs, size_t n_vars, fe* delta, cudaStream_t s, const fe* points_dev, fe* scratch_in) {
    fe *scratch, *wh, *wl;
    int lb;
    MLB_TRY(build_weights(inputs, n_vars, 0, s, &scratch, &wh, &wl, &lb, points_dev, scratch_in));
    const size_t n = (size_t)1 << n_vars;
    size_t blocks = (n + 255) / 256;
    if (blocks > (size_t)ctx->sm_count * 16) blocks = (size_t)ctx->sm_count * 16;
    ProfScope prof(PROF_EQ_TABLE, 16.0 * (double)n, s);
    outer_product_kernel<<<(unsigned)blocks, 256, 0, s>>>(wh, wl, lb, n, delta);
    MLB_KERNEL_CHECK();
    return scratch ? dev_free_async(scratch, s) : ML_OK;
}
// Polynomial::evaluate (src/ntt/mod.rs:62-67): sum_i c_i x^i with x^i = XH[i >> 12] * XL[i & 4095]
int poly_eval_launch(Ctx* ctx, const fe* coeffs, size_t n, hfe x, hfe* out, cudaStream_t s) {
    if (n == 0) { *out = 0; return ML_OK; }
    const int lb = 12;
    const size_t rows = (n + ((size_t)1 << lb) - 1) >> lb;
    fe* scratch;
    MLB_TRY(dev_alloc_async((void**)&scratch, (((size_t)1 << lb) + rows) * 16, s));
    fe *xl = scratch, *xh = scratch + ((size_t)1 << lb);
    power_table_kernel<<<(1u << lb) / 256, 256, 0, s>>>(to_dev_fe_h(x), 0, 1u << lb, xl);
    MLB_KERNEL_CHECK();
    power_table_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, s>>>(to_dev_fe_h(x), lb, (unsigned)rows, xh);
    MLB_KERNEL_CHECK();
    int st = sepdot(ctx, coeffs, n, xh, xl, lb, rows, out, s);
    MLB_TRY(dev_free_async(scratch, s));
    return st;
}

}  // namespace mlb
