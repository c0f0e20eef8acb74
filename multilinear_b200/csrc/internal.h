// Internal declarations shared by the .cu translation units of libmultilinear_b200.so.
#pragma once
#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/multilinear_b200.h"
#include "../../include/multilinear_b200_instr.h"

namespace mlb {

// ------------------------------------------------------------------ errors / launch accounting
void set_error(const char* fmt, ...);
extern std::atomic<unsigned long long> g_kernel_launches;
#define MLB_COUNT_LAUNCH() (++::mlb::g_kernel_launches)

#define MLB_CUDA(expr)                                                                          \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            ::mlb::set_error("CUDA error %s at %s:%d (%s)", cudaGetErrorString(_e), __FILE__, __LINE__, #expr); \
            return ML_ERR_CUDA;                                                                 \
        }                                                                                       \
    } while (0)
#define MLB_TRY(expr)                  \
    do {                               \
        int _st = (expr);              \
        if (_st != ML_OK) return _st;  \
    } while (0)
#define MLB_KERNEL_CHECK()                                                                      \
    do {                                                                                        \
        MLB_COUNT_LAUNCH();                                                                     \
        cudaError_t _e = cudaGetLastError();                                                    \
        if (_e != cudaSuccess) {                                                                \
            ::mlb::set_error("kernel launch failed: %s at %s:%d", cudaGetErrorString(_e), __FILE__, __LINE__); \
            return ML_ERR_CUDA;                                                                 \
        }                                                                                       \
    } while (0)

// ------------------------------------------------------------------ optional per-kernel timing (CUDA events on the launch stream)
enum ProfId { PROF_NTT_PASS = 0, PROF_MERKLE_LEAF, PROF_MERKLE_NODES, PROF_MERKLE_TOP, PROF_FRI_FOLD, PROF_SUMCHECK_SUMS,
              PROF_SUMCHECK_FOLD, PROF_MOBIUS, PROF_EQ_TABLE, PROF_BITREV, PROF_GATHER, PROF_TAIL, PROF_TRANSCRIPT, PROF_COUNT };
extern bool g_prof_on;
long prof_begin(int id, double alg_bytes, cudaStream_t s);  // returns a record index
void prof_end(long rec, cudaStream_t s);
struct ProfScope {  // brackets the kernel launches issued inside its lifetime (thread-safe: several host threads may drive streams)
    cudaStream_t s; long rec;
    ProfScope(int id, double alg_bytes, cudaStream_t s_) : s(s_), rec(g_prof_on ? prof_begin(id, alg_bytes, s_) : -1) {}
    ~ProfScope() { if (rec >= 0) prof_end(rec, s); }
};

// ------------------------------------------------------------------ host scalar field (transcript challenges,
// round polynomials, root-of-unity parameters).  Scalars only: all array work is on the GPU.
typedef unsigned __int128 hfe;
static const hfe HFE_M = ((((hfe)0xFFFFFFFFFFFFFFFFULL) << 64) | (hfe)0xFFFFD30000000001ULL);
static const uint64_t HFE_C = 0x2CFFFFFFFFFFULL;

static inline hfe hfe_new(hfe x) { return x >= HFE_M ? x - HFE_M : x; }
static inline hfe hfe_from_i64(int64_t v) { return hfe_new((hfe)(__int128)v); }
static inline hfe hfe_load(const uint8_t* p) { hfe x; memcpy(&x, p, 16); return x; }
static inline void hfe_store(uint8_t* p, hfe x) { memcpy(p, &x, 16); }
static inline hfe hfe_add(hfe a, hfe b) { hfe s = a + b; return (s < a || s >= HFE_M) ? s - HFE_M : s; }
static inline hfe hfe_sub(hfe a, hfe b) { return a >= b ? a - b : a + (HFE_M - b); }
static inline hfe hfe_neg(hfe a) { return a ? HFE_M - a : 0; }
static inline hfe hfe_mul(hfe a, hfe b) {
    uint64_t a0 = (uint64_t)a, a1 = (uint64_t)(a >> 64), b0 = (uint64_t)b, b1 = (uint64_t)(b >> 64);
    hfe p00 = (hfe)a0 * b0, p01 = (hfe)a0 * b1, p10 = (hfe)a1 * b0, p11 = (hfe)a1 * b1;
    hfe mid = (p00 >> 64) + (uint64_t)p01 + (uint64_t)p10;
    hfe lo = ((hfe)(uint64_t)mid << 64) | (uint64_t)p00;
    hfe hi = p11 + (p01 >> 64) + (p10 >> 64) + (mid >> 64);
    while (hi) {  // fold 2^128 == c
        hfe q0 = (hfe)(uint64_t)hi * HFE_C, q1 = (hfe)(uint64_t)(hi >> 64) * HFE_C;
        hfe t = q0 + (q1 << 64);
        hfe nhi = (q1 >> 64) + (t < q0);
        hfe s = lo + t;
        nhi += (s < lo);
        lo = s;
        hi = nhi;
    }
    return hfe_new(lo);
}
static inline hfe hfe_pow(hfe b, hfe e) {
    hfe r = 1;
    while (e) { if (e & 1) r = hfe_mul(r, b); b = hfe_mul(b, b); e >>= 1; }
    return r;
}
static inline hfe hfe_inv(hfe a) { return a ? hfe_pow(a, HFE_M - 2) : 0; }
static inline hfe hfe_div(hfe a, hfe b) { return hfe_mul(a, hfe_inv(b)); }
static inline hfe hfe_half(hfe a) { return hfe_mul(a, (HFE_M + 1) >> 1); }
// NttField::pow_2_generator (src/ntt/mod.rs:42-54); returns false for log_size > 40
static inline bool hfe_pow2_generator(uint64_t log_size, hfe* out) {
    if (log_size > 40) return false;
    *out = hfe_pow(3, (HFE_M - 1) >> log_size);
    return true;
}
static inline bool is_pow2(size_t n) { return n && !(n & (n - 1)); }
static inline unsigned ilog2(size_t n) { return 63u - (unsigned)__builtin_clzll((unsigned long long)n); }

struct fe;  // device element (field.cuh)

// ------------------------------------------------------------------ per-device context
// Root-of-unity tables for one domain size N = 2^log_n, generator w = pow_2_generator(log_n):
//   lo[i]  = w^i              i < 2^LO_BITS (or N if smaller)
//   hi[i]  = w^(i << LO_BITS) i < N >> LO_BITS
//   lo_ninv[i] = lo[i] / N    (inverse transforms fold the 1/N scaling into the inter-pass twiddle)
// so w^e = hi[e >> LO_BITS] * lo[e & mask] for any e < N, and w^-e = w^(N-e).
static const int LO_BITS = 12;
struct RootTables {
    int log_n = 0;
    fe* lo = nullptr;
    fe* hi = nullptr;
    fe* lo_ninv = nullptr;
    hfe gen = 0;
    // inter-pass twiddle matrices of the multi-pass NTT plan for this size: pass_tw[inverse][pass][k*B + b] =
    // w_N^(+-k*b*A) (times 1/N for pass 0 of the inverse), laid out like the data so the store loop reads it coalesced
    fe* pass_tw[2][4] = {{nullptr, nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr, nullptr}};
};
struct Ctx {
    int device = -1;
    cudaStream_t stream = nullptr;  // library stream for host-pointer entry points
    std::map<int, RootTables> roots;
    std::mutex roots_mu;  // guards `roots` and the lazily built tables inside it
    fe* small_fwd = nullptr;  // w_4096^i, i < 2048   (in-tile twiddles for every pass radix <= 4096)
    fe* small_inv = nullptr;  // w_4096^-i
    int sm_count = 148;
};
int get_ctx(Ctx** out);  // context of the current device (lazily created)
// stream used by host-pointer entry points: the calling thread's override (ml_set_thread_stream) or the context stream
cudaStream_t lib_stream(Ctx* ctx);
// a stream owned by the library with its private allocation pool (what ml_stream_create hands out); non_blocking: not ordered
// against the legacy default stream
int lib_stream_create(cudaStream_t* out, bool non_blocking);
int lib_stream_destroy(cudaStream_t s);
int get_root_tables(Ctx* ctx, int log_n, cudaStream_t s, const RootTables** out);

// stream-ordered scratch allocation
int dev_alloc_async(void** p, size_t bytes, cudaStream_t s);
int dev_free_async(void* p, cudaStream_t s);

// ------------------------------------------------------------------ kernels (launchers)
// ntt.cu
// bitrev_in: the n live coefficients are stored bit-reversed (PCS encode); fused into pass 0, multi-pass sizes only.
// tmp: 2^log_n elements of scratch for the multi-pass plans (nullptr: a stream-ordered allocation per call)
int ntt_launch(Ctx* ctx, const fe* in, fe* out, int log_n, bool inverse, bool rs_zero_padded, cudaStream_t s, bool bitrev_in = false,
               fe* tmp = nullptr);
int ntt_prepare(Ctx* ctx, int log_n, cudaStream_t s);
static inline bool ntt_fuses_bitrev(int log_n) { return log_n > 12; }
int powers_launch(Ctx* ctx, int log_n, fe* out, cudaStream_t s);
int bit_reverse_launch(const void* in, void* out, size_t n, size_t elem_bytes, cudaStream_t s);
// field_ops.cu
int fe_vec_launch(int op, const fe* a, const fe* b, size_t n, fe* out, cudaStream_t s);
int fe_pow_vec_launch(const fe* a, hfe e, size_t n, fe* out, cudaStream_t s);
int fe_from_i64_launch(const int64_t* v, size_t n, fe* out, cudaStream_t s);
int fe_from_wide_launch(const void* v, size_t n, int variant, fe* out, cudaStream_t s);
int synthetic_launch(uint64_t seed, size_t n, fe* out, cudaStream_t s);
// mle.cu
int mobius_launch(const fe* in, fe* out, size_t len, bool subtract, cudaStream_t s);
int mle_evals_evaluate_launch(Ctx* ctx, const fe* evals, size_t len, const hfe* args, size_t n_args, hfe* out, cudaStream_t s);
int mle_coeffs_evaluate_launch(Ctx* ctx, const fe* coeffs, size_t len, const hfe* args, size_t n_args, hfe* out, cudaStream_t s);
// points_dev: the n_vars points already in HBM (inputs unused, no upload); scratch: eq_weights_elems(n_vars) elements (nullptr: allocated)
int eq_table_launch(Ctx* ctx, const hfe* inputs, size_t n_vars, fe* delta, cudaStream_t s, const fe* points_dev = nullptr, fe* scratch = nullptr);
size_t eq_weights_elems(size_t n_vars);
int poly_eval_launch(Ctx* ctx, const fe* coeffs, size_t n, hfe x, hfe* out, cudaStream_t s);
// merkle.cu — digests buffer holds all layers back to back: layer l starts at digest index 2L - (2L >> l)
static inline size_t merkle_layer_offset(size_t n_leaves, size_t layer) { return 2 * n_leaves - ((2 * n_leaves) >> layer); }
int merkle_rs_launch(const fe* code, size_t n_code, uint8_t* digests, cudaStream_t s);  // leaves (code[i], code[i+n/2])
int merkle_bytes_launch(const uint8_t* const* data_dev_ptrs, size_t n_batches, size_t item_bytes, size_t n_items, uint8_t* digests, cudaStream_t s);
int merkle_batched_rs_launch(const fe* const* codes_dev_ptrs, size_t n_codes, size_t n_code, uint8_t* digests, cudaStream_t s);
int merkle_batched_pairs_launch(const uint8_t* const* pairs_dev_ptrs, size_t n_codes, size_t n_leaves, uint8_t* digests, cudaStream_t s);
int merkle_batched_pairs_strided_launch(const uint8_t* pairs_base, size_t n_codes, size_t n_leaves, uint8_t* digests, cudaStream_t s);
int merkle_upper_launch(uint8_t* digests, size_t n_leaves, cudaStream_t s);  // layers 1.. from layer 0
// fri.cu — r_dev (optional): device pointer to {r, r/2} written by a transcript kernel; overrides the host value r
int fri_fold_launch(Ctx* ctx, const fe* cur, size_t n_cur, fe* next, hfe r, const fe* r_dev, size_t k, int log_n0, cudaStream_t s);
// rho_dev (optional): the fingerprint challenge read from HBM instead of fingerprint_r
int fri_batched_fold_launch(Ctx* ctx, const fe* const* codes_dev_ptrs, size_t n_codes, size_t n, fe* next, hfe fingerprint_r, hfe r,
                            const fe* r_dev, int log_n0, cudaStream_t s, const fe* rho_dev = nullptr);
// r_dev: rho read from HBM instead of r
int fingerprint_rows_launch(const fe* const* polys_dev_ptrs, size_t n_polys, size_t n, hfe r, fe* out, cudaStream_t s, const fe* r_dev = nullptr);
// sumcheck.cu
int sumcheck_sums_launch(Ctx* ctx, const fe* m, const fe* d, size_t height, hfe* s1, hfe* s2, cudaStream_t s);
int sumcheck_partial_sum_launch(Ctx* ctx, const fe* m, const fe* d, size_t height, hfe r, hfe* out, cudaStream_t s);
int sumcheck_fold_launch(fe* m, fe* d, size_t height, hfe r, const fe* r_dev, cudaStream_t s);
int wsumcheck_limits(int what);  // 0 max width, 1 max terms, 2 max column references
int wsumcheck_partial_sum_launch(const fe* m, const fe* d, size_t height, size_t width, hfe r, const fe* coef, const uint32_t* len,
                                 const uint32_t* off, const uint32_t* cols, size_t n_terms, size_t n_cols, hfe* out, cudaStream_t s);
int wsumcheck_fold_launch(fe* m, fe* d, size_t height, size_t width, hfe r, cudaStream_t s);
int wsumcheck_points_launch(const fe* m, const fe* d, size_t height, size_t width, const fe* coef, const uint32_t* len, const uint32_t* off,
                            const uint32_t* cols, size_t n_terms, size_t n_cols, int td, hfe* evals_out, cudaStream_t s);
// width-w composition as a sparse polynomial over the row (device arrays): comp(x) = sum_t coef[t] * prod_{k < len[t]} x[cols[off[t] + k]]
struct WTerms {
    const fe* coef;
    const uint32_t* len;
    const uint32_t* off;
    const uint32_t* cols;
    int n_terms, n_cols;
};
static const int W_MAX_WIDTH = 16, W_MAX_TERMS = 64, W_MAX_COLS = 256, W_MAX_TD = 4;
// device-chain pieces of the width-w sumcheck: per-CTA partials of all td points (td per CTA), fold with the challenge in HBM
int wsumcheck_points_partials_launch(const fe* m, const fe* d, size_t height, size_t width, const WTerms& t, int td, fe* partials, int* n_blocks,
                                     cudaStream_t s);
int wsumcheck_fold_dev_launch(fe* m, fe* d, size_t height, size_t width, const fe* r_dev, cudaStream_t s);
int sumcheck_fold_sums_launch(fe* m, fe* d, size_t height, const fe* r_dev, fe* partials /* 2 per CTA */, int* n_blocks, cudaStream_t s);
int sumcheck_sums_partials_launch(const fe* m, const fe* d, size_t height, fe* partials /* 2 per CTA */, int* n_blocks, cudaStream_t s);
int sumcheck_max_blocks();
// chain.cu — device-resident transcript steps and the fused tail of the fold chain
struct DevTranscript;
static const int TAIL_LOG = 12;          // the tail kernel takes over once the current code has <= 2^TAIL_LOG elements
static const int TAIL_MAX_ROUNDS = 12;
struct TailArgs {
    fe* codes[TAIL_MAX_ROUNDS + 1];         // codes[0]: current committed layer (n0 elements); codes[i+1]: output of tail round i
    uint8_t* digests[TAIL_MAX_ROUNDS + 1];  // digests[i]: all Merkle layers of codes[i]
    size_t n0;
    int k0, log_n0;
    const fe* lo;
    const fe* hi;
    DevTranscript* tr;
    uint8_t* roots_out;       // 32 bytes per committed tail layer
    uint8_t* first_root_out;  // where to copy codes[0]'s root when it is absorbed here
    fe* last_out;             // 2 elements; [0] = last_element
    int* status;
    int absorb_first_root;
    fe* m;                    // sumcheck tables (nullptr: plain FRI)
    fe* d;
    size_t height;
    fe* prev;
    fe* sc_out;               // (c1, c2) per tail round
};
int chain_challenge_launch(DevTranscript* tr, const uint8_t* absorb, int absorb_len, uint8_t* copy_out, fe* r_out, bool want_challenge,
                           cudaStream_t s);
int chain_sumcheck_finish_launch(const fe* partials, int nb, fe* prev, DevTranscript* tr, const uint8_t* absorb, int absorb_len,
                                 uint8_t* copy_out, fe* sc_out, fe* r_out, cudaStream_t s);
int chain_tail_launch(const TailArgs& a, cudaStream_t s);
int chain_sumcheck_tail_launch(fe* m, fe* d, size_t height, fe* prev, DevTranscript* tr, fe* sc_out, fe* r_out, cudaStream_t s);
int chain_last_launch(const fe* two, DevTranscript* tr, fe* last_out, int* status, cudaStream_t s);
// the 128 query indices of a domain of 2^(log_half+1) and last_random from the transcript at tr_in; final state to tr_out
int fri_query_indices_launch(const DevTranscript* tr_in, DevTranscript* tr_out, int log_half, unsigned long long* indices, uint8_t* last_random,
                             cudaStream_t s);
// width-w sumcheck rounds on the device (sumcheck.rs:174-202): lag = the (td+1) x (td+1) Lagrange coefficient matrix over x = 0..td
static const int WTAIL_LOG = 12;  // the tail kernel runs every remaining round once the tables have <= 2^WTAIL_LOG rows
int wchain_finish_launch(const fe* partials, int nb, int td, const fe* lag, fe* prev, DevTranscript* tr, fe* coef_out, fe* r_store, fe* r_dev,
                         cudaStream_t s);
int wchain_tail_launch(fe* m, fe* d, size_t height, int width, const WTerms& t, int td, const fe* lag, fe* prev, DevTranscript* tr, fe* coef_out,
                       fe* rs_out, cudaStream_t s);

}  // namespace mlb
