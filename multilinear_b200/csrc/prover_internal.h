// Host-side helpers of prover.cu shared with shard.cu (the sharded batched prover).  Orchestration only.
#pragma once
#include <functional>
#include <vector>

#include "field.cuh"
#include "handles.h"
#include "internal.h"
#include "transcript.cuh"

namespace mlbp {
using namespace mlb;

struct Scratch {  // RAII stream-ordered scratch
    void* p = nullptr;
    cudaStream_t s;
    explicit Scratch(cudaStream_t st) : s(st) {}
    int alloc(size_t bytes) { return dev_alloc_async(&p, bytes, s); }
    void* release() { void* r = p; p = nullptr; return r; }
    ~Scratch() { if (p) cudaFreeAsync(p, s); }
    template <class T> T* as() { return (T*)p; }
};

int pmalloc(void** p, size_t bytes, cudaStream_t s);
void pfree(void* p, cudaStream_t s);
int h2d(void* dst, const void* src, size_t bytes, cudaStream_t s);
int d2h_sync(void* dst, const void* src, size_t bytes, cudaStream_t s);
int stream_wait_blocking(cudaStream_t s);
void trace(const char* tag);

void absorb_fe(ml_transcript* t, hfe x);
hfe challenge(ml_transcript* t);
void free_fri(ml_fri* f);
void free_sumcheck(ml_sumcheck* s);
int encode_into(Ctx* ctx, const fe* evals_dev, size_t n, fe* code, cudaStream_t s);
void derive_indices(ml_transcript* t, size_t domain_size, std::vector<size_t>& idx);
void fill_dirs(PathH& p, size_t index, int depth);
// appends layer `code` (n elements) to f with its Merkle tree (build_tree) but without reading the root back
int fri_push_layer(ml_fri* f, fe* code, size_t n, bool owns_code, cudaStream_t s, bool build_tree);
int fri_open_queries(const ml_fri* f, const std::vector<size_t>& indices, std::vector<QueryH>& out, cudaStream_t s);
// the RESTRICTION on a caller's gen_pows (include/multilinear_b200.h): NULL, or the powers of pow_2_generator(log_n0)
int check_gen_pows(int log_n0, const uint8_t* gen_pows, size_t gen_pows_len);
hfe fingerprint_host(hfe r, const hfe* c, size_t n);
// width-w composition terms (ml_wsumcheck_set_composition's checks): per-term offsets into term_cols and the total count
int wsumcheck_check_terms(size_t width, size_t n_terms, const uint32_t* term_lens, const uint32_t* term_cols, std::vector<uint32_t>& off, size_t* total);
// Lagrange coefficient matrix over x = 0..td: lag[i][j] = coefficient of x^i in L_j (polynomials.rs:51-86 for unit vectors)
int wsumcheck_lagrange(size_t td, std::vector<uint8_t>& lag);

// Optional pieces of the sync-free fold chain supplied by the caller.
struct ChainHooks {
    // Round 0 of a batched proof (f has no layer yet): produce the fold of the whole batch, half the domain long, from the
    // challenge left in HBM at r_dev ({r, r/2}).  *owns = the buffer came from pmalloc and passes to the FriProverData.
    std::function<int(const fe* r_dev, fe** next, bool* owns)> first_fold;
    const DevTranscript* tr_dev = nullptr;  // transcript state already in HBM (device copy instead of uploading the host state)
    const fe* prev_dev = nullptr;           // running sumcheck claim already in HBM
};
int fold_chain_dev(Ctx* ctx, ml_fri* f, const ChainHooks* hooks, ml_sumcheck* sc, hfe prev, hfe* sc_out, size_t k_start, bool pending,
                   ml_transcript* t, cudaStream_t s);

}  // namespace mlbp
