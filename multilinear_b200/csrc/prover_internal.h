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
// evals (n) -> to_coefficient -> bit_reverse -> reed_solomon into code (2n); work: 3n elements of scratch or nullptr
int encode_into(Ctx* ctx, const fe* evals_dev, size_t n, fe* code, cudaStream_t s, fe* work = nullptr);
void derive_indices(ml_transcript* t, size_t domain_size, std::vector<size_t>& idx);
void fill_dirs(PathH& p, size_t index, int depth);
// appends layer `code` (n elements) to f with its Merkle tree (build_tree) but without reading the root back; digests: the
// tree's buffer (2 * n/2 digests, not owned) or nullptr for a pool allocation
int fri_push_layer(ml_fri* f, fe* code, size_t n, bool owns_code, cudaStream_t s, bool build_tree, uint8_t* digests = nullptr);
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
    // buffers of a prove plan, indexed by layer: the code and the Merkle digests of every layer the chain commits (instead of
    // pool allocations; the layers do not own them).  In a batched chain layer 0 is first_fold's output, whose tree goes to
    // layer_digests[0].
    fe* const* layer_code = nullptr;
    uint8_t* const* layer_digests = nullptr;
};
// the fold chain's scratch block: transcript | r, r/2 | prev | last[2] | status | roots[64] | sc[2*64] | sumcheck partials
static const size_t CHAIN_OFF_TR = 0, CHAIN_OFF_R = 128, CHAIN_OFF_PREV = CHAIN_OFF_R + 32, CHAIN_OFF_LAST = CHAIN_OFF_PREV + 16,
                    CHAIN_OFF_STATUS = CHAIN_OFF_LAST + 32, CHAIN_OFF_ROOTS = CHAIN_OFF_STATUS + 16, CHAIN_OFF_SC = CHAIN_OFF_ROOTS + 64 * 32,
                    CHAIN_OFF_PART = CHAIN_OFF_SC + 2 * 64 * 16;
size_t chain_scratch_bytes();
struct ChainRun {
    size_t first_new_layer = 0;  // layers whose roots the chain wrote at CHAIN_OFF_ROOTS
    bool used_tail = false;      // the chain produced last_element (at CHAIN_OFF_LAST)
};
int fold_chain_enqueue(Ctx* ctx, ml_fri* f, const ChainHooks* hooks, ml_sumcheck* sc, hfe prev, size_t k_start, bool pending,
                       ml_transcript* t, uint8_t* base, ChainRun* run, cudaStream_t s);
// BatchedPCSProverData::init's claim (batched_pcs.rs:44-49) and BatchedFriProverData::init after the batch tree
// (batched_fri.rs:80-86) on one thread: transcript from tr_in; with absorb_claim, absorb inputs (n_inputs) then outputs
// (n_outputs); absorb the root, draw rho and absorb it; transcript to tr_out (may equal tr_in).  rho_out = rho; prev_out
// (optional) = fingerprint(rho, outputs); r_out (optional) = {r_0, r_0 / 2}, the next challenge (batched_fri.rs:194).
int batch_root_launch(const DevTranscript* tr_in, DevTranscript* tr_out, const uint8_t* root, const fe* inputs, int n_inputs, const fe* outputs,
                      int n_outputs, bool absorb_claim, fe* rho_out, fe* prev_out, fe* r_out, cudaStream_t s);
int fold_chain_dev(Ctx* ctx, ml_fri* f, const ChainHooks* hooks, ml_sumcheck* sc, hfe prev, hfe* sc_out, size_t k_start, bool pending,
                   ml_transcript* t, cudaStream_t s);

}  // namespace mlbp
