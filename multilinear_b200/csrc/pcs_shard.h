// Stages of the block-sharded provers, shared by pcs_shard.cu (one PCSProof::prove, ml_pcs_shard_*), bpcs_shard.cu (one
// BatchedPCSProof::prove, ml_bpcs_shard_*), fri_shard.cu (one FriProof::prove, ml_fri_shard_*) and bfri_shard.cu (one
// BatchedFriProof::prove, ml_bfri_shard_*).  All split every polynomial by block over G ranks and keep the sharded layers in the
// segment layout described at the top of pcs_shard.cu; the batched provers add a batched layer 0 and round 0 (implemented in
// bpcs_shard.cu), the FRI provers drop the sumcheck tables (their table-free stages are implemented in fri_shard.cu).
#pragma once
#include "peer.h"
#include "prover_internal.h"

namespace mlbs {
using namespace mlb;
using namespace mlbp;

// PR0 + k: round k (L <= 4); PB: batched provers only; PT: batched PCS prover only; PC: FRI provers only (coefficient transpose)
enum Phase { PX = 0, PR0 = 1, PG = PR0 + 4, PF, PB, PT, PC, N_PHASES };
static const int MAXR = PEER_MAXR;
static const int MAX_L = 4;
static const size_t MAIL_ROOTS = (size_t)MAXR * MAXR / 2;  // run roots of layer 0 at G = ML_MAX_PEERS

struct Layout {
    size_t flags, status, tr, prev, r, sc, roots_out, final_tr, mail[MAX_L], top[MAX_L], part;  // mailbox (cleared at create)
    size_t rho, outs, eptrs, segptrs;                                                          // batched prover only
    size_t ycode, recv, coef, layer[MAX_L], dig[MAX_L], m, d, tail_code, tail_m, tail_d, total;  // coef: FRI provers only
};
// B = 0: one polynomial; B >= 1: a batch of B polynomials (layer 0 holds B codes); fri: no sumcheck tables, with a receive buffer
// for the transposed coefficients instead (batched: B slices of n/G inside layer 0, which is written only after they are encoded)
Layout make_layout(size_t n, int G, size_t B, bool fri = false);
// mailbox of round k: run root of run q at roots + 32 q, partial pair of rank g at partials + 32 g
inline size_t mail_partials(const Layout& a, int k) { return a.mail[k] + MAIL_ROOTS * 32; }

struct ShardCore {
    int world = 1, L = 0;
    size_t n_vars = 0, n = 0, NL = 0, R = 0, nloc = 0, B = 0;
    const char* who = "ml_pcs_shard";  // prefix of error messages
    Layout lay;
    std::vector<PeerRank> local;
    PeerGroup grp;
    // device-time marks of the last call on the first local rank's main stream (include/multilinear_b200_instr.h)
    static const int N_MARKS = 8;
    cudaEvent_t mark[N_MARKS] = {nullptr};
    int n_marks = 0;
};

inline fe* at(const PeerRank& r, size_t off) { return reinterpret_cast<fe*>(r.arena + off); }
void mark_phase(ShardCore* sh, int idx);
PeerRank* rank0_of(ShardCore* sh);

// handle plumbing (arguments already checked by the caller)
int shard_init(ShardCore* sh, int world, int n_local, const int* local_ranks, const int* local_devices, size_t n_vars, size_t B, const char* who,
               bool fri = false);
void shard_free(ShardCore* sh);
int shard_export(ShardCore* sh, uint8_t* records_out);
int shard_connect(ShardCore* sh, const uint8_t* records, size_t n_records, const char* who);
void* shard_stream(const ShardCore* sh, int local_index);
int shard_phase_ms(const ShardCore* sh, double* out, int cap);

// S0 exchange: slice r of the local code `ycode` -> rank r's recv at off_recv (G > 1)
int exchange_launch(ShardCore* sh, PeerRank& r, const fe* ycode, size_t off_recv, cudaStream_t s);
// cyclic transpose of a local table of nloc entries into the owners' tables at off_m: entry o of the block goes to rank
// (o mod G), or rank rev_L(o mod G) with rev_dest (the FRI prover's coefficients), at (b*nloc + o) / G
int tables_launch(ShardCore* sh, PeerRank& r, const fe* src, size_t off_m, cudaStream_t s, bool rev_dest = false);
// the eq table of rank `rank`'s cyclic share of the 2^v rows (rows i = m*2^L + rank): eq over the low v-L variables times the
// rank's factor for the top L variables (L = 0: eq over all variables); also used by wsumcheck_shard.cu
int local_eq_table(Ctx* ctx, const std::vector<hfe>& pts, int v, int L, int rank, fe* d, cudaStream_t s);
// S1: layer 0 from the received columns; mobius: the local codes encode evaluations (PCS), else coefficients (FRI)
int combine_launch(int L, const fe* recv, size_t R, int rank, int log_N, const RootTables* rt, fe* layer0, cudaStream_t s, bool mobius = true);
// run roots of `segs` segment subtrees (digests at dig, segment p at 32 * p * 2 R) -> every rank's mailbox at off_roots, and
// (nb >= 0) the rank's partial sums from its CTA partials -> off_partials; then flag `phase` there
int post_launch(ShardCore* sh, PeerRank& r, const uint8_t* dig, size_t R, int segs, int nb, size_t off_roots, size_t off_partials, int phase);
// wait for `phase` from every rank, then hash the top of a tree over cnt run roots of mailbox k into top[k]
int top_launch(ShardCore* sh, PeerRank& r, int phase, int k, int cnt);
// round polynomial of round k from the posted partial sums (absorbing `root` first if given), challenge r_k, claim update
int finish_launch(ShardCore* sh, PeerRank& r, int k, const uint8_t* root);

// sharded round k >= 0 of a single code layer: A (subtrees + post), B (top + transcript), C (folds)
int stage_post(ShardCore* sh, PeerRank& r, int k, int nb);
int stage_round(ShardCore* sh, PeerRank& r, int k);
int stage_fold(ShardCore* sh, PeerRank& r, int k, int* nb);  // fold_code + fold_tables
// FRI fold of the code of layer k into fold_target
int fold_code(ShardCore* sh, PeerRank& r, int k);
// where round k writes its fold: layer k+1 in the segment layout, or rank 0's tail code after the last sharded round
fe* fold_target(ShardCore* sh, PeerRank& r, int k);
// fold of the tables of round k; after the last sharded round, hand the tables to rank 0 and flag PG
int fold_tables(ShardCore* sh, PeerRank& r, int k, int* nb);

// rank 0: the fold chain from layer L (first_fold: a batched round 0 at G = 1), sumcheck coefficients and roots of the sharded
// rounds (sumcheck: 2 * n_vars, or nullptr for a plain FRI proof without tables; roots_lo: 32 * L); marks mark_base and
// mark_base + 1
int tail_chain(ShardCore* sh, PeerRank& r0, ml_fri* f, const ChainHooks& hooks, hfe* sumcheck, uint8_t* roots_lo, ml_transcript* t, int mark_base);
// rank 0: records (value pair | path) of layers j0 .. L-1 for every query index, from the owners' arenas; record (q, j) at
// (q * L + j) * *stride
int open_sharded(ShardCore* sh, PeerRank& r0, const std::vector<size_t>& idx, int j0, std::vector<uint8_t>& host, int* stride);
// rank 0: openings and the FriProof of one code (fri/mod.rs:261-285): layers < L from the owners' arenas, layers >= L from the
// tail's FriProverData; roots_lo: the roots of the sharded layers
int assemble_fri(ShardCore* sh, PeerRank& r0, const ml_fri* f, ml_transcript* t, ml_fri_proof* p, const uint8_t* roots_lo);
// rank 0: final transcript to every rank (releases their buffers); the other local ranks wait for it and adopt it
int tail_release(ShardCore* sh, PeerRank& r0, ml_transcript* t);
// rank 0 after a failed call: its status into every rank's status word, then the same release (finish_ranks returns it)
int tail_fail(ShardCore* sh, PeerRank& r0, int st);
int finish_ranks(ShardCore* sh, ml_transcript* t, int st);

// ---- the FRI provers (fri_shard.cu): no sumcheck tables, every layer root absorbed before its challenge
// transcript state and status word of one rank at the start of a call
int fri_begin(ShardCore* sh, PeerRank& r, const uint8_t* tr_state);
// S0 of a given code: slice [r*R, (r+1)*R) of this rank's block `code` (N/G elements) = run `rank` of rank r's code at off_code
int place_launch(ShardCore* sh, PeerRank& r, const fe* code, size_t off_code, cudaStream_t s);
// round k, phase B: top of the layer tree; absorb its root, draw r_k (identical on every rank)
int fri_round(ShardCore* sh, PeerRank& r, int k);
// round k, phase C: fold; after the last sharded round layer L is in rank 0's tail code (flag PG)
int fri_fold(ShardCore* sh, PeerRank& r, int k);

// ---- the batched provers (bpcs_shard.cu): B codes in layer 0 under one batched tree
struct BatchCore : ShardCore {
    struct Events { cudaEvent_t done[2] = {nullptr, nullptr}, free[2] = {nullptr, nullptr}, join = nullptr; };
    std::vector<Events> ev;  // per local rank: the S0 encode / exchange pipeline
    size_t R0 = 0;           // leaves of a layer-0 segment (R, or N/2 at G = 1)
    int segs0 = 1, cnt0 = 1; // layer-0 segments per rank, run roots of the batch tree
};
// after shard_init: the pipeline events and the code pointers of every layer-0 segment
int batch_init(BatchCore* sh);
void batch_free(BatchCore* sh);  // the events; then shard_free
// S0 of local rank li (G > 1): per code j, encode(j, y, main) into one of two buffers on the main stream while the side stream
// stores slice r of code j-1 into rank r's recv slice j-1; flag PX -> all
int batch_encode_exchange(BatchCore* sh, size_t li, const std::function<int(size_t j, fe* y, cudaStream_t s)>& encode);
// S1: G > 1: wait PX, then (combine) recv slice j -> layer-0 code j for every j; batched subtree of every segment, run roots -> all
// (flag PB)
int batch_commit(BatchCore* sh, PeerRank& r, bool combine, bool mobius);
const uint8_t* batch_root(const BatchCore* sh, const PeerRank& r);
// round 0: fingerprint (rho from the arena) + fold of the B layer-0 codes with the global leaf index into out
int batch_fold0_launch(BatchCore* sh, PeerRank& r, const fe* r_dev, fe* out, cudaStream_t s);
// rank 0: openings and the BatchedFriProof (batched_fri.rs:296-308): layer 0 and layers 1 .. L-1 from the owners' arenas, the
// rest from the tail's FriProverData; roots_lo: the roots of the sharded layers (round 0 absorbed none)
int assemble_bfri(BatchCore* sh, PeerRank& r0, const ml_fri* f, ml_transcript* t, ml_bfri_proof* p, const uint8_t* roots_lo);

// segment-layout helpers on the device
__device__ __forceinline__ int ilog2_dev(size_t x) { return 63 - __clzll((unsigned long long)x); }
// merkle_layer_offset on the device: layer l of a tree with n leaves starts at digest 2n - (2n >> l)
__device__ __forceinline__ size_t layer_off(size_t n_leaves, int layer) { return 2 * n_leaves - ((2 * n_leaves) >> layer); }
__device__ __forceinline__ fe root_pow(const fe* __restrict__ lo, const fe* __restrict__ hi, size_t e) {
    fe w = fe_load_nc(lo + (e & (((size_t)1 << LO_BITS) - 1)));
    if (e >> LO_BITS) w = fe_mul(w, fe_load_nc(hi + (e >> LO_BITS)));
    return w;
}
// position of element j of run p in a layer with `runs` runs per rank (segment layout; one run: plain)
__device__ __forceinline__ size_t run_pos(size_t runs, size_t p, size_t j, size_t R) {
    if (runs == 1) return j;
    const size_t half = runs >> 1;
    return (p & (half - 1)) * 2 * R + (p >= half ? R : 0) + j;
}

}  // namespace mlbs
