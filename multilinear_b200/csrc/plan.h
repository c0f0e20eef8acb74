// What the stream-ordered provers (plan.cu: FriProof / PCSProof, bplan.cu: BatchedFriProof / BatchedPCSProof) share: the device-side
// statement of the FriProof wire format, one query at a time, and the host-side argument checks of an enqueue call.
#pragma once
#include "prover_internal.h"

namespace mlbp {

const int PLAN_MAX_LAYERS = 40;  // log_domain <= 40: at most 39 committed layers

// The bincode wire format of a FriProof (fri/mod.rs:239-249, :367-369; Writer in prover.cu) at log_domain D, N = 2^D:
//   u64 nc | nc x 32 B commitments | u64 128 | 128 queries | Field128 last_element (u64 16 + 16 B) | 32 B last_random
// nc = D - 1 (layers N .. 4), query = u64 nc | nc paths; path j (depth d_j = D - 1 - j) =
//   u64 16 | value 16 B | u64 16 | minus_value 16 B | u64 d_j | d_j x (32 B sibling digest | u32 direction)
// Every offset depends on D alone.  Writer (prover.cu) states the same format for ml_fri_proof objects; the parity tests of
// tests/test_prove_plan.py and tests/test_batched_prove_plan.py compare the two byte for byte at every size.
__host__ __device__ inline size_t path_offset(int D, int j) {  // within a query
    const size_t jj = (size_t)j;
    return 8 + 56 * jj + 36 * (jj * (size_t)(D - 1) - jj * (jj - 1) / 2);
}
__host__ __device__ inline size_t query_bytes(int D) { return path_offset(D, D - 1); }
__host__ __device__ inline size_t header_bytes(int D) { return 16 + 32 * (size_t)(D - 1); }

// every field of a blob starts at a multiple of 4 bytes from its 16-byte aligned start
__device__ __forceinline__ void put32(uint8_t* p, uint32_t v) { *reinterpret_cast<uint32_t*>(p) = v; }
__device__ __forceinline__ void put64(uint8_t* p, unsigned long long v) { put32(p, (uint32_t)v); put32(p + 4, (uint32_t)(v >> 32)); }
__device__ __forceinline__ uint32_t word(const void* p, int i) { return reinterpret_cast<const uint32_t*>(p)[i]; }

// Merkle path of leaf idx in a tree of L leaves (all layers at `digests`, merkle_layer_offset): depth = log2 L entries of
// (32 B sibling | u32 direction) at out, entry t written by the threads t, t + nthreads, ... (sibling and direction as
// merkle_tree/mod.rs:43-55)
__device__ __forceinline__ void write_path_tail(uint8_t* out, const uint8_t* digests, unsigned long long L, unsigned long long idx, int depth,
                                                int t0, int nthreads) {
    for (int t = t0; t < depth; t += nthreads) {
        const uint8_t* src = digests + 32 * ((2 * L - ((2 * L) >> t)) + ((idx >> t) ^ 1ull));
        uint8_t* dst = out + 36 * (size_t)t;
#pragma unroll
        for (int w = 0; w < 8; w++) put32(dst + 4 * w, word(src, w));
        put32(dst + 32, ((idx >> t) & 1ull) ? 0u : 1u);  // even index: the sibling is on the Right
    }
}

// One FriProof query (open_query_at, fri/mod.rs:154-174) at log_domain D over layers code[0 .. D-2] (layer j: 2^(D-j) elements,
// its tree at digests[j]) for index idx0 in [0, 2^(D-1)), at qo (query_bytes(D) bytes).  Called by every thread of a CTA: one
// warp per layer, lanes 0..7 the value pair and lengths, every lane one sibling digest of the path.
__device__ __forceinline__ void write_fri_query(uint8_t* qo, const fe* const* code, const uint8_t* const* digests, int D, unsigned long long idx0) {
    const int nc = D - 1, tid = threadIdx.x, lane = tid & 31;
    if (tid == 0) put64(qo, (unsigned long long)nc);
    for (int j = tid >> 5; j < nc; j += blockDim.x >> 5) {
        const int depth = D - 1 - j;
        const unsigned long long L = 1ull << depth, idx = idx0 & (L - 1);  // the index folds with the domain (cur %= cur_n)
        uint8_t* po = qo + path_offset(D, j);
        if (lane == 0) { put64(po, 16); put64(po + 24, 16); put64(po + 48, (unsigned long long)depth); }
        if (lane < 4) put32(po + 8 + 4 * lane, word(code[j] + idx, lane));
        else if (lane < 8) put32(po + 32 + 4 * (lane - 4), word(code[j] + idx + L, lane - 4));
        write_path_tail(po + 56, digests[j], L, idx, depth, lane, 32);
    }
}

// ------------------------------------------------------------------ host-side checks of an enqueue call
struct PlanBuf {
    const void* p;
    size_t bytes;
    bool out;
    const char* name;
    long index = -1;  // position in a caller's pointer array, or -1
};
// null, misaligned and overlapping buffers (an output may overlap nothing else): ML_ERR_ARG before anything is enqueued
int plan_check_bufs(const PlanBuf* b, size_t n);

}  // namespace mlbp
