// Device-resident Fiat-Shamir transcript (src/transcript.rs:16-39): one running SHA-256 over everything absorbed;
// `random()` finalises a CLONE, so challenges are idempotent until the next absorb.
//
// The transcript is strictly sequential (root -> challenge -> fold -> root ...).  Keeping it on the host costs a
// device->host round trip per FRI round; here one thread of a tiny kernel (or of the fused tail kernel) advances
// it in HBM / shared memory, so a whole fold chain is enqueued without any host synchronisation.
// The state layout equals mlb::HostSha256 (sha256.cuh), so host and device states are memcpy-compatible.
#pragma once
#include "field.cuh"
#include "sha256.cuh"

namespace mlb {

struct DevTranscript {
    uint32_t h[8];
    uint8_t buf[64];
    unsigned long long len;
};
static_assert(sizeof(DevTranscript) == sizeof(HostSha256), "device and host transcript states must be memcpy-compatible");

// one call site per kernel keeps the 22 KB unrolled compression out of every absorb/digest expansion; a translation
// unit that already owns a non-inlined compression routes the transcript through it with MLB_DT_COMPRESS
#ifndef MLB_DT_COMPRESS
#define MLB_DT_COMPRESS(h, w) sha_compress(h, w)
#endif
static __device__ __noinline__ void dt_compress_block(uint32_t h[8], const uint8_t* p) {
    uint32_t w[16];
#pragma unroll
    for (int i = 0; i < 16; i++)
        w[i] = ((uint32_t)p[4 * i] << 24) | ((uint32_t)p[4 * i + 1] << 16) | ((uint32_t)p[4 * i + 2] << 8) | (uint32_t)p[4 * i + 3];
    MLB_DT_COMPRESS(h, w);
}
__device__ inline void dt_absorb(DevTranscript* t, const uint8_t* p, int n) {  // Transcript::absorb (:31-33)
    int fill = (int)(t->len & 63ull);
    t->len += (unsigned long long)n;
    for (int i = 0; i < n; i++) {
        t->buf[fill++] = p[i];
        if (fill == 64) {
            dt_compress_block(t->h, t->buf);
            fill = 0;
        }
    }
}
__device__ inline void dt_absorb_fe(DevTranscript* t, fe x) {
    uint8_t b[16];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        b[4 * i] = (uint8_t)x.v[i]; b[4 * i + 1] = (uint8_t)(x.v[i] >> 8); b[4 * i + 2] = (uint8_t)(x.v[i] >> 16); b[4 * i + 3] = (uint8_t)(x.v[i] >> 24);
    }
    dt_absorb(t, b, 16);
}
// Transcript::random (:23-29): digest of a clone; st_out receives the eight big-endian state words
__device__ inline void dt_digest_words(const DevTranscript* t, uint32_t st_out[8]) {
    uint32_t h[8];
    uint8_t blk[64];
#pragma unroll
    for (int i = 0; i < 8; i++) h[i] = t->h[i];
    const int fill = (int)(t->len & 63ull);
    for (int i = 0; i < 64; i++) blk[i] = i < fill ? t->buf[i] : (i == fill ? 0x80 : 0);
    if (fill >= 56) {
        dt_compress_block(h, blk);
        for (int i = 0; i < 64; i++) blk[i] = 0;
    }
    const unsigned long long bits = t->len * 8ull;
#pragma unroll
    for (int i = 0; i < 8; i++) blk[56 + i] = (uint8_t)(bits >> (56 - 8 * i));
    dt_compress_block(h, blk);
#pragma unroll
    for (int i = 0; i < 8; i++) st_out[i] = h[i];
}
// Transcript::next_challenge (:35-38): first 16 digest bytes as a little-endian u128, then BaseElement::new
__device__ inline fe dt_challenge(const DevTranscript* t) {
    uint32_t st[8];
    dt_digest_words(t, st);
    // digest bytes are the big-endian state words; bytes 0..15 read as LE u128 -> limb i = bswap(st[i])
    return fe_new(fe{{sha_bswap(st[0]), sha_bswap(st[1]), sha_bswap(st[2]), sha_bswap(st[3])}});
}

// BatchedFriProverData::init after the batch tree (batched_fri.rs:80-86) and the claim of BatchedPCSProof::prove
// (batched_pcs.rs:92-94): absorb the batch root, draw rho = fingerprint_r and absorb it; returns fingerprint(rho, outputs)
__device__ inline fe dt_batch_root(DevTranscript* t, const uint8_t* root, const fe* outputs, int n_outputs, fe* rho_out) {
    dt_absorb(t, root, 32);
    const fe rho = dt_challenge(t);
    dt_absorb_fe(t, rho);
    fe acc = fe_zero();
    for (int j = 0; j < n_outputs; j++) acc = fe_add(fe_mul(acc, rho), fe_load(outputs + j));
    *rho_out = rho;
    return acc;
}

}  // namespace mlb
