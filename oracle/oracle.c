/*
 * ORACLE — TEST INFRASTRUCTURE ONLY (see oracle/oracle.h).  PARITY UNPINNED.
 *
 * CPU restatement, loop for loop, of fr34za/multilinear's PCS hot path.  All
 * citations are relative to /root/reference/.  OpenMP pragmas only spread the
 * reference's (single-threaded) loops over host cores; integer arithmetic is
 * exact so results do not depend on the thread count.
 */
#include "oracle.h"
#include "field.h"
#include "sha256.h"
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

static int g_threads = 1;
void or_set_threads(int n) {
    if (n < 1) n = 1;
    g_threads = n;
#ifdef _OPENMP
    omp_set_num_threads(n);
#endif
}
int or_get_threads(void) { return g_threads; }
#define PAR_FOR _Pragma("omp parallel for schedule(static) if (g_threads > 1)")

static int is_pow2(size_t n) { return n != 0 && (n & (n - 1)) == 0; }
static uint64_t bitrev64(uint64_t x) { /* usize::reverse_bits */
    x = ((x >> 1) & 0x5555555555555555ULL) | ((x & 0x5555555555555555ULL) << 1);
    x = ((x >> 2) & 0x3333333333333333ULL) | ((x & 0x3333333333333333ULL) << 2);
    x = ((x >> 4) & 0x0F0F0F0F0F0F0F0FULL) | ((x & 0x0F0F0F0F0F0F0F0FULL) << 4);
    return __builtin_bswap64(x);
}
static unsigned ctz_sz(size_t n) { return n == 0 ? 64u : (unsigned)__builtin_ctzll((unsigned long long)n); }

/* ------------------------------------------------------------------ field */
void or_fe_add(const uint8_t a[16], const uint8_t b[16], uint8_t out[16]) { fe_store(out, fe_add(fe_load(a), fe_load(b))); }
void or_fe_sub(const uint8_t a[16], const uint8_t b[16], uint8_t out[16]) { fe_store(out, fe_sub(fe_load(a), fe_load(b))); }
void or_fe_mul(const uint8_t a[16], const uint8_t b[16], uint8_t out[16]) { fe_store(out, fe_mul(fe_load(a), fe_load(b))); }
void or_fe_div(const uint8_t a[16], const uint8_t b[16], uint8_t out[16]) { fe_store(out, fe_div(fe_load(a), fe_load(b))); }
void or_fe_neg(const uint8_t a[16], uint8_t out[16]) { fe_store(out, fe_neg(fe_load(a))); }
void or_fe_pow(const uint8_t a[16], const uint8_t e[16], uint8_t out[16]) { fe_store(out, fe_pow(fe_load(a), fe_load(e))); }
void or_fe_from_i64(int64_t v, uint8_t out[16]) { fe_store(out, fe_from_i64(v)); }
void or_fe_from_u128(const uint8_t v[16], uint8_t out[16]) { fe_store(out, fe_new(fe_load(v))); }
void or_fe_mul_vec(const uint8_t *a, const uint8_t *b, size_t n, uint8_t *out) {
    PAR_FOR for (size_t i = 0; i < n; i++) fe_store(out + 16 * i, fe_mul(fe_load(a + 16 * i), fe_load(b + 16 * i)));
}
void or_fe_add_vec(const uint8_t *a, const uint8_t *b, size_t n, uint8_t *out) {
    PAR_FOR for (size_t i = 0; i < n; i++) fe_store(out + 16 * i, fe_add(fe_load(a + 16 * i), fe_load(b + 16 * i)));
}
void or_fe_sub_vec(const uint8_t *a, const uint8_t *b, size_t n, uint8_t *out) {
    PAR_FOR for (size_t i = 0; i < n; i++) fe_store(out + 16 * i, fe_sub(fe_load(a + 16 * i), fe_load(b + 16 * i)));
}

static inline uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
/* synthetic inputs: element i = new(lo | hi<<64), lo = splitmix64(seed + 2i), hi = splitmix64(seed + 2i + 1) */
void or_synthetic_elements(uint64_t seed, size_t n, uint8_t *out) {
    PAR_FOR for (size_t i = 0; i < n; i++) {
        u128 v = (u128)splitmix64(seed + 2 * i) | ((u128)splitmix64(seed + 2 * i + 1) << 64);
        fe_store(out + 16 * i, fe_new(v));
    }
}

/* -------------------------------------------------------------------- NTT */
/* src/ntt/mod.rs:42-54 */
static int pow2_generator(uint64_t log_size, fe *out) {
    u128 m1 = FE_M - 1;
    unsigned max_log = 0;
    while (((m1 >> max_log) & 1) == 0) max_log++;
    if (log_size > max_log) return OR_ERR_RANGE;
    *out = fe_pow(fe_from_i64(3), m1 / ((u128)1 << log_size));
    return OR_OK;
}
int or_pow2_generator(uint64_t log_size, uint8_t out[16]) {
    fe g;
    int st = pow2_generator(log_size, &g);
    if (st == OR_OK) fe_store(out, g);
    return st;
}
/* src/ntt/mod.rs:18-28 — sequential running product; chunked when threaded */
static void powers_of(fe gen, size_t size, fe *out) {
    if (g_threads <= 1 || size < (1u << 14)) {
        fe cur = fe_from_i64(1);
        for (size_t i = 0; i < size; i++) { out[i] = cur; cur = fe_mul(cur, gen); }
        return;
    }
    size_t chunk = 1u << 12, nchunks = (size + chunk - 1) / chunk;
    PAR_FOR for (size_t c = 0; c < nchunks; c++) {
        size_t b = c * chunk, e = b + chunk < size ? b + chunk : size;
        fe cur = fe_pow(gen, (u128)b);
        for (size_t i = b; i < e; i++) { out[i] = cur; cur = fe_mul(cur, gen); }
    }
}
int or_pow2_generator_powers(uint64_t log_size, uint8_t *out) {
    fe g;
    int st = pow2_generator(log_size, &g);
    if (st != OR_OK) return st;
    powers_of(g, (size_t)1 << log_size, (fe *)out);
    return OR_OK;
}

/* src/ntt/mod.rs:113-123 */
static void bit_reverse_fe(fe *v, size_t n) {
    unsigned bits = ctz_sz(n);
    if (bits == 0 || bits >= 64) return;
    for (size_t i = 0; i < n; i++) {
        size_t j = (size_t)(bitrev64((uint64_t)i) >> (64 - bits));
        if (i < j) { fe t = v[i]; v[i] = v[j]; v[j] = t; }
    }
}
int or_bit_reverse_permutation(uint8_t *values, size_t n, size_t eb) {
    unsigned bits = ctz_sz(n);
    if (bits == 0 || bits >= 64) return OR_OK;
    uint8_t tmp[256];
    if (eb > sizeof tmp) return OR_ERR_SIZE;
    /* the reference uses trailing_zeros(n) bits even when n is not a power of two */
    for (size_t i = 0; i < n; i++) {
        size_t j = (size_t)(bitrev64((uint64_t)i) >> (64 - bits));
        if (i < j && j < n) {
            memcpy(tmp, values + i * eb, eb); memcpy(values + i * eb, values + j * eb, eb); memcpy(values + j * eb, tmp, eb);
        }
    }
    return OR_OK;
}

/* shared radix-2 DIT network of ntt (:76-109) and intt (:138-168) */
static void dit_network(fe *values, size_t n, fe gen) {
    bit_reverse_fe(values, n);
    if (n < 2) return;
    PAR_FOR for (size_t i = 0; i < n; i += 2) { /* :81-86 unrolled first step */
        fe u = values[i], v = values[i + 1];
        values[i] = fe_add(u, v);
        values[i + 1] = fe_sub(u, v);
    }
    fe *gen_pows = (fe *)malloc((n / 2 + 1) * sizeof(fe));
    for (size_t len = 4; len <= n; len *= 2) {
        fe current_gen = fe_pow(gen, (u128)(n / len)); /* :89 */
        size_t half = len / 2;
        powers_of(current_gen, half, gen_pows);         /* :90-97 */
        size_t total = n / 2;
        PAR_FOR for (size_t t = 0; t < total; t++) {    /* :98-105 */
            size_t i = (t / half) * len, j = t % half;
            fe v = fe_mul(values[i + j + half], gen_pows[j]);
            fe u = values[i + j];
            values[i + j] = fe_add(u, v);
            values[i + j + half] = fe_sub(u, v);
        }
    }
    free(gen_pows);
}
int or_ntt(const uint8_t *coeffs, size_t n, const uint8_t gen[16], uint8_t *evals) {
    if (!is_pow2(n)) return OR_ERR_NOT_POW2; /* :71-74 */
    if (evals != coeffs) memcpy(evals, coeffs, n * 16); /* :76 clone */
    dit_network((fe *)evals, n, fe_load(gen));
    return OR_OK;
}
int or_intt(const uint8_t *evals, size_t n, const uint8_t gen[16], uint8_t *coeffs) {
    if (!is_pow2(n)) return OR_ERR_NOT_POW2; /* :134 */
    if (coeffs != evals) memcpy(coeffs, evals, n * 16);
    fe gen_inv = fe_div(fe_from_i64(1), fe_load(gen)); /* :140 */
    dit_network((fe *)coeffs, n, gen_inv);
    fe n_inv = fe_div(fe_from_i64(1), fe_from_i64((int64_t)n)); /* :170 */
    fe *v = (fe *)coeffs;
    PAR_FOR for (size_t i = 0; i < n; i++) v[i] = fe_mul(v[i], n_inv); /* :171 */
    return OR_OK;
}
int or_poly_evaluate(const uint8_t *coeffs, size_t n, const uint8_t x[16], uint8_t out[16]) {
    fe acc = 0, xx = fe_load(x);
    for (size_t i = n; i-- > 0;) acc = fe_add(fe_mul(acc, xx), fe_load(coeffs + 16 * i));
    fe_store(out, acc);
    return OR_OK;
}
/* src/fri/mod.rs:19-28 */
int or_reed_solomon(const uint8_t *coeffs, size_t n, const uint8_t gen[16], uint8_t *code) {
    size_t blowup = (size_t)1 << OR_LOG_BLOWUP;
    if (!is_pow2(blowup * n)) return OR_ERR_NOT_POW2;
    memcpy(code, coeffs, n * 16);
    memset(code + n * 16, 0, (blowup - 1) * n * 16); /* :24 resize with zeros */
    dit_network((fe *)code, blowup * n, fe_load(gen));
    return OR_OK;
}

/* --------------------------------------------------- multilinear polynomials */
/* src/polynomials.rs:150-163 / :111-124 — n = trailing_zeros(len), loops j in 0..(1<<n) */
static void mobius(fe *c, size_t len, int subtract) {
    unsigned n = ctz_sz(len);
    if (n >= 64) return;
    size_t span = (size_t)1 << n;
    for (unsigned i = 0; i < n; i++) {
        size_t mask = (size_t)1 << i;
        PAR_FOR for (size_t j = 0; j < span; j++) {
            if (j & mask) c[j] = subtract ? fe_sub(c[j], c[j ^ mask]) : fe_add(c[j], c[j ^ mask]);
        }
    }
}
int or_mle_to_coefficient(const uint8_t *evals, size_t len, uint8_t *coeffs) {
    if (coeffs != evals) memcpy(coeffs, evals, len * 16);
    mobius((fe *)coeffs, len, 1);
    return OR_OK;
}
int or_mle_to_evaluation(const uint8_t *coeffs, size_t len, uint8_t *evals) {
    if (evals != coeffs) memcpy(evals, coeffs, len * 16);
    mobius((fe *)evals, len, 0);
    return OR_OK;
}
static size_t next_pow2(size_t n) { size_t p = 1; while (p < n) p <<= 1; return p; }
/* src/polynomials.rs:165-187 */
int or_mle_evals_evaluate(const uint8_t *evals, size_t len, const uint8_t *args, size_t n_args, uint8_t out[16]) {
    if (n_args >= 64 || ((size_t)1 << n_args) != next_pow2(len)) return OR_ERR_SIZE;
    const fe *e = (const fe *)evals, *a = (const fe *)args;
    fe one = fe_from_i64(1), acc = 0;
    int nt = g_threads > 1 ? g_threads : 1;
    fe *part = (fe *)calloc((size_t)nt, sizeof(fe));
#pragma omp parallel num_threads(nt) if (g_threads > 1)
    {
        int tid = 0;
#ifdef _OPENMP
        tid = omp_get_thread_num();
#endif
        fe s = 0;
#pragma omp for schedule(static)
        for (size_t pos = 0; pos < len; pos++) {
            fe term = e[pos];
            for (size_t b = 0; b < n_args; b++) { /* args.iter().rev().enumerate() */
                fe arg = a[n_args - 1 - b];
                term = fe_mul(term, ((pos >> b) & 1) ? arg : fe_sub(one, arg));
            }
            s = fe_add(s, term);
        }
        part[tid] = s;
    }
    for (int i = 0; i < nt; i++) acc = fe_add(acc, part[i]);
    free(part);
    fe_store(out, acc);
    return OR_OK;
}
/* src/polynomials.rs:126-146 */
int or_mle_coeffs_evaluate(const uint8_t *coeffs, size_t len, const uint8_t *args, size_t n_args, uint8_t out[16]) {
    if (n_args >= 64 || ((size_t)1 << n_args) != next_pow2(len)) return OR_ERR_SIZE;
    const fe *c = (const fe *)coeffs, *a = (const fe *)args;
    fe acc = 0;
    for (size_t pos = 0; pos < len; pos++) {
        fe term = c[pos];
        for (size_t b = 0; b < n_args; b++)
            if ((pos >> b) & 1) term = fe_mul(term, a[n_args - 1 - b]);
        acc = fe_add(acc, term);
    }
    fe_store(out, acc);
    return OR_OK;
}
/* src/polynomials.rs:51-98 — Lagrange interpolation over x = 0..n-1 with poly_mul */
static void interpolate(const fe *evals, size_t n, fe *coeffs) {
    fe *lj = (fe *)malloc((n + 1) * sizeof(fe)), *tmp = (fe *)malloc((n + 1) * sizeof(fe));
    for (size_t i = 0; i < n; i++) coeffs[i] = 0;
    for (size_t j = 0; j < n; j++) {
        size_t deg = 1; /* lj has `deg` coefficients */
        lj[0] = fe_from_i64(1);
        fe xj = fe_from_i64((int64_t)j), denom = fe_from_i64(1);
        for (size_t m = 0; m < n; m++) {
            if (m == j) continue;
            fe xm = fe_from_i64((int64_t)m);
            fe b0 = fe_neg(xm), b1 = fe_from_i64(1); /* (x - xm) */
            for (size_t i = 0; i <= deg; i++) tmp[i] = 0;
            for (size_t i = 0; i < deg; i++) {
                tmp[i] = fe_add(tmp[i], fe_mul(lj[i], b0));
                tmp[i + 1] = fe_add(tmp[i + 1], fe_mul(lj[i], b1));
            }
            deg++;
            memcpy(lj, tmp, deg * sizeof(fe));
            denom = fe_mul(denom, fe_sub(xj, xm));
        }
        fe scale = fe_div(evals[j], denom);
        for (size_t i = 0; i < n && i < deg; i++) coeffs[i] = fe_add(coeffs[i], fe_mul(scale, lj[i]));
    }
    free(lj); free(tmp);
}
int or_interpolate(const uint8_t *evals, size_t n, uint8_t *coeffs) {
    interpolate((const fe *)evals, n, (fe *)coeffs);
    return OR_OK;
}
static fe poly_eval(const fe *coeffs, size_t n, fe x) { /* src/polynomials.rs:9-14 */
    fe acc = 0;
    for (size_t i = n; i-- > 0;) acc = fe_add(fe_mul(acc, x), coeffs[i]);
    return acc;
}

/* ------------------------------------------------------------- transcript */
struct or_transcript { or_sha256_ctx s; };
void or_sha256_oneshot(const uint8_t *data, size_t len, uint8_t out[32]) { or_sha256(data, len, out); }
or_transcript *or_transcript_new(void) {
    or_transcript *t = (or_transcript *)malloc(sizeof *t);
    or_sha256_init(&t->s);
    return t;
}
or_transcript *or_transcript_clone(const or_transcript *t) {
    or_transcript *c = (or_transcript *)malloc(sizeof *c);
    *c = *t;
    return c;
}
void or_transcript_free(or_transcript *t) { free(t); }
void or_transcript_absorb(or_transcript *t, const uint8_t *bytes, size_t len) { or_sha256_update(&t->s, bytes, len); }
void or_transcript_random(const or_transcript *t, uint8_t out[32]) {
    or_sha256_ctx c = t->s; /* finalize a clone, src/transcript.rs:23-29 */
    or_sha256_final(&c, out);
}
static fe transcript_challenge(or_transcript *t) { /* src/transcript.rs:35-38 */
    uint8_t d[32];
    or_transcript_random(t, d);
    return fe_new(fe_load(d));
}
void or_transcript_next_challenge(or_transcript *t, uint8_t out[16]) { fe_store(out, transcript_challenge(t)); }
static void absorb_fe(or_transcript *t, fe x) { uint8_t b[16]; fe_store(b, x); or_transcript_absorb(t, b, 16); }

/* ----------------------------------------------------------------- Merkle */
struct or_merkle {
    size_t n_leaves, n_layers, item_bytes, n_batches; /* n_batches = 0 for Merkle<T> */
    uint8_t **layers;                                 /* layer l: (n_leaves >> l) digests */
    uint8_t **data;                                   /* 1 array, or n_batches arrays */
};
static void hash_node(const uint8_t *l, const uint8_t *r, uint8_t *out) { /* :184-189 */
    or_sha256_ctx c;
    or_sha256_init(&c);
    or_sha256_update(&c, l, 32);
    or_sha256_update(&c, r, 32);
    or_sha256_final(&c, out);
}
static void build_upper_layers(or_merkle *m) { /* :75-82 / :121-128 */
    size_t cnt = m->n_leaves;
    m->n_layers = 1;
    while (cnt > 1) {
        size_t nxt = cnt / 2;
        uint8_t *cur = m->layers[m->n_layers - 1], *out = (uint8_t *)malloc(nxt * 32);
        PAR_FOR for (size_t i = 0; i < nxt; i++) hash_node(cur + 64 * i, cur + 64 * i + 32, out + 32 * i);
        m->layers[m->n_layers++] = out;
        cnt = nxt;
    }
}
or_merkle *or_merkle_commit(const uint8_t *data, size_t item_bytes, size_t n_items) {
    if (!is_pow2(n_items)) return NULL; /* :66-69 */
    or_merkle *m = (or_merkle *)calloc(1, sizeof *m);
    m->n_leaves = n_items; m->item_bytes = item_bytes; m->n_batches = 0;
    m->layers = (uint8_t **)calloc(66, sizeof(uint8_t *));
    m->data = (uint8_t **)calloc(1, sizeof(uint8_t *));
    m->data[0] = (uint8_t *)malloc(n_items * item_bytes + 1);
    memcpy(m->data[0], data, n_items * item_bytes);
    m->layers[0] = (uint8_t *)malloc(n_items * 32);
    PAR_FOR for (size_t i = 0; i < n_items; i++) or_sha256(data + i * item_bytes, item_bytes, m->layers[0] + 32 * i); /* :71 hash_leaf */
    build_upper_layers(m);
    return m;
}
or_merkle *or_merkle_batch_commit(const uint8_t *const *data, size_t n_batches, size_t item_bytes, size_t n_items) {
    if (n_batches == 0 || !is_pow2(n_items)) return NULL; /* :94-99 */
    or_merkle *m = (or_merkle *)calloc(1, sizeof *m);
    m->n_leaves = n_items; m->item_bytes = item_bytes; m->n_batches = n_batches;
    m->layers = (uint8_t **)calloc(66, sizeof(uint8_t *));
    m->data = (uint8_t **)calloc(n_batches, sizeof(uint8_t *));
    for (size_t b = 0; b < n_batches; b++) {
        m->data[b] = (uint8_t *)malloc(n_items * item_bytes + 1);
        memcpy(m->data[b], data[b], n_items * item_bytes);
    }
    m->layers[0] = (uint8_t *)malloc(n_items * 32);
    PAR_FOR for (size_t i = 0; i < n_items; i++) { /* :110-116 */
        or_sha256_ctx c;
        or_sha256_init(&c);
        for (size_t b = 0; b < n_batches; b++) or_sha256_update(&c, data[b] + i * item_bytes, item_bytes);
        or_sha256_final(&c, m->layers[0] + 32 * i);
    }
    build_upper_layers(m);
    return m;
}
void or_merkle_free(or_merkle *m) {
    if (!m) return;
    for (size_t l = 0; l < m->n_layers; l++) free(m->layers[l]);
    size_t nd = m->n_batches ? m->n_batches : 1;
    for (size_t b = 0; b < nd; b++) free(m->data[b]);
    free(m->layers); free(m->data); free(m);
}
void or_merkle_root(const or_merkle *m, uint8_t out[32]) { memcpy(out, m->layers[m->n_layers - 1], 32); }
size_t or_merkle_num_layers(const or_merkle *m) { return m->n_layers; }
size_t or_merkle_layer_len(const or_merkle *m, size_t l) { return m->n_leaves >> l; }
void or_merkle_layer(const or_merkle *m, size_t l, uint8_t *out) { memcpy(out, m->layers[l], (m->n_leaves >> l) * 32); }
int or_merkle_open(const or_merkle *m, size_t index, uint8_t *value, uint8_t *digests, uint8_t *dirs, size_t *path_len) {
    if (index >= m->n_leaves) return OR_ERR_RANGE; /* :35-37 / :144-146 */
    if (m->n_batches == 0) memcpy(value, m->data[0] + index * m->item_bytes, m->item_bytes);
    else for (size_t b = 0; b < m->n_batches; b++) memcpy(value + b * m->item_bytes, m->data[b] + index * m->item_bytes, m->item_bytes);
    size_t cur = index, n = 0;
    for (size_t l = 0; l < m->n_layers; l++) { /* :43-55 */
        size_t sib; uint8_t dir;
        if (cur % 2 == 0) { sib = cur + 1; dir = 1; } else { sib = cur - 1; dir = 0; }
        if (sib >= (m->n_leaves >> l)) break;
        memcpy(digests + 32 * n, m->layers[l] + 32 * sib, 32);
        dirs[n++] = dir;
        cur /= 2;
    }
    *path_len = n;
    return OR_OK;
}
int or_merkle_path_verify(const uint8_t *value, size_t value_bytes, const uint8_t *digests, const uint8_t *dirs,
                          size_t path_len, const uint8_t root[32], size_t index) {
    uint8_t h[32], nx[32];
    or_sha256(value, value_bytes, h);
    size_t computed = 0;
    for (size_t i = 0; i < path_len; i++) {
        if (dirs[i] == 0) { computed += (size_t)1 << i; hash_node(digests + 32 * i, h, nx); }
        else hash_node(h, digests + 32 * i, nx);
        memcpy(h, nx, 32);
    }
    if (memcmp(h, root, 32) != 0) return OR_V_INCLUSION_HASH;
    if (computed != index) return OR_V_INCLUSION_INDEX;
    return OR_V_OK;
}

/* -------------------------------------------------------------------- FRI */
typedef struct { uint8_t *value; size_t value_bytes, path_len; uint8_t *digests, *dirs; } path_t;
static void path_free(path_t *p) { free(p->value); free(p->digests); free(p->dirs); }
static path_t path_open(const or_merkle *m, size_t index) {
    path_t p;
    p.value_bytes = (m->n_batches ? m->n_batches : 1) * m->item_bytes;
    p.value = (uint8_t *)malloc(p.value_bytes);
    p.digests = (uint8_t *)malloc(32 * 64);
    p.dirs = (uint8_t *)malloc(64);
    or_merkle_open(m, index, p.value, p.digests, p.dirs, &p.path_len);
    return p;
}
typedef struct { size_t n_paths; path_t *paths; } query_t;

struct or_fri { or_merkle **trees; size_t n_trees; int has_last; fe last; };
struct or_fri_proof {
    size_t n_commitments; uint8_t *commitments;
    size_t n_queries; query_t *queries;
    fe last_elem; uint8_t last_random[32];
};

/* src/fri/mod.rs:45-55 */
static or_merkle *commit_rs_code(const fe *code, size_t n) {
    size_t half = n / 2;
    fe *pairs = (fe *)malloc((2 * half + 1) * sizeof(fe));
    PAR_FOR for (size_t i = 0; i < half; i++) { pairs[2 * i] = code[i]; pairs[2 * i + 1] = code[i + half]; }
    or_merkle *m = or_merkle_commit((const uint8_t *)pairs, 32, half);
    free(pairs);
    return m;
}
static void fri_push(or_fri *f, or_merkle *m) {
    f->trees = (or_merkle **)realloc(f->trees, (f->n_trees + 1) * sizeof(or_merkle *));
    f->trees[f->n_trees++] = m;
}
or_fri *or_fri_init(const uint8_t *code, size_t n, or_transcript *t) {
    if (!is_pow2(n) || n < 2) return NULL; /* :60-63; n=1 panics inside Merkle::commit(empty) */
    or_fri *f = (or_fri *)calloc(1, sizeof *f);
    or_merkle *m = commit_rs_code((const fe *)code, n);
    uint8_t root[32];
    or_merkle_root(m, root);
    fri_push(f, m);
    or_transcript_absorb(t, root, 32); /* :71 */
    return f;
}
/* the common tail of fold_step (:116-133) and batched_fold_step (batched_fri.rs:152-180) */
static int fold_finish(or_fri *f, fe *next, size_t half_n, or_transcript *t) {
    size_t blowup = (size_t)1 << OR_LOG_BLOWUP;
    if (half_n == blowup) {
        for (size_t i = 0; i < half_n; i++)
            if (next[i] != next[0]) return OR_ERR_NOT_RS; /* assert "not an RS code" */
        f->last = next[0]; f->has_last = 1;
        absorb_fe(t, next[0]);
        return OR_OK;
    }
    or_merkle *m = commit_rs_code(next, half_n);
    uint8_t root[32];
    or_merkle_root(m, root);
    fri_push(f, m);
    or_transcript_absorb(t, root, 32);
    return OR_OK;
}
int or_fri_fold_step(or_fri *f, const uint8_t *gen_pows_b, size_t gen_pows_len, size_t k, const uint8_t r_b[16], or_transcript *t) {
    const or_merkle *lastm = f->trees[f->n_trees - 1];
    const fe *last = (const fe *)lastm->data[0]; /* pairs: [2i]=value, [2i+1]=minus_value (:80) */
    size_t n = lastm->n_leaves * 2, blowup = (size_t)1 << OR_LOG_BLOWUP;
    if (n <= blowup) return OR_OK; /* :83-85 */
    size_t half_n = n >> 1;
    const fe *gen_pows = (const fe *)gen_pows_b;
    fe r = fe_load(r_b);
    fe *next = (fe *)malloc(half_n * sizeof(fe));
    fe half = fe_div(fe_from_i64(1), fe_from_i64(2)); /* :90 */
    {
        fe a = last[0], b = last[1]; /* :93-95 */
        next[0] = fe_mul(fe_add(fe_add(a, b), fe_mul(r, fe_sub(a, b))), half);
    }
    PAR_FOR for (size_t i = 1; i < half_n; i++) { /* :96-114 */
        fe a = last[2 * i], b = last[2 * i + 1];
        fe even = fe_add(a, b);
        size_t gen_pow_index = i * ((size_t)1 << k);
        fe odd = fe_mul(fe_sub(a, b), gen_pows[gen_pows_len - gen_pow_index]);
        next[i] = fe_mul(fe_add(even, fe_mul(r, odd)), half);
    }
    int st = fold_finish(f, next, half_n, t);
    free(next);
    return st;
}
or_fri *or_fri_fold(const uint8_t *gen_pows, size_t gen_pows_len, const uint8_t *code, size_t n, or_transcript *t, int *status) {
    *status = OR_OK;
    or_fri *f = or_fri_init(code, n, t);
    if (!f) { *status = OR_ERR_NOT_POW2; return NULL; }
    size_t num_steps = ctz_sz(n) - OR_LOG_BLOWUP; /* :138 */
    for (size_t k = 0; k < num_steps; k++) {
        uint8_t r[16];
        or_transcript_next_challenge(t, r); /* :140 */
        int st = or_fri_fold_step(f, gen_pows, gen_pows_len, k, r, t);
        if (st != OR_OK) { *status = st; or_fri_free(f); return NULL; }
    }
    if (!f->has_last) { *status = OR_ERR_SIZE; or_fri_free(f); return NULL; } /* :143 assert */
    return f;
}
void or_fri_free(or_fri *f) {
    if (!f) return;
    for (size_t i = 0; i < f->n_trees; i++) or_merkle_free(f->trees[i]);
    free(f->trees); free(f);
}
size_t or_fri_num_trees(const or_fri *f) { return f->n_trees; }
const or_merkle *or_fri_tree(const or_fri *f, size_t i) { return f->trees[i]; }
void or_fri_tree_data(const or_fri *f, size_t i, uint8_t *out) { memcpy(out, f->trees[i]->data[0], f->trees[i]->n_leaves * 32); }
void or_fri_fold_roots(const or_fri *f, uint8_t *out) { for (size_t i = 0; i < f->n_trees; i++) or_merkle_root(f->trees[i], out + 32 * i); }
int or_fri_last_element(const or_fri *f, uint8_t out[16]) { if (f->has_last) fe_store(out, f->last); return f->has_last; }

/* src/fri/mod.rs:154-174 */
static query_t fri_open_query_at(const or_fri *f, size_t index) {
    query_t q;
    q.n_paths = f->n_trees;
    q.paths = (path_t *)calloc(f->n_trees ? f->n_trees : 1, sizeof(path_t));
    size_t cur = index, cur_n = f->n_trees ? f->trees[0]->n_leaves : 0;
    for (size_t j = 0; j < f->n_trees; j++) {
        q.paths[j] = path_open(f->trees[j], cur);
        cur_n /= 2;
        if (cur_n) cur %= cur_n;
    }
    return q;
}
static size_t next_query_index(or_transcript *t, size_t domain_size) { /* :269-271 */
    uint8_t d[32];
    or_transcript_random(t, d);
    uint64_t v;
    memcpy(&v, d, 8);
    return (size_t)(v % (uint64_t)(domain_size / 2));
}
static void absorb_index(or_transcript *t, size_t idx) { uint64_t v = idx; or_transcript_absorb(t, (const uint8_t *)&v, 8); } /* :276 usize LE */

static or_fri_proof *assemble_fri_proof(const or_fri *f, size_t domain_size, or_transcript *t) {
    or_fri_proof *p = (or_fri_proof *)calloc(1, sizeof *p);
    p->n_queries = OR_NUM_QUERIES;
    p->queries = (query_t *)calloc(OR_NUM_QUERIES, sizeof(query_t));
    for (size_t q = 0; q < OR_NUM_QUERIES; q++) { /* :268-277 */
        size_t idx = next_query_index(t, domain_size);
        p->queries[q] = fri_open_query_at(f, idx);
        absorb_index(t, idx);
    }
    p->n_commitments = f->n_trees;
    p->commitments = (uint8_t *)malloc(32 * (f->n_trees + 1));
    or_fri_fold_roots(f, p->commitments);
    p->last_elem = f->last;
    or_transcript_random(t, p->last_random);
    return p;
}
or_fri_proof *or_fri_prove(const uint8_t *code, size_t n, const uint8_t *gen_pows, size_t gen_pows_len, or_transcript *t, int *status) {
    or_fri *f = or_fri_fold(gen_pows, gen_pows_len, code, n, t, status);
    if (!f) return NULL;
    or_fri_proof *p = assemble_fri_proof(f, n, t);
    or_fri_free(f);
    return p;
}
void or_fri_proof_free(or_fri_proof *p) {
    if (!p) return;
    for (size_t q = 0; q < p->n_queries; q++) {
        for (size_t j = 0; j < p->queries[q].n_paths; j++) path_free(&p->queries[q].paths[j]);
        free(p->queries[q].paths);
    }
    free(p->queries); free(p->commitments); free(p);
}
size_t or_fri_proof_num_commitments(const or_fri_proof *p) { return p->n_commitments; }
void or_fri_proof_commitments(const or_fri_proof *p, uint8_t *out) { memcpy(out, p->commitments, 32 * p->n_commitments); }
void or_fri_proof_last(const or_fri_proof *p, uint8_t last_elem[16], uint8_t last_random[32]) {
    fe_store(last_elem, p->last_elem);
    memcpy(last_random, p->last_random, 32);
}

/* QueryProof::verify, src/fri/mod.rs:184-236 */
static int query_verify(const query_t *q, const uint8_t *commitments, size_t n_commitments, fe last_element, size_t n,
                        size_t index, fe gen, const fe *random_elements) {
    if (q->n_paths != n_commitments) return OR_V_WRONG_NUM_PATHS;
    size_t cur_n = n, cur_idx = index;
    fe cur_gen = gen, two = fe_from_i64(2);
    for (size_t i = 0; i < q->n_paths; i++) {
        const path_t *p = &q->paths[i];
        int st = or_merkle_path_verify(p->value, p->value_bytes, p->digests, p->dirs, p->path_len, commitments + 32 * i, cur_idx);
        if (st != OR_V_OK) return st;
        fe value = fe_load(p->value), minus_value = fe_load(p->value + 16);
        fe gp = fe_pow(cur_gen, (u128)cur_idx);
        fe even = fe_div(fe_add(value, minus_value), two);
        fe odd = fe_div(fe_sub(value, minus_value), fe_mul(two, gp));
        fe expect = fe_add(even, fe_mul(random_elements[i], odd));
        if (i == q->n_paths - 1) {
            if (last_element != expect) return OR_V_QUERY_MISMATCH;
            break;
        }
        size_t next_idx = cur_idx % (cur_n / 2);
        const path_t *np = &q->paths[i + 1];
        fe next_value = next_idx == cur_idx ? fe_load(np->value) : fe_load(np->value + 16);
        if (next_value != expect) return OR_V_QUERY_MISMATCH;
        cur_gen = fe_mul(cur_gen, cur_gen);
        cur_n /= 2;
        cur_idx = next_idx;
    }
    return OR_V_OK;
}
/* FriProof::verify_queries, src/fri/mod.rs:311-340 */
static int fri_verify_queries(const or_fri_proof *p, or_transcript *t, const fe *random_elements) {
    size_t log_domain = p->n_commitments + OR_LOG_BLOWUP, domain = (size_t)1 << log_domain;
    fe gen;
    if (pow2_generator(log_domain, &gen) != OR_OK) return OR_V_QUERY_MISMATCH;
    for (size_t q = 0; q < p->n_queries; q++) {
        size_t n = domain / 2;
        size_t idx = next_query_index(t, domain);
        absorb_index(t, idx);
        int st = query_verify(&p->queries[q], p->commitments, p->n_commitments, p->last_elem, n, idx, gen, random_elements);
        if (st != OR_V_OK) return st;
    }
    uint8_t lr[32];
    or_transcript_random(t, lr);
    return memcmp(lr, p->last_random, 32) == 0 ? OR_V_OK : OR_V_LAST_RANDOM;
}
int or_fri_verify(const or_fri_proof *p) { /* :287-309 */
    if (p->n_queries != OR_NUM_QUERIES) return OR_V_WRONG_NUM_QUERIES;
    or_transcript *t = or_transcript_new();
    fe *rs = (fe *)malloc((p->n_commitments + 1) * sizeof(fe));
    for (size_t i = 0; i < p->n_commitments; i++) {
        or_transcript_absorb(t, p->commitments + 32 * i, 32);
        rs[i] = transcript_challenge(t);
    }
    absorb_fe(t, p->last_elem);
    int st = fri_verify_queries(p, t, rs);
    free(rs);
    or_transcript_free(t);
    return st;
}

/* --- wire format: bincode 2 `standard().with_little_endian().with_fixed_int_encoding()` through serde
 * (src/fri/mod.rs:367-369): Vec -> u64 len + items; Field128 -> serialize_bytes -> u64(16) + 16 bytes
 * (src/field.rs:40-48); HashDigest (GenericArray, serde tuple) and [u8;32] -> 32 raw bytes; Direction -> u32. */
typedef struct { uint8_t *p; size_t n; } wr_t;
static void w_bytes(wr_t *w, const void *b, size_t n) { if (w->p) memcpy(w->p + w->n, b, n); w->n += n; }
static void w_u64(wr_t *w, uint64_t v) { w_bytes(w, &v, 8); }
static void w_u32(wr_t *w, uint32_t v) { w_bytes(w, &v, 4); }
static void w_fe_bytes(wr_t *w, const uint8_t *b) { w_u64(w, 16); w_bytes(w, b, 16); }
static void w_pair(wr_t *w, const uint8_t *pair) { w_fe_bytes(w, pair); w_fe_bytes(w, pair + 16); }
static void w_path_tail(wr_t *w, const path_t *p) {
    w_u64(w, p->path_len);
    for (size_t i = 0; i < p->path_len; i++) { w_bytes(w, p->digests + 32 * i, 32); w_u32(w, p->dirs[i]); }
}
static void w_query(wr_t *w, const query_t *q) {
    w_u64(w, q->n_paths);
    for (size_t j = 0; j < q->n_paths; j++) { w_pair(w, q->paths[j].value); w_path_tail(w, &q->paths[j]); }
}
static void fri_proof_write(const or_fri_proof *p, wr_t *w) {
    w_u64(w, p->n_commitments);
    w_bytes(w, p->commitments, 32 * p->n_commitments);
    w_u64(w, p->n_queries);
    for (size_t q = 0; q < p->n_queries; q++) w_query(w, &p->queries[q]);
    uint8_t le[16];
    fe_store(le, p->last_elem);
    w_fe_bytes(w, le);
    w_bytes(w, p->last_random, 32);
}
size_t or_fri_proof_serialized_len(const or_fri_proof *p) { wr_t w = {NULL, 0}; fri_proof_write(p, &w); return w.n; }
void or_fri_proof_serialize(const or_fri_proof *p, uint8_t *out) { wr_t w = {out, 0}; fri_proof_write(p, &w); }

/* --------------------------------------------------------------- sumcheck */
struct or_sumcheck { fe *matrix, *delta; size_t width, height; };
/* Mask::evaluate, src/constraint_system/evaluation.rs:56-73 */
static fe mask_evaluate(size_t index, size_t n_vars, const fe *points) {
    fe one = fe_from_i64(1), prod = fe_from_i64(1);
    for (size_t i = 0; i < n_vars; i++) {
        fe point = points[n_vars - 1 - i];
        prod = fe_mul(prod, ((index >> i) & 1) ? point : fe_sub(one, point));
    }
    return prod;
}
or_sumcheck *or_sumcheck_build_tables_for_pcs(const uint8_t *inputs, size_t n_vars, const uint8_t *evals, size_t height) {
    if (n_vars >= 64 || ((size_t)1 << n_vars) != height) return NULL; /* :131 */
    or_sumcheck *s = (or_sumcheck *)calloc(1, sizeof *s);
    s->width = 1; s->height = height;
    s->matrix = (fe *)malloc(height * sizeof(fe));
    s->delta = (fe *)malloc(height * sizeof(fe));
    memcpy(s->matrix, evals, height * 16); /* :132 */
    const fe *pts = (const fe *)inputs;
    PAR_FOR for (size_t idx = 0; idx < height; idx++) s->delta[idx] = mask_evaluate(idx, n_vars, pts); /* :133-138 */
    return s;
}
void or_sumcheck_free(or_sumcheck *s) { if (s) { free(s->matrix); free(s->delta); free(s); } }
size_t or_sumcheck_height(const or_sumcheck *s) { return s->height; }
void or_sumcheck_tables(const or_sumcheck *s, uint8_t *m, uint8_t *d) {
    memcpy(m, s->matrix, s->height * 16);
    memcpy(d, s->delta, s->height * 16);
}
/* :204-232 with width 1 and composition |x| x[0] (multilinear_pcs.rs:56) */
static fe partial_sum(const or_sumcheck *s, fe r) {
    size_t offset = s->height >> 1;
    fe one = fe_from_i64(1), sm1 = fe_sub(one, r), acc = 0;
    int is_one = (r == one);
    int nt = g_threads > 1 ? g_threads : 1;
    fe *part = (fe *)calloc((size_t)nt, sizeof(fe));
#pragma omp parallel num_threads(nt) if (g_threads > 1)
    {
        int tid = 0;
#ifdef _OPENMP
        tid = omp_get_thread_num();
#endif
        fe a = 0;
#pragma omp for schedule(static)
        for (size_t i = 0; i < offset; i++) {
            fe d, m;
            if (is_one) {
                d = fe_mul(r, s->delta[i + offset]);
                m = fe_mul(r, s->matrix[i + offset]);
            } else {
                d = fe_add(fe_mul(sm1, s->delta[i]), fe_mul(r, s->delta[i + offset]));
                m = fe_add(fe_mul(sm1, s->matrix[i]), fe_mul(r, s->matrix[i + offset]));
            }
            a = fe_add(a, fe_mul(m, d));
        }
        part[tid] = a;
    }
    for (int i = 0; i < nt; i++) acc = fe_add(acc, part[i]);
    free(part);
    return acc;
}
void or_sumcheck_partial_sum(const or_sumcheck *s, const uint8_t r[16], uint8_t out[16]) { fe_store(out, partial_sum(s, fe_load(r))); }
static void sumcheck_fold(or_sumcheck *s, fe r) { /* :234-247 */
    s->height >>= 1;
    size_t offset = s->height;
    fe sm1 = fe_sub(fe_from_i64(1), r);
    PAR_FOR for (size_t i = 0; i < offset; i++) {
        s->delta[i] = fe_add(fe_mul(sm1, s->delta[i]), fe_mul(r, s->delta[i + offset]));
        s->matrix[i] = fe_add(fe_mul(sm1, s->matrix[i]), fe_mul(r, s->matrix[i + offset]));
    }
}
void or_sumcheck_fold(or_sumcheck *s, const uint8_t r[16]) { sumcheck_fold(s, fe_load(r)); }
/* :174-202 */
static fe sumcheck_round(or_sumcheck *s, size_t total_degree, fe *previous_sum, or_transcript *t, fe *nonzero_out) {
    size_t np = total_degree + 1;
    fe *evals = (fe *)calloc(np, sizeof(fe)), *coeffs = (fe *)calloc(np, sizeof(fe));
    for (size_t i = 1; i < np; i++) evals[i] = partial_sum(s, fe_from_i64((int64_t)i)); /* :185-187 */
    evals[0] = fe_sub(*previous_sum, evals[1]);                                          /* :188 */
    interpolate(evals, np, coeffs);                                                       /* :189-192 */
    for (size_t i = 1; i < np; i++) { nonzero_out[i - 1] = coeffs[i]; absorb_fe(t, coeffs[i]); } /* :193-197 */
    fe r = transcript_challenge(t);                                                       /* :198 */
    *previous_sum = poly_eval(coeffs, np, r);                                             /* :199 */
    sumcheck_fold(s, r);                                                                  /* :200 */
    free(evals); free(coeffs);
    return r;
}
int or_sumcheck_compute_polynomial(or_sumcheck *s, size_t total_degree, uint8_t previous_sum[16], or_transcript *t,
                                   uint8_t *nonzero_coeffs_out, uint8_t r_out[16]) {
    if (total_degree == 0) return OR_ERR_SIZE; /* :188 indexes evals[1] */
    fe prev = fe_load(previous_sum);
    fe r = sumcheck_round(s, total_degree, &prev, t, (fe *)nonzero_coeffs_out);
    fe_store(previous_sum, prev);
    fe_store(r_out, r);
    return OR_OK;
}
void or_sumcheck_compute_polynomials(or_sumcheck *s, size_t composition_degree, or_transcript *t, const uint8_t sum[16],
                                     uint8_t *coeffs_out, uint8_t *randoms_out) { /* :147-172 */
    fe prev = fe_load(sum);
    size_t total_degree = composition_degree + 1, n_rounds = ctz_sz(s->height);
    for (size_t k = 0; k < n_rounds; k++) {
        fe r = sumcheck_round(s, total_degree, &prev, t, (fe *)coeffs_out + k * total_degree);
        fe_store(randoms_out + 16 * k, r);
    }
}
/* ---------------------------------------------------------- width-w sumcheck tables (System path)
 * SumcheckTables with an arbitrary trace width (src/constraint_system/sumcheck.rs:10-15, System::build_tables :22-38,
 * partial_sum :204-232, fold :234-247, compute_sumcheck_polynomial(s) :147-202).  The reference passes the composition as a
 * Rust closure (`&impl Fn(&[F]) -> F`, :176; System::evaluate_composition, evaluation.rs:5-12 = sum_k mask_k * expr_k(row)).
 * A closure cannot cross a C ABI, so a composition is given as the sparse polynomial it computes over the row:
 *     comp(x) = sum_t coef[t] * prod_{k < len[t]} x[cols[off[t] + k]]       (len[t] = 0: the constant coef[t]) */
struct or_wsumcheck {
    fe *matrix, *delta;
    size_t width, height;
    size_t n_terms;
    fe *coef;
    uint32_t *len, *off, *cols;
};
or_wsumcheck *or_wsumcheck_build(const uint8_t *row_point, size_t n_vars, const uint8_t *matrix, size_t width, size_t height) {
    if (n_vars >= 64 || ((size_t)1 << n_vars) != height || width == 0) return NULL;
    or_wsumcheck *s = (or_wsumcheck *)calloc(1, sizeof *s);
    s->width = width; s->height = height;
    s->matrix = (fe *)malloc(height * width * sizeof(fe));
    s->delta = (fe *)malloc(height * sizeof(fe));
    memcpy(s->matrix, matrix, height * width * 16);                                          /* :33 */
    const fe *pts = (const fe *)row_point;
    PAR_FOR for (size_t idx = 0; idx < height; idx++) s->delta[idx] = mask_evaluate(idx, n_vars, pts); /* :26-31 */
    return s;
}
void or_wsumcheck_free(or_wsumcheck *s) {
    if (s) { free(s->matrix); free(s->delta); free(s->coef); free(s->len); free(s->off); free(s->cols); free(s); }
}
size_t or_wsumcheck_height(const or_wsumcheck *s) { return s->height; }
void or_wsumcheck_tables(const or_wsumcheck *s, uint8_t *m, uint8_t *d) {
    memcpy(m, s->matrix, s->height * s->width * 16);
    memcpy(d, s->delta, s->height * 16);
}
int or_wsumcheck_set_composition(or_wsumcheck *s, size_t n_terms, const uint8_t *coefs, const uint32_t *term_lens, const uint32_t *term_cols) {
    size_t total = 0;
    for (size_t t = 0; t < n_terms; t++) {
        for (uint32_t k = 0; k < term_lens[t]; k++) if (term_cols[total + k] >= s->width) return 1;
        total += term_lens[t];
    }
    free(s->coef); free(s->len); free(s->off); free(s->cols);
    s->n_terms = n_terms;
    s->coef = (fe *)malloc((n_terms ? n_terms : 1) * sizeof(fe));
    s->len = (uint32_t *)malloc((n_terms ? n_terms : 1) * sizeof(uint32_t));
    s->off = (uint32_t *)malloc((n_terms ? n_terms : 1) * sizeof(uint32_t));
    s->cols = (uint32_t *)malloc((total ? total : 1) * sizeof(uint32_t));
    memcpy(s->coef, coefs, n_terms * 16);
    memcpy(s->len, term_lens, n_terms * sizeof(uint32_t));
    memcpy(s->cols, term_cols, total * sizeof(uint32_t));
    uint32_t o = 0;
    for (size_t t = 0; t < n_terms; t++) { s->off[t] = o; o += term_lens[t]; }
    return 0;
}
static fe wcomposition(const or_wsumcheck *s, const fe *row) {
    fe acc = 0;
    for (size_t t = 0; t < s->n_terms; t++) {
        fe p = s->coef[t];
        for (uint32_t k = 0; k < s->len[t]; k++) p = fe_mul(p, row[s->cols[s->off[t] + k]]);
        acc = fe_add(acc, p);
    }
    return acc;
}
static fe wpartial_sum(const or_wsumcheck *s, fe r) { /* :204-232 */
    size_t offset = s->height >> 1, w = s->width;
    fe one = fe_from_i64(1), sm1 = fe_sub(one, r), acc = 0;
    int is_one = (r == one);
    fe *row = (fe *)malloc(w * sizeof(fe));
    for (size_t i = 0; i < offset; i++) {
        fe d;
        if (is_one) {
            d = fe_mul(r, s->delta[i + offset]);
            for (size_t j = 0; j < w; j++) row[j] = fe_mul(r, s->matrix[(i + offset) * w + j]);
        } else {
            d = fe_add(fe_mul(sm1, s->delta[i]), fe_mul(r, s->delta[i + offset]));
            for (size_t j = 0; j < w; j++) row[j] = fe_add(fe_mul(sm1, s->matrix[i * w + j]), fe_mul(r, s->matrix[(i + offset) * w + j]));
        }
        acc = fe_add(acc, fe_mul(wcomposition(s, row), d));
    }
    free(row);
    return acc;
}
void or_wsumcheck_partial_sum(const or_wsumcheck *s, const uint8_t r[16], uint8_t out[16]) { fe_store(out, wpartial_sum(s, fe_load(r))); }
static void wfold(or_wsumcheck *s, fe r) { /* :234-247 */
    s->height >>= 1;
    size_t offset = s->height, w = s->width;
    fe sm1 = fe_sub(fe_from_i64(1), r);
    for (size_t i = 0; i < offset; i++) {
        s->delta[i] = fe_add(fe_mul(sm1, s->delta[i]), fe_mul(r, s->delta[i + offset]));
        for (size_t j = 0; j < w; j++)
            s->matrix[i * w + j] = fe_add(fe_mul(sm1, s->matrix[i * w + j]), fe_mul(r, s->matrix[(i + offset) * w + j]));
    }
}
void or_wsumcheck_fold(or_wsumcheck *s, const uint8_t r[16]) { wfold(s, fe_load(r)); }
void or_wsumcheck_compute_polynomials(or_wsumcheck *s, size_t composition_degree, or_transcript *t, const uint8_t sum[16],
                                      uint8_t *coeffs_out, uint8_t *randoms_out) { /* :147-202 */
    fe prev = fe_load(sum);
    size_t total_degree = composition_degree + 1, np = total_degree + 1, n_rounds = ctz_sz(s->height);
    fe *evals = (fe *)calloc(np, sizeof(fe)), *coeffs = (fe *)calloc(np, sizeof(fe));
    for (size_t k = 0; k < n_rounds; k++) {
        for (size_t i = 1; i < np; i++) evals[i] = wpartial_sum(s, fe_from_i64((int64_t)i));
        evals[0] = fe_sub(prev, evals[1]);
        interpolate(evals, np, coeffs);
        for (size_t i = 1; i < np; i++) { fe_store(coeffs_out + 16 * (k * total_degree + i - 1), coeffs[i]); absorb_fe(t, coeffs[i]); }
        fe r = transcript_challenge(t);
        prev = poly_eval(coeffs, np, r);
        wfold(s, r);
        fe_store(randoms_out + 16 * k, r);
    }
    free(evals); free(coeffs);
}
/* Trace::evaluate (evaluation.rs:33-48): res[j] = sum_index Mask(index)(points) * matrix[index][j] */
void or_trace_evaluate(const uint8_t *matrix, size_t width, size_t height, const uint8_t *points, uint8_t *out) {
    size_t n_vars = ctz_sz(height);
    const fe *m = (const fe *)matrix, *pts = (const fe *)points;
    for (size_t j = 0; j < width; j++) fe_store(out + 16 * j, 0);
    fe *res = (fe *)calloc(width, sizeof(fe));
    for (size_t index = 0; index < height; index++) {
        fe c = mask_evaluate(index, n_vars, pts);
        for (size_t j = 0; j < width; j++) res[j] = fe_add(res[j], fe_mul(c, m[index * width + j]));
    }
    for (size_t j = 0; j < width; j++) fe_store(out + 16 * j, res[j]);
    free(res);
}
/* Mask::evaluate for one index (evaluation.rs:56-73): used for System's constraint_mask (system.rs:91-93) */
void or_mask_evaluate(size_t index, size_t n_vars, const uint8_t *points, uint8_t out[16]) {
    fe_store(out, mask_evaluate(index, n_vars, (const fe *)points));
}

/* Delta::evaluate, src/constraint_system/evaluation.rs:80-90 */
static fe delta_evaluate(const fe *data, const fe *points, size_t n) {
    fe one = fe_from_i64(1), prod = fe_from_i64(1);
    for (size_t i = 0; i < n; i++) {
        fe a = data[i], b = points[i];
        prod = fe_mul(prod, fe_add(fe_mul(a, b), fe_mul(fe_sub(one, a), fe_sub(one, b))));
    }
    return prod;
}
void or_delta_evaluate(const uint8_t *data, const uint8_t *points, size_t n, uint8_t out[16]) {
    fe_store(out, delta_evaluate((const fe *)data, (const fe *)points, n));
}
/* SumcheckPolynomial::to_polynomial (:269-276): returns total_degree+1 coefficients */
static void to_polynomial(const fe *nonzero, size_t deg, fe sum, fe *coeffs) {
    fe sc = 0;
    for (size_t i = 0; i < deg; i++) sc = fe_add(sc, nonzero[i]);
    coeffs[0] = fe_div(fe_sub(sum, sc), fe_from_i64(2));
    for (size_t i = 0; i < deg; i++) coeffs[i + 1] = nonzero[i];
}

/* ---------------------------------------------------------- multilinear PCS */
struct or_pcs_proof { or_fri_proof *fri; size_t n_rounds; fe *sc; fe *inputs; size_t n_inputs; fe output; };

/* evals -> to_coefficient -> bit reverse -> reed_solomon (multilinear_pcs.rs:101-107, batched_pcs.rs:144-148) */
static fe *encode_poly(const uint8_t *evals, size_t n, fe gen) {
    fe *coeffs = (fe *)malloc(n * sizeof(fe));
    memcpy(coeffs, evals, n * 16);
    mobius(coeffs, n, 1);
    bit_reverse_fe(coeffs, n);
    fe *code = (fe *)malloc(2 * n * sizeof(fe));
    uint8_t g[16];
    fe_store(g, gen);
    or_reed_solomon((const uint8_t *)coeffs, n, g, (uint8_t *)code);
    free(coeffs);
    return code;
}

or_pcs_proof *or_pcs_prove(const uint8_t *inputs, size_t n_vars, const uint8_t output[16], const uint8_t *evals, size_t n,
                           or_transcript *t, int *status) {
    *status = OR_OK;
    if (!is_pow2(n) || n < 2 || ((size_t)1 << n_vars) != n) { *status = OR_ERR_SIZE; return NULL; }
    size_t log_domain = ctz_sz(n) + OR_LOG_BLOWUP, domain = (size_t)1 << log_domain; /* :97 */
    fe *gen_pows = (fe *)malloc(domain * sizeof(fe));
    if (or_pow2_generator_powers(log_domain, (uint8_t *)gen_pows) != OR_OK) { free(gen_pows); *status = OR_ERR_RANGE; return NULL; }
    fe gen = gen_pows[1];
    fe *code = encode_poly(evals, n, gen);
    /* PCSProverData::fold (:43-76) */
    or_fri *f = or_fri_init((const uint8_t *)code, domain, t);
    or_sumcheck *sc = or_sumcheck_build_tables_for_pcs(inputs, n_vars, evals, n);
    size_t num_steps = ctz_sz(domain) - OR_LOG_BLOWUP;
    or_pcs_proof *p = (or_pcs_proof *)calloc(1, sizeof *p);
    p->n_rounds = num_steps;
    p->sc = (fe *)malloc(2 * num_steps * sizeof(fe) + 16);
    fe prev = fe_load(output);
    for (size_t k = 0; k < num_steps; k++) {
        fe r = sumcheck_round(sc, 2, &prev, t, p->sc + 2 * k); /* :61-66 */
        uint8_t rb[16];
        fe_store(rb, r);
        int st = or_fri_fold_step(f, (const uint8_t *)gen_pows, domain, k, rb, t); /* :72 */
        if (st != OR_OK) { *status = st; break; }
    }
    if (*status == OR_OK && !f->has_last) *status = OR_ERR_SIZE;
    if (*status == OR_OK) {
        p->fri = assemble_fri_proof(f, domain, t); /* :113-129 */
        p->n_inputs = n_vars;
        p->inputs = (fe *)malloc(n_vars * sizeof(fe) + 16);
        memcpy(p->inputs, inputs, n_vars * 16);
        p->output = fe_load(output);
    }
    or_fri_free(f); or_sumcheck_free(sc); free(code); free(gen_pows);
    if (*status != OR_OK) { or_pcs_proof_free(p); return NULL; }
    return p;
}
void or_pcs_proof_free(or_pcs_proof *p) { if (p) { or_fri_proof_free(p->fri); free(p->sc); free(p->inputs); free(p); } }
const or_fri_proof *or_pcs_proof_fri(const or_pcs_proof *p) { return p->fri; }
size_t or_pcs_proof_num_rounds(const or_pcs_proof *p) { return p->n_rounds; }
void or_pcs_proof_sumcheck_coeffs(const or_pcs_proof *p, uint8_t *out) { memcpy(out, p->sc, p->n_rounds * 32); }

/* the sumcheck replay shared by PCSProof::verify (:169-184) and BatchedPCSProof::verify (batched_pcs.rs:225-247) */
static int sumcheck_replay(const fe *sc, size_t n_rounds, fe sum, const fe *inputs, const fe *rs, fe last_elem) {
    fe pol[3];
    to_polynomial(sc, 2, sum, pol);
    for (size_t i = 1; i < n_rounds; i++) to_polynomial(sc + 2 * i, 2, poly_eval(pol, 3, rs[i - 1]), pol);
    fe r = rs[n_rounds - 1];
    fe delta = delta_evaluate(inputs, rs, n_rounds);
    return fe_mul(delta, last_elem) == poly_eval(pol, 3, r) ? OR_V_OK : OR_V_SUMCHECK;
}
int or_pcs_verify(const or_pcs_proof *p, or_transcript *t) { /* :138-190 */
    const or_fri_proof *fp = p->fri;
    if (fp->n_queries != OR_NUM_QUERIES) return OR_V_WRONG_NUM_QUERIES;
    size_t n = fp->n_commitments;
    if (n != p->n_rounds || n != p->n_inputs || n == 0) return OR_ERR_SIZE;
    fe *rs = (fe *)malloc(n * sizeof(fe));
    for (size_t i = 0; i < n; i++) {
        or_transcript_absorb(t, fp->commitments + 32 * i, 32);
        absorb_fe(t, p->sc[2 * i]);
        absorb_fe(t, p->sc[2 * i + 1]);
        rs[i] = transcript_challenge(t);
    }
    absorb_fe(t, fp->last_elem);
    int st = sumcheck_replay(p->sc, n, p->output, p->inputs, rs, fp->last_elem);
    if (st == OR_V_OK) st = fri_verify_queries(fp, t, rs);
    free(rs);
    return st;
}

/* ------------------------------------------------------------ batched FRI */
void or_fingerprint(const uint8_t r_b[16], const uint8_t *coeffs, size_t n, uint8_t out[16]) { /* batched_fri.rs:30-38 */
    fe r = fe_load(r_b), acc = 0;
    for (size_t i = 0; i < n; i++) acc = fe_add(fe_mul(acc, r), fe_load(coeffs + 16 * i));
    fe_store(out, acc);
}
typedef struct { or_merkle *batch_layer; fe fingerprint_r; or_fri *fri; size_t n_codes; } bfri_t;
typedef struct { path_t batch_path; query_t query; } bquery_t;
struct or_bfri_proof {
    uint8_t batch_commitment[32];
    size_t n_commitments; uint8_t *commitments;
    size_t n_queries; bquery_t *queries;
    fe last_elem; uint8_t last_random[32];
};

static void bfri_free(bfri_t *b) { if (b) { or_merkle_free(b->batch_layer); or_fri_free(b->fri); free(b); } }
/* BatchedFriProverData::init, batched_fri.rs:41-99 */
static bfri_t *bfri_init(const uint8_t *const *codes, size_t n_codes, size_t n, or_transcript *t) {
    if (n_codes == 0 || !is_pow2(n) || n < 2) return NULL;
    size_t half = n / 2;
    uint8_t **pairs = (uint8_t **)calloc(n_codes, sizeof(uint8_t *));
    for (size_t j = 0; j < n_codes; j++) { /* :62-74 */
        const fe *code = (const fe *)codes[j];
        fe *pj = (fe *)malloc((2 * half + 1) * sizeof(fe));
        PAR_FOR for (size_t i = 0; i < half; i++) { pj[2 * i] = code[i]; pj[2 * i + 1] = code[i + half]; }
        pairs[j] = (uint8_t *)pj;
    }
    bfri_t *b = (bfri_t *)calloc(1, sizeof *b);
    b->n_codes = n_codes;
    b->batch_layer = or_merkle_batch_commit((const uint8_t *const *)pairs, n_codes, 32, half); /* :77 */
    for (size_t j = 0; j < n_codes; j++) free(pairs[j]);
    free(pairs);
    uint8_t root[32];
    or_merkle_root(b->batch_layer, root);
    or_transcript_absorb(t, root, 32);          /* :80 */
    b->fingerprint_r = transcript_challenge(t); /* :83 */
    absorb_fe(t, b->fingerprint_r);             /* :86 */
    b->fri = (or_fri *)calloc(1, sizeof(or_fri)); /* :89-92 empty */
    return b;
}
/* batched_fold_step, batched_fri.rs:101-181 */
static int bfri_batched_fold_step(bfri_t *b, const fe *gen_pows, size_t gen_pows_len, fe r, or_transcript *t) {
    const or_merkle *bl = b->batch_layer;
    size_t n = bl->n_leaves * 2, blowup = (size_t)1 << OR_LOG_BLOWUP;
    if (n <= blowup) return OR_OK;
    size_t half_n = n >> 1;
    fe *next = (fe *)malloc(half_n * sizeof(fe));
    fe half = fe_div(fe_from_i64(1), fe_from_i64(2)), fr = b->fingerprint_r;
    PAR_FOR for (size_t i = 0; i < half_n; i++) {
        fe a = 0, bb = 0;
        for (size_t j = 0; j < b->n_codes; j++) { /* :126-131 fingerprints over the batch */
            const fe *d = (const fe *)bl->data[j];
            a = fe_add(fe_mul(a, fr), d[2 * i]);
            bb = fe_add(fe_mul(bb, fr), d[2 * i + 1]);
        }
        if (i == 0) next[i] = fe_mul(fe_add(fe_add(a, bb), fe_mul(r, fe_sub(a, bb))), half);
        else {
            fe even = fe_add(a, bb);
            fe odd = fe_mul(fe_sub(a, bb), gen_pows[gen_pows_len - i]);
            next[i] = fe_mul(fe_add(even, fe_mul(r, odd)), half);
        }
    }
    int st = fold_finish(b->fri, next, half_n, t);
    free(next);
    return st;
}
/* BatchedFriProverData::open_query_at, batched_fri.rs:207-225 */
static int bfri_open_query_at(const bfri_t *b, size_t index, bquery_t *out) {
    if (b->fri->n_trees == 0) return OR_ERR_RANGE; /* merkle_trees[0] would panic */
    out->batch_path = path_open(b->batch_layer, index);
    size_t n = b->batch_layer->n_leaves / 2;
    out->query = fri_open_query_at(b->fri, index % n);
    return OR_OK;
}
static or_bfri_proof *bfri_assemble(const bfri_t *b, size_t domain_size, or_transcript *t, int *status) {
    or_bfri_proof *p = (or_bfri_proof *)calloc(1, sizeof *p);
    p->n_queries = OR_NUM_QUERIES;
    p->queries = (bquery_t *)calloc(OR_NUM_QUERIES, sizeof(bquery_t));
    for (size_t q = 0; q < OR_NUM_QUERIES; q++) {
        size_t idx = next_query_index(t, domain_size);
        int st = bfri_open_query_at(b, idx, &p->queries[q]);
        if (st != OR_OK) { *status = st; p->n_queries = q; or_bfri_proof_free(p); return NULL; }
        absorb_index(t, idx);
    }
    or_merkle_root(b->batch_layer, p->batch_commitment);
    p->n_commitments = b->fri->n_trees;
    p->commitments = (uint8_t *)malloc(32 * (p->n_commitments + 1));
    or_fri_fold_roots(b->fri, p->commitments);
    p->last_elem = b->fri->last;
    or_transcript_random(t, p->last_random);
    return p;
}
or_bfri_proof *or_batched_fri_prove(const uint8_t *const *codes, size_t n_codes, size_t n, const uint8_t *gen_pows,
                                    size_t gen_pows_len, or_transcript *t, int *status) {
    *status = OR_OK;
    bfri_t *b = bfri_init(codes, n_codes, n, t);
    if (!b) { *status = OR_ERR_NOT_POW2; return NULL; }
    size_t num_steps = ctz_sz(n) - OR_LOG_BLOWUP; /* batched_fri.rs:191 */
    fe r = transcript_challenge(t);               /* :194 */
    int st = bfri_batched_fold_step(b, (const fe *)gen_pows, gen_pows_len, r, t);
    for (size_t k = 1; k < num_steps && st == OR_OK; k++) { /* :198-201 */
        uint8_t rb[16];
        or_transcript_next_challenge(t, rb);
        st = or_fri_fold_step(b->fri, gen_pows, gen_pows_len, k, rb, t);
    }
    if (st == OR_OK && !b->fri->has_last) st = OR_ERR_SIZE;
    or_bfri_proof *p = NULL;
    if (st == OR_OK) p = bfri_assemble(b, n, t, &st);
    *status = st;
    bfri_free(b);
    return p;
}
void or_bfri_proof_free(or_bfri_proof *p) {
    if (!p) return;
    for (size_t q = 0; q < p->n_queries; q++) {
        path_free(&p->queries[q].batch_path);
        for (size_t j = 0; j < p->queries[q].query.n_paths; j++) path_free(&p->queries[q].query.paths[j]);
        free(p->queries[q].query.paths);
    }
    free(p->queries); free(p->commitments); free(p);
}
/* BatchedQueryProof::verify, batched_fri.rs:228-282 */
static int bquery_verify(const bquery_t *bq, const or_bfri_proof *fp, size_t n, size_t index, fe gen, const fe *rs, fe fr) {
    if (bq->query.n_paths != fp->n_commitments) return OR_V_WRONG_NUM_PATHS;
    const path_t *p = &bq->batch_path;
    int st = or_merkle_path_verify(p->value, p->value_bytes, p->digests, p->dirs, p->path_len, fp->batch_commitment, index);
    if (st != OR_V_OK) return st;
    size_t nb = p->value_bytes / 32;
    fe value = 0, minus_value = 0, two = fe_from_i64(2);
    for (size_t j = 0; j < nb; j++) {
        value = fe_add(fe_mul(value, fr), fe_load(p->value + 32 * j));
        minus_value = fe_add(fe_mul(minus_value, fr), fe_load(p->value + 32 * j + 16));
    }
    fe gp = fe_pow(gen, (u128)index);
    fe even = fe_div(fe_add(value, minus_value), two);
    fe odd = fe_div(fe_sub(value, minus_value), fe_mul(two, gp));
    fe expect = fe_add(even, fe_mul(rs[0], odd));
    if (bq->query.n_paths == 0) return fp->last_elem == expect ? OR_V_OK : OR_V_QUERY_MISMATCH;
    size_t next_n = n / 2, next_index = index % next_n;
    fe next_gen = fe_mul(gen, gen);
    const path_t *np = &bq->query.paths[0];
    fe next_value = next_index == index ? fe_load(np->value) : fe_load(np->value + 16);
    if (next_value != expect) return OR_V_QUERY_MISMATCH;
    return query_verify(&bq->query, fp->commitments, fp->n_commitments, fp->last_elem, next_n, next_index, next_gen, rs + 1);
}
/* BatchedFriProof::verify_queries, batched_fri.rs:356-397 */
static int bfri_verify_queries(const or_bfri_proof *p, or_transcript *t, const fe *rs, fe fr) {
    if (p->n_queries != OR_NUM_QUERIES) return OR_V_WRONG_NUM_QUERIES;
    size_t log_domain = p->n_commitments + 1 + OR_LOG_BLOWUP, domain = (size_t)1 << log_domain;
    fe gen;
    if (pow2_generator(log_domain, &gen) != OR_OK) return OR_V_QUERY_MISMATCH;
    for (size_t q = 0; q < p->n_queries; q++) {
        size_t n = domain / 2;
        size_t idx = next_query_index(t, domain);
        int st = bquery_verify(&p->queries[q], p, n, idx, gen, rs, fr);
        if (st != OR_V_OK) return st;
        absorb_index(t, idx);
    }
    uint8_t lr[32];
    or_transcript_random(t, lr);
    return memcmp(lr, p->last_random, 32) == 0 ? OR_V_OK : OR_V_LAST_RANDOM;
}
int or_batched_fri_verify(const or_bfri_proof *p) { /* batched_fri.rs:320-354 */
    or_transcript *t = or_transcript_new();
    or_transcript_absorb(t, p->batch_commitment, 32);
    fe fr = transcript_challenge(t);
    absorb_fe(t, fr);
    fe *rs = (fe *)malloc((p->n_commitments + 2) * sizeof(fe));
    rs[0] = transcript_challenge(t);
    for (size_t i = 0; i < p->n_commitments; i++) {
        or_transcript_absorb(t, p->commitments + 32 * i, 32);
        rs[i + 1] = transcript_challenge(t);
    }
    absorb_fe(t, p->last_elem);
    int st = bfri_verify_queries(p, t, rs, fr);
    free(rs);
    or_transcript_free(t);
    return st;
}
/* BatchedFriProof has no serde derive in the reference; same bincode conventions as FriProof, field order of the struct */
static void bfri_proof_write(const or_bfri_proof *p, wr_t *w) {
    w_bytes(w, p->batch_commitment, 32);
    w_u64(w, p->n_commitments);
    w_bytes(w, p->commitments, 32 * p->n_commitments);
    w_u64(w, p->n_queries);
    for (size_t q = 0; q < p->n_queries; q++) {
        const path_t *bp = &p->queries[q].batch_path;
        size_t nb = bp->value_bytes / 32;
        w_u64(w, nb);
        for (size_t j = 0; j < nb; j++) w_pair(w, bp->value + 32 * j);
        w_path_tail(w, bp);
        w_query(w, &p->queries[q].query);
    }
    uint8_t le[16];
    fe_store(le, p->last_elem);
    w_fe_bytes(w, le);
    w_bytes(w, p->last_random, 32);
}
size_t or_bfri_proof_serialized_len(const or_bfri_proof *p) { wr_t w = {NULL, 0}; bfri_proof_write(p, &w); return w.n; }
void or_bfri_proof_serialize(const or_bfri_proof *p, uint8_t *out) { wr_t w = {out, 0}; bfri_proof_write(p, &w); }
void or_bfri_proof_batch_commitment(const or_bfri_proof *p, uint8_t out[32]) { memcpy(out, p->batch_commitment, 32); }
size_t or_bfri_proof_num_commitments(const or_bfri_proof *p) { return p->n_commitments; }
void or_bfri_proof_commitments(const or_bfri_proof *p, uint8_t *out) { memcpy(out, p->commitments, 32 * p->n_commitments); }
void or_bfri_proof_last(const or_bfri_proof *p, uint8_t last_elem[16], uint8_t last_random[32]) {
    fe_store(last_elem, p->last_elem);
    memcpy(last_random, p->last_random, 32);
}

/* ------------------------------------------------------------ batched PCS */
struct or_bpcs_proof { or_bfri_proof *fri; size_t n_rounds; fe *sc; fe *inputs; size_t n_inputs; fe *outputs; size_t n_outputs; };

or_bpcs_proof *or_batched_pcs_prove(const uint8_t *inputs, size_t n_vars, const uint8_t *outputs, size_t n_polys,
                                    const uint8_t *const *evals, size_t n, or_transcript *t, int *status) {
    *status = OR_OK;
    if (n_polys == 0 || !is_pow2(n) || n < 2 || ((size_t)1 << n_vars) != n) { *status = OR_ERR_SIZE; return NULL; }
    size_t log_domain = ctz_sz(n) + OR_LOG_BLOWUP, domain = (size_t)1 << log_domain; /* batched_pcs.rs:136 */
    fe *gen_pows = (fe *)malloc(domain * sizeof(fe));
    if (or_pow2_generator_powers(log_domain, (uint8_t *)gen_pows) != OR_OK) { free(gen_pows); *status = OR_ERR_RANGE; return NULL; }
    fe gen = gen_pows[1];
    fe **codes = (fe **)malloc(n_polys * sizeof(fe *));
    for (size_t j = 0; j < n_polys; j++) codes[j] = encode_poly(evals[j], n, gen); /* :144-149 */
    /* BatchedPCSProverData::init (:37-77) */
    or_transcript_absorb(t, inputs, n_vars * 16);   /* :44-46 */
    or_transcript_absorb(t, outputs, n_polys * 16); /* :47-49 */
    bfri_t *b = bfri_init((const uint8_t *const *)codes, n_polys, domain, t);
    fe fr = b->fingerprint_r;
    fe *fp_evals = (fe *)malloc(n * sizeof(fe));
    PAR_FOR for (size_t i = 0; i < n; i++) { /* :55-60 */
        fe acc = 0;
        for (size_t j = 0; j < n_polys; j++) acc = fe_add(fe_mul(acc, fr), ((const fe *)evals[j])[i]);
        fp_evals[i] = acc;
    }
    or_sumcheck *sc = or_sumcheck_build_tables_for_pcs(inputs, n_vars, (const uint8_t *)fp_evals, n); /* :66-67 */
    free(fp_evals);
    size_t num_steps = ctz_sz(domain) - OR_LOG_BLOWUP; /* :90 */
    fe prev;
    { uint8_t o[16]; uint8_t frb[16]; fe_store(frb, fr); or_fingerprint(frb, outputs, n_polys, o); prev = fe_load(o); } /* :92-94 */
    or_bpcs_proof *p = (or_bpcs_proof *)calloc(1, sizeof *p);
    p->n_rounds = num_steps;
    p->sc = (fe *)malloc(2 * num_steps * sizeof(fe) + 16);
    int st = OR_OK;
    for (size_t k = 0; k < num_steps && st == OR_OK; k++) { /* :100-123 */
        fe r = sumcheck_round(sc, 2, &prev, t, p->sc + 2 * k);
        if (k == 0) st = bfri_batched_fold_step(b, gen_pows, domain, r, t);
        else { uint8_t rb[16]; fe_store(rb, r); st = or_fri_fold_step(b->fri, (const uint8_t *)gen_pows, domain, k, rb, t); }
    }
    if (st == OR_OK && !b->fri->has_last) st = OR_ERR_SIZE;
    if (st == OR_OK) p->fri = bfri_assemble(b, domain, t, &st); /* :155-173 */
    if (st == OR_OK) {
        p->n_inputs = n_vars; p->n_outputs = n_polys;
        p->inputs = (fe *)malloc(n_vars * 16 + 16); memcpy(p->inputs, inputs, n_vars * 16);
        p->outputs = (fe *)malloc(n_polys * 16 + 16); memcpy(p->outputs, outputs, n_polys * 16);
    }
    for (size_t j = 0; j < n_polys; j++) free(codes[j]);
    free(codes); free(gen_pows); or_sumcheck_free(sc); bfri_free(b);
    *status = st;
    if (st != OR_OK) { or_bpcs_proof_free(p); return NULL; }
    return p;
}
void or_bpcs_proof_free(or_bpcs_proof *p) { if (p) { or_bfri_proof_free(p->fri); free(p->sc); free(p->inputs); free(p->outputs); free(p); } }
const or_bfri_proof *or_bpcs_proof_fri(const or_bpcs_proof *p) { return p->fri; }
size_t or_bpcs_proof_num_rounds(const or_bpcs_proof *p) { return p->n_rounds; }
void or_bpcs_proof_sumcheck_coeffs(const or_bpcs_proof *p, uint8_t *out) { memcpy(out, p->sc, p->n_rounds * 32); }

int or_batched_pcs_verify(const or_bpcs_proof *p, or_transcript *t) { /* batched_pcs.rs:182-253 */
    const or_bfri_proof *fp = p->fri;
    if (fp->n_queries != OR_NUM_QUERIES) return OR_V_WRONG_NUM_QUERIES;
    size_t n = fp->n_commitments + 1;
    if (n != p->n_rounds || n != p->n_inputs) return OR_ERR_SIZE;
    fe *rs = (fe *)malloc(n * sizeof(fe));
    or_transcript_absorb(t, (const uint8_t *)p->inputs, p->n_inputs * 16);
    or_transcript_absorb(t, (const uint8_t *)p->outputs, p->n_outputs * 16);
    fe fr = 0;
    for (size_t i = 0; i < n; i++) {
        if (i == 0) {
            or_transcript_absorb(t, fp->batch_commitment, 32);
            fr = transcript_challenge(t);
            absorb_fe(t, fr);
        } else or_transcript_absorb(t, fp->commitments + 32 * (i - 1), 32);
        absorb_fe(t, p->sc[2 * i]);
        absorb_fe(t, p->sc[2 * i + 1]);
        rs[i] = transcript_challenge(t);
    }
    absorb_fe(t, fp->last_elem);
    uint8_t frb[16], sumb[16];
    fe_store(frb, fr);
    or_fingerprint(frb, (const uint8_t *)p->outputs, p->n_outputs, sumb);
    int st = sumcheck_replay(p->sc, n, fe_load(sumb), p->inputs, rs, fp->last_elem);
    if (st == OR_V_OK) st = bfri_verify_queries(fp, t, rs, fr);
    free(rs);
    return st;
}
