// Handle-level C ABI: Merkle trees, FRI prover data and proofs, sumcheck tables, PCS / batched PCS provers.
// Host code here is orchestration only (Fiat-Shamir transcript, 3-coefficient round polynomials, query
// bookkeeping); every array operation is a CUDA kernel from the sibling translation units.
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <thread>
#include "prover_internal.h"

using namespace mlb;

#define API_BEGIN \
    Ctx* ctx;     \
    MLB_TRY(get_ctx(&ctx));
#define ST(stream_arg) ((cudaStream_t)(stream_arg))

namespace mlbp {

// handle-owned buffers come from the stream-ordered pool (cudaMalloc/cudaFree would serialise the device per layer)
int pmalloc(void** p, size_t bytes, cudaStream_t s) { return dev_alloc_async(p, bytes, s); }
void pfree(void* p, cudaStream_t s) { if (p) cudaFreeAsync(p, s); }

// ---- optional host-side phase trace (MLB_TRACE=1): (thread, tag, seconds) tuples dumped by ml_trace_dump()
struct TraceRec { size_t tid; const char* tag; double t; };
static std::mutex g_trace_mu;
static std::vector<TraceRec> g_trace;
void trace(const char* tag) {
    static const bool on = getenv("MLB_TRACE") != nullptr;
    if (!on) return;
    const double t = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
    std::lock_guard<std::mutex> lock(g_trace_mu);
    static std::atomic<size_t> next_id{0};
    thread_local size_t my_id = next_id++;
    g_trace.push_back(TraceRec{my_id, tag, t});
}
static void trace_dump_impl() {
    std::lock_guard<std::mutex> lock(g_trace_mu);
    if (g_trace.empty()) return;
    const double t0 = g_trace.front().t;
    for (const TraceRec& r : g_trace) fprintf(stderr, "TRACE %03zu %-14s %9.3f ms\n", r.tid, r.tag, (r.t - t0) * 1e3);
    g_trace.clear();
}
// Host -> device upload.  Large uploads from concurrent callers to ONE device are serialised (one at a time, each waited for
// under that device's lock): a copy engine shared by n uploads finishes all of them late, so n commits submitted together would all
// start their NTT after the LAST byte of the LAST input arrived and then run in lock-step — copy phase with idle SMs, compute phase
// with an idle copy engine (measured with 8 host-pointer commits in flight: 113-136 ms per step in lock-step, 75 ms when staggered).
// One upload at a time makes the stagger structural: commit k computes while commit k+1 uploads.
// The caller's own earlier work on `s` is drained BEFORE the lock is taken, so under the lock only the copy itself is waited for and
// a caller with kernels queued delays nobody but itself.  Host-pointer entry points are therefore host-synchronous for inputs of
// 16 MB and more (documented in include/multilinear_b200.h).
static const int MAX_UPLOAD_DEVICES = 64;
static std::mutex g_upload_mu[MAX_UPLOAD_DEVICES];
// Pageable host memory (a plain Vec<Field128> / malloc / numpy array the caller never page-locked): cudaMemcpyAsync stages it through
// the driver's own bounce buffer on ONE thread, 11.5 GB/s on the bench box against 55 GB/s from pinned memory, and page-locking it
// in place costs more than the copy (cudaHostRegister 45 ms + unregister 17 ms for 256 MiB; tools/h2d_probe.py).  So the library
// stages it itself: STAGE_THREADS host threads copy 4 MiB chunks into a per-device ring of pinned slots (two per thread) and
// queue the DMA of each slot on the caller's stream; the host copies of different threads and the DMA overlap.
static const size_t STAGE_CHUNK = (size_t)4 << 20;
static const int STAGE_THREADS = 4, STAGE_SLOTS = 2 * STAGE_THREADS;
struct Stager {
    uint8_t* slot[STAGE_SLOTS] = {nullptr};
    cudaEvent_t ev[STAGE_SLOTS] = {nullptr};
    bool ready = false, failed = false;
};
static Stager g_stager[MAX_UPLOAD_DEVICES];  // used under g_upload_mu[dev]
static bool stager_init(Stager& st) {
    if (st.ready || st.failed) return st.ready;
    for (int i = 0; i < STAGE_SLOTS; i++)
        if (cudaMallocHost((void**)&st.slot[i], STAGE_CHUNK) != cudaSuccess || cudaEventCreateWithFlags(&st.ev[i], cudaEventDisableTiming) != cudaSuccess) {
            cudaGetLastError();
            st.failed = true;  // fall back to the driver's staging for good
            return false;
        }
    st.ready = true;
    return true;
}
static bool is_pageable(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}
static int staged_upload(void* dst, const void* src, size_t bytes, cudaStream_t s, int dev, Stager& st) {
    const size_t n_chunks = (bytes + STAGE_CHUNK - 1) / STAGE_CHUNK;
    std::atomic<size_t> next{0};
    std::atomic<int> status{ML_OK};
    auto work = [&](int w) {
        if (cudaSetDevice(dev) != cudaSuccess) { status = ML_ERR_CUDA; return; }
        for (size_t k = 0;; k++) {
            const size_t c = next.fetch_add(1);
            if (c >= n_chunks || status != ML_OK) return;
            const int sl = 2 * w + (int)(k & 1);
            if (k >= 2 && cudaEventSynchronize(st.ev[sl]) != cudaSuccess) { status = ML_ERR_CUDA; return; }  // the slot's previous DMA is done
            const size_t off = c * STAGE_CHUNK, len = bytes - off < STAGE_CHUNK ? bytes - off : STAGE_CHUNK;
            memcpy(st.slot[sl], (const uint8_t*)src + off, len);
            if (cudaMemcpyAsync((uint8_t*)dst + off, st.slot[sl], len, cudaMemcpyHostToDevice, s) != cudaSuccess ||
                cudaEventRecord(st.ev[sl], s) != cudaSuccess) { status = ML_ERR_CUDA; return; }
        }
    };
    std::thread th[STAGE_THREADS - 1];
    for (int w = 1; w < STAGE_THREADS; w++) {
        try {
            th[w - 1] = std::thread(work, w);
        } catch (...) {  // no thread to be had: the remaining chunks are picked up by the threads that did start
        }
    }
    work(0);
    for (auto& t : th)
        if (t.joinable()) t.join();
    if (status != ML_OK) { set_error("staged upload failed: %s", cudaGetErrorString(cudaGetLastError())); return status; }
    return ML_OK;
}
int h2d(void* dst, const void* src, size_t bytes, cudaStream_t s) {
    if (!bytes) return ML_OK;
    if (bytes < ((size_t)16 << 20)) {
        MLB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s));
        return ML_OK;
    }
    int dev = 0;
    MLB_CUDA(cudaGetDevice(&dev));
    MLB_TRY(stream_wait_blocking(s));  // not under the lock: this stream's earlier work is this caller's own business
    trace("upload_wait");
    std::lock_guard<std::mutex> lock(g_upload_mu[dev % MAX_UPLOAD_DEVICES]);
    trace("upload_begin");
    static const bool no_stage = getenv("MLB_NO_STAGED_UPLOAD") != nullptr;
    Stager& stg = g_stager[dev % MAX_UPLOAD_DEVICES];
    if (!no_stage && is_pageable(src) && stager_init(stg)) MLB_TRY(staged_upload(dst, src, bytes, s, dev, stg));
    else MLB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s));
    int st = stream_wait_blocking(s);  // the stream holds nothing but the copy now
    trace("upload_done");
    return st;
}
// Wait for a stream without spinning: the end-of-chain waits last milliseconds, and with several commits in flight per GPU
// and one process per GPU the default spin-wait of cudaStreamSynchronize keeps (streams x GPUs) host cores busy — more than an
// 8-GPU box has, which starved the threads still enqueueing kernels (8 GPUs: 68.6 ms per step instead of 53.8).
// A blocking-sync event lets the thread sleep until the GPU signals.
int stream_wait_blocking(cudaStream_t s) {
    static const bool spin = getenv("MLB_SPIN_SYNC") != nullptr;
    if (spin) { MLB_CUDA(cudaStreamSynchronize(s)); return ML_OK; }
    thread_local cudaEvent_t ev = nullptr;
    thread_local int ev_dev = -1;
    int dev = 0;
    MLB_CUDA(cudaGetDevice(&dev));
    if (ev == nullptr || ev_dev != dev) {
        if (ev) cudaEventDestroy(ev);
        MLB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventBlockingSync | cudaEventDisableTiming));
        ev_dev = dev;
    }
    MLB_CUDA(cudaEventRecord(ev, s));
    MLB_CUDA(cudaEventSynchronize(ev));
    return ML_OK;
}
int d2h_sync(void* dst, const void* src, size_t bytes, cudaStream_t s) {
    if (bytes) MLB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s));
    return stream_wait_blocking(s);
}
int fri_push_layer(ml_fri* f, fe* code, size_t n, bool owns_code, cudaStream_t s, bool build_tree);
void absorb_fe(ml_transcript* t, hfe x) {
    uint8_t b[16];
    hfe_store(b, x);
    t->sha.update(b, 16);
}
hfe challenge(ml_transcript* t) {  // Transcript::next_challenge, src/transcript.rs:35-38
    uint8_t d[32];
    t->sha.digest(d);
    return hfe_new(hfe_load(d));
}

// ------------------------------------------------------------------ path / value gathers for openings
struct PathJob {
    const uint8_t* digests;         // tree digests (all layers)
    const fe* code;                 // RS code of the tree (value = code[index], code[index + n_leaves]) or null
    unsigned long long n_leaves, index, dig_off, val_off;
    int depth;
};
__global__ void gather_paths_kernel(const PathJob* __restrict__ jobs, uint8_t* __restrict__ out) {
    const PathJob j = jobs[blockIdx.x];
    const int t = threadIdx.x;
    if (t < j.depth) {  // sibling at layer t (src/merkle_tree/mod.rs:43-55)
        const unsigned long long sib = (j.index >> t) ^ 1ull;
        const uint4* src = reinterpret_cast<const uint4*>(j.digests + 32 * ((2 * j.n_leaves - ((2 * j.n_leaves) >> t)) + sib));
        uint4* dst = reinterpret_cast<uint4*>(out + j.dig_off + 32ull * t);
        dst[0] = src[0];
        dst[1] = src[1];
    }
    if (j.code && t >= 62 && t < 64) {
        const fe* src = j.code + j.index + (t == 63 ? j.n_leaves : 0);
        *reinterpret_cast<uint4*>(out + j.val_off + 16ull * (t - 62)) = *reinterpret_cast<const uint4*>(src);
    }
}
// byte items: out[b*item_bytes + k] = data[b][index*item_bytes + k]
__global__ void gather_bytes_kernel(const uint8_t* const* __restrict__ data, int n_batches, size_t item_bytes, size_t index,
                                    uint8_t* __restrict__ out) {
    const size_t total = (size_t)n_batches * item_bytes;
    for (size_t p = threadIdx.x; p < total; p += blockDim.x) {
        size_t b = p / item_bytes, k = p - b * item_bytes;
        out[p] = data[b][index * item_bytes + k];
    }
}
// batch layer values: for query q, code b: pair (code_b[idx_q], code_b[idx_q + L]) -> out[(q*B + b)*32]
__global__ void gather_batch_values_kernel(const fe* const* __restrict__ codes, int n_codes, size_t n_leaves,
                                           const unsigned long long* __restrict__ indices, uint8_t* __restrict__ out) {
    const size_t q = blockIdx.x;
    const unsigned long long idx = indices[q];
    for (int b = threadIdx.x; b < n_codes; b += blockDim.x) {
        const fe* c = codes[b];
        uint4* dst = reinterpret_cast<uint4*>(out + (q * n_codes + b) * 32);
        dst[0] = *reinterpret_cast<const uint4*>(c + idx);
        dst[1] = *reinterpret_cast<const uint4*>(c + idx + n_leaves);
    }
}

void free_merkle(ml_merkle* m) {
    if (!m) return;
    if (m->owns_digests) pfree(m->digests, m->stream);
    if (m->owns_data)
        for (void* p : m->data) pfree(p, m->stream);
    pfree(m->data_ptrs_dev, m->stream);
    delete m;
}
int new_merkle(size_t n_leaves, cudaStream_t s, ml_merkle** out) {
    ml_merkle* m = new ml_merkle();
    m->n_leaves = n_leaves;
    m->stream = s;
    if (pmalloc((void**)&m->digests, (2 * n_leaves) * 32, s) != ML_OK) { delete m; return ML_ERR_ALLOC; }
    cudaGetDevice(&m->device);
    *out = m;
    return ML_OK;
}
int merkle_fetch_root(ml_merkle* m, cudaStream_t s) {
    const int top = (int)ilog2(m->n_leaves);
    return d2h_sync(m->root, m->digests + 32 * merkle_layer_offset(m->n_leaves, top), 32, s);
}
int merkle_set_ptrs(ml_merkle* m, cudaStream_t s) {
    MLB_TRY(pmalloc((void**)&m->data_ptrs_dev, m->data.size() * sizeof(void*), s));
    return h2d(m->data_ptrs_dev, m->data.data(), m->data.size() * sizeof(void*), s);
}

// FRI layer commit: commit_rs_code (src/fri/mod.rs:45-55) + absorb root (:71, :133)
int fri_commit_layer(ml_fri* f, fe* code, size_t n, bool owns_code, ml_transcript* t, cudaStream_t s) {
    ml_merkle* m;
    MLB_TRY(new_merkle(n / 2, s, &m));
    m->kind = ml_merkle::RS_CODE;
    m->item_bytes = 32;
    m->data.push_back(code);
    m->owns_data = false;
    int st = merkle_rs_launch(code, n, m->digests, s);
    if (st == ML_OK) st = merkle_fetch_root(m, s);
    if (st != ML_OK) { free_merkle(m); return st; }
    t->sha.update(m->root, 32);
    ml_fri::Layer L;
    L.code = code; L.n = n; L.owns_code = owns_code; L.tree = m;
    f->layers.push_back(L);
    return ML_OK;
}
void free_fri(ml_fri* f) {
    if (!f) return;
    for (auto& L : f->layers) {
        if (L.owns_code) pfree(L.code, f->stream);
        free_merkle(L.tree);
    }
    delete f;
}
// tail shared by fold_step (:116-133) and batched_fold_step (batched_fri.rs:152-180); takes ownership of `next`
int fold_finish(ml_fri* f, fe* next, size_t half_n, ml_transcript* t, cudaStream_t s) {
    if (half_n == ((size_t)1 << ML_LOG_BLOWUP)) {
        uint8_t b[32];
        int st = d2h_sync(b, next, 32, s);
        pfree(next, s);
        MLB_TRY(st);
        if (memcmp(b, b + 16, 16) != 0) { set_error("not an RS code"); return ML_ERR_NOT_RS_CODE; }
        f->last = hfe_load(b);
        f->has_last = true;
        t->sha.update(b, 16);
        return ML_OK;
    }
    int st = fri_commit_layer(f, next, half_n, true, t, s);
    if (st != ML_OK) pfree(next, s);
    return st;
}
int fri_fold_step_impl(Ctx* ctx, ml_fri* f, size_t k, hfe r, ml_transcript* t, cudaStream_t s) {
    if (f->layers.empty()) { set_error("fold_step on empty FriProverData"); return ML_ERR_ARG; }
    const ml_fri::Layer& last = f->layers.back();
    const size_t n = last.n;
    if (n <= ((size_t)1 << ML_LOG_BLOWUP)) return ML_OK;  // :83-85
    const size_t half_n = n >> 1;
    if ((half_n << k) > ((size_t)1 << f->log_n0)) { set_error("fold_step: k = %zu out of range for this domain", k); return ML_ERR_ARG; }
    fe* next;
    MLB_TRY(pmalloc((void**)&next, half_n * 16, s));
    int st = fri_fold_launch(ctx, last.code, n, next, r, nullptr, k, f->log_n0, s);
    if (st != ML_OK) { pfree(next, s); return st; }
    return fold_finish(f, next, half_n, t, s);
}
int fri_init_owned(ml_fri** out, fe* code, size_t n, bool owns, ml_transcript* t, cudaStream_t s) {
    ml_fri* f = new ml_fri();
    f->log_n0 = (int)ilog2(n);
    f->stream = s;
    int st = fri_commit_layer(f, code, n, owns, t, s);
    if (st != ML_OK) { if (owns) pfree(code, s); free_fri(f); return st; }
    *out = f;
    return ML_OK;
}
int fri_new_unabsorbed(ml_fri** out, fe* code, size_t n, bool owns, cudaStream_t s) {
    ml_fri* f = new ml_fri();
    f->log_n0 = (int)ilog2(n);
    f->stream = s;
    int st = fri_push_layer(f, code, n, owns, s, true);
    if (st != ML_OK) { if (owns) pfree(code, s); free_fri(f); return st; }
    *out = f;
    return ML_OK;
}
int check_code_len(size_t n) {
    if (!is_pow2(n) || n < 2) { set_error("Input size must be a power of two (>= 2)"); return ML_ERR_NOT_POW2; }
    return ML_OK;
}
int fri_fold_all(Ctx* ctx, ml_fri* f, ml_transcript* t, cudaStream_t s) {  // :138-143
    const size_t num_steps = (size_t)f->log_n0 - ML_LOG_BLOWUP;
    for (size_t k = 0; k < num_steps; k++) {
        hfe r = challenge(t);
        MLB_TRY(fri_fold_step_impl(ctx, f, k, r, t, s));
    }
    if (!f->has_last) { set_error("fold: last_element is None"); return ML_ERR_SIZE; }
    return ML_OK;
}

// ------------------------------------------------------------------ query phase
size_t next_query_index(ml_transcript* t, size_t domain_size) {  // :269-271
    uint8_t d[32];
    t->sha.digest(d);
    uint64_t v;
    memcpy(&v, d, 8);
    return (size_t)(v % (uint64_t)(domain_size / 2));
}
void absorb_index(ml_transcript* t, size_t idx) {  // :276 usize little-endian
    uint64_t v = idx;
    t->sha.update(&v, 8);
}
void fill_dirs(PathH& p, size_t index, int depth) {
    p.dirs.resize(depth);
    for (int l = 0; l < depth; l++) p.dirs[l] = ((index >> l) & 1) ? 0 : 1;  // even index: sibling on the Right
}
// open_query_at (:154-174) for many indices at once: one gather kernel, one D2H copy
int fri_open_queries(const ml_fri* f, const std::vector<size_t>& indices, std::vector<QueryH>& out, cudaStream_t s) {
    const size_t nq = indices.size(), nt = f->layers.size();
    out.assign(nq, QueryH());
    if (nq == 0 || nt == 0) return ML_OK;
    std::vector<PathJob> jobs;
    jobs.reserve(nq * nt);
    size_t off = 0;
    for (size_t q = 0; q < nq; q++) {
        size_t cur = indices[q], cur_n = f->layers[0].n / 2;
        out[q].paths.resize(nt);
        for (size_t j = 0; j < nt; j++) {
            const ml_fri::Layer& L = f->layers[j];
            PathJob pj;
            pj.digests = L.tree->digests; pj.code = L.code; pj.n_leaves = L.n / 2; pj.index = cur;
            pj.depth = (int)ilog2(L.n / 2);
            pj.val_off = off; off += 32;
            pj.dig_off = off; off += 32ull * pj.depth;
            jobs.push_back(pj);
            cur_n /= 2;
            if (cur_n) cur %= cur_n;
        }
    }
    Scratch djobs(s), dout(s);
    MLB_TRY(djobs.alloc(jobs.size() * sizeof(PathJob)));
    MLB_TRY(dout.alloc(off));
    MLB_TRY(h2d(djobs.p, jobs.data(), jobs.size() * sizeof(PathJob), s));
    ProfScope prof(PROF_GATHER, 2.0 * (double)off, s);
    gather_paths_kernel<<<(unsigned)jobs.size(), 64, 0, s>>>(djobs.as<PathJob>(), dout.as<uint8_t>());
    MLB_KERNEL_CHECK();
    std::vector<uint8_t> host(off);
    MLB_TRY(d2h_sync(host.data(), dout.p, off, s));
    size_t ji = 0;
    for (size_t q = 0; q < nq; q++)
        for (size_t j = 0; j < nt; j++, ji++) {
            const PathJob& pj = jobs[ji];
            PathH& p = out[q].paths[j];
            p.value.assign(host.begin() + pj.val_off, host.begin() + pj.val_off + 32);
            p.digests.assign(host.begin() + pj.dig_off, host.begin() + pj.dig_off + 32ull * pj.depth);
            fill_dirs(p, pj.index, pj.depth);
        }
    return ML_OK;
}
// the 128 query indices (:268-277): they depend on the transcript only, so derive them all before gathering
void derive_indices(ml_transcript* t, size_t domain_size, std::vector<size_t>& idx) {
    idx.resize(ML_NUM_QUERIES);
    for (int q = 0; q < ML_NUM_QUERIES; q++) {
        idx[q] = next_query_index(t, domain_size);
        absorb_index(t, idx[q]);
    }
}
int assemble_fri_proof(const ml_fri* f, size_t domain_size, ml_transcript* t, ml_fri_proof* p, cudaStream_t s) {
    std::vector<size_t> idx;
    derive_indices(t, domain_size, idx);
    MLB_TRY(fri_open_queries(f, idx, p->queries, s));
    p->commitments.resize(32 * f->layers.size());
    for (size_t j = 0; j < f->layers.size(); j++) memcpy(&p->commitments[32 * j], f->layers[j].tree->root, 32);
    p->last_elem = f->last;
    t->sha.digest(p->last_random);
    return ML_OK;
}

// ------------------------------------------------------------------ sumcheck round (host part of :174-202)
// Lagrange interpolation over x = 0..n-1 (src/polynomials.rs:51-86), tiny n
void interpolate(const std::vector<hfe>& evals, std::vector<hfe>& coeffs) {
    const size_t n = evals.size();
    coeffs.assign(n, 0);
    for (size_t j = 0; j < n; j++) {
        std::vector<hfe> lj(1, 1);
        hfe denom = 1;
        for (size_t m = 0; m < n; m++) {
            if (m == j) continue;
            std::vector<hfe> nl(lj.size() + 1, 0);
            hfe xm = hfe_new((hfe)m);
            for (size_t i = 0; i < lj.size(); i++) {
                nl[i] = hfe_sub(nl[i], hfe_mul(lj[i], xm));
                nl[i + 1] = hfe_add(nl[i + 1], lj[i]);
            }
            lj.swap(nl);
            denom = hfe_mul(denom, hfe_sub(hfe_new((hfe)j), xm));
        }
        hfe scale = hfe_div(evals[j], denom);
        for (size_t i = 0; i < n; i++) coeffs[i] = hfe_add(coeffs[i], hfe_mul(scale, lj[i]));
    }
}
hfe poly_eval(const std::vector<hfe>& c, hfe x) {
    hfe acc = 0;
    for (size_t i = c.size(); i-- > 0;) acc = hfe_add(hfe_mul(acc, x), c[i]);
    return acc;
}
int sumcheck_round(Ctx* ctx, ml_sumcheck* sc, size_t total_degree, hfe* previous_sum, ml_transcript* t, hfe* nonzero_out, hfe* r_out,
                   cudaStream_t s) {
    std::vector<hfe> evals(total_degree + 1, 0), coeffs;
    if (total_degree == 2) {  // the PCS path: both partial sums in one pass over the tables
        MLB_TRY(sumcheck_sums_launch(ctx, sc->matrix, sc->delta, sc->height, &evals[1], &evals[2], s));
    } else {
        for (size_t i = 1; i <= total_degree; i++)
            MLB_TRY(sumcheck_partial_sum_launch(ctx, sc->matrix, sc->delta, sc->height, hfe_new((hfe)i), &evals[i], s));
    }
    evals[0] = hfe_sub(*previous_sum, evals[1]);                          // :188 (total_degree >= 1)
    interpolate(evals, coeffs);                                           // :189-192
    for (size_t i = 1; i <= total_degree; i++) { nonzero_out[i - 1] = coeffs[i]; absorb_fe(t, coeffs[i]); }  // :193-197
    hfe r = challenge(t);                                                 // :198
    *previous_sum = poly_eval(coeffs, r);                                 // :199
    MLB_TRY(sumcheck_fold_launch(sc->matrix, sc->delta, sc->height, r, nullptr, s));  // :200
    sc->height >>= 1;
    *r_out = r;
    return ML_OK;
}
void free_sumcheck(ml_sumcheck* s) {
    if (!s) return;
    if (s->owns_matrix) pfree(s->matrix, s->stream);
    pfree(s->delta, s->stream);
    delete s;
}
int sumcheck_build(Ctx* ctx, const uint8_t* inputs, size_t n_vars, const void* evals, bool evals_on_device, size_t height, cudaStream_t s,
                   ml_sumcheck** out) {
    if (n_vars >= 40 || ((size_t)1 << n_vars) != height) { set_error("assert_eq!(1 << n_vars, height) failed"); return ML_ERR_SIZE; }
    ml_sumcheck* sc = new ml_sumcheck();
    sc->height = height;
    sc->stream = s;
    if (pmalloc((void**)&sc->matrix, height * 16, s) != ML_OK || pmalloc((void**)&sc->delta, height * 16, s) != ML_OK) {
        free_sumcheck(sc);
        return ML_ERR_ALLOC;
    }
    cudaError_t e = cudaMemcpyAsync(sc->matrix, evals, height * 16, evals_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) { free_sumcheck(sc); set_error("copy failed: %s", cudaGetErrorString(e)); return ML_ERR_CUDA; }
    std::vector<hfe> pts(n_vars);
    for (size_t i = 0; i < n_vars; i++) pts[i] = hfe_load(inputs + 16 * i);
    int st = eq_table_launch(ctx, pts.data(), n_vars, sc->delta, s);
    if (st == ML_OK && cudaStreamSynchronize(s) != cudaSuccess) st = ML_ERR_CUDA;  // pts is a host temporary
    if (st != ML_OK) { free_sumcheck(sc); return st; }
    *out = sc;
    return ML_OK;
}

// evals -> to_coefficient -> bit_reverse -> reed_solomon (multilinear_pcs.rs:101-107): returns a new owned code of 2n elements
// writes the code of one polynomial given by evaluations into `code` (2n elements)
int encode_into(Ctx* ctx, const fe* evals_dev, size_t n, fe* code, cudaStream_t s) {
    const int log_domain = (int)ilog2(n) + ML_LOG_BLOWUP;
    Scratch coeffs(s);
    MLB_TRY(coeffs.alloc(n * 16));
    MLB_TRY(mobius_launch(evals_dev, coeffs.as<fe>(), n, true, s));
    if (ntt_fuses_bitrev(log_domain))  // bit_reverse_permutation (:104) folded into the first NTT pass's addressing
        return ntt_launch(ctx, coeffs.as<fe>(), code, log_domain, false, true, s, true);
    Scratch rev(s);
    MLB_TRY(rev.alloc(n * 16));
    MLB_TRY(bit_reverse_launch(coeffs.p, rev.p, n, 16, s));
    return ntt_launch(ctx, rev.as<fe>(), code, log_domain, false, true, s);
}
int encode_poly(Ctx* ctx, const fe* evals_dev, size_t n, fe** code_out, cudaStream_t s) {
    fe* code;
    MLB_TRY(pmalloc((void**)&code, (n << ML_LOG_BLOWUP) * 16, s));
    int st = encode_into(ctx, evals_dev, n, code, s);
    if (st != ML_OK) { pfree(code, s); return st; }
    *code_out = code;
    return ML_OK;
}

// ------------------------------------------------------------------ sync-free fold chain (device transcript)

// build the tree of a layer without reading the root back (the chain absorbs it on the device)
int fri_push_layer(ml_fri* f, fe* code, size_t n, bool owns_code, cudaStream_t s, bool build_tree) {
    ml_merkle* m;
    MLB_TRY(new_merkle(n / 2, s, &m));
    m->kind = ml_merkle::RS_CODE;
    m->item_bytes = 32;
    m->data.push_back(code);
    m->owns_data = false;
    if (build_tree) {
        int st = merkle_rs_launch(code, n, m->digests, s);
        if (st != ML_OK) { free_merkle(m); return st; }
    }
    ml_fri::Layer L;
    L.code = code; L.n = n; L.owns_code = owns_code; L.tree = m;
    f->layers.push_back(L);
    return ML_OK;
}
uint8_t* layer_root_ptr(const ml_fri::Layer& L) {
    const size_t leaves = L.n / 2;
    return L.tree->digests + 32 * merkle_layer_offset(leaves, (int)ilog2(leaves));
}

// Runs fold steps k_start.. to the end with the transcript advanced on the device.
//   f       : FriProverData; its last layer is the current code (tree built).  Empty only with `b` (batched first fold).
//   pending : the last layer's root has not been absorbed yet
//   sc/prev : sumcheck tables + running claim for the PCS interleave (nullptr/unused for plain FRI)
//   sc_out  : host array receiving (c1, c2) per round from k_start on
// On return every layer root, last_element and the host transcript are up to date.
int fold_chain_dev(Ctx* ctx, ml_fri* f, const ChainHooks* hooks, ml_sumcheck* sc, hfe prev, hfe* sc_out, size_t k_start, bool pending,
                   ml_transcript* t, cudaStream_t s) {
    const size_t total_steps = (size_t)f->log_n0 - ML_LOG_BLOWUP;
    if (k_start >= total_steps) {
        if (!f->has_last) { set_error("fold: last_element is None"); return ML_ERR_SIZE; }
        return ML_OK;
    }
    // one scratch block: transcript | r, r/2 | prev | last[2] | status | roots[64] | sc[2*64] | partials
    const int max_nb = sumcheck_max_blocks();
    Scratch blk(s);
    const size_t off_tr = 0, off_r = 128, off_prev = off_r + 32, off_last = off_prev + 16, off_status = off_last + 32,
                 off_roots = off_status + 16, off_sc = off_roots + 64 * 32, off_part = off_sc + 2 * 64 * 16,
                 total = off_part + (size_t)(2 * max_nb + 2) * 16;
    MLB_TRY(blk.alloc(total));
    uint8_t* base = blk.as<uint8_t>();
    DevTranscript* tr_dev = (DevTranscript*)(base + off_tr);
    fe* r_dev = (fe*)(base + off_r);
    fe* prev_dev = (fe*)(base + off_prev);
    fe* last_dev = (fe*)(base + off_last);
    int* status_dev = (int*)(base + off_status);
    uint8_t* roots_dev = base + off_roots;
    fe* sc_dev = (fe*)(base + off_sc);
    fe* partials = (fe*)(base + off_part);
    MLB_CUDA(cudaMemsetAsync(base, 0, off_part, s));
    if (hooks && hooks->tr_dev) MLB_CUDA(cudaMemcpyAsync(tr_dev, hooks->tr_dev, sizeof(DevTranscript), cudaMemcpyDeviceToDevice, s));
    else MLB_TRY(h2d(tr_dev, &t->sha, sizeof(DevTranscript), s));
    if (sc) {
        if (hooks && hooks->prev_dev) {
            MLB_CUDA(cudaMemcpyAsync(prev_dev, hooks->prev_dev, 16, cudaMemcpyDeviceToDevice, s));
        } else {
            uint8_t pb[16];
            hfe_store(pb, prev);
            MLB_TRY(h2d(prev_dev, pb, 16, s));
        }
    }
    const RootTables* rt;
    MLB_TRY(get_root_tables(ctx, f->log_n0, s, &rt));

    const size_t first_new_layer = f->layers.size() - (pending ? 1 : 0);  // roots to fetch afterwards: layers >= this index
    bool used_tail = false, have_partials = false;
    int sc_nb = 0;
    size_t k = k_start;
    for (; k < total_steps; k++) {
        const bool batched_round = f->layers.empty();
        const size_t n = batched_round ? ((size_t)1 << f->log_n0) : f->layers.back().n;
        if (n <= ((size_t)1 << ML_LOG_BLOWUP)) break;
        const size_t half_n = n >> 1;
        if (!batched_round && n <= ((size_t)1 << TAIL_LOG)) {
            // ---- fused tail: every remaining round in one launch
            TailArgs a;
            memset(&a, 0, sizeof a);
            const size_t tail_base = f->layers.size() - 1;
            a.codes[0] = f->layers.back().code;
            a.digests[0] = f->layers.back().tree->digests;
            a.n0 = n; a.k0 = (int)k; a.log_n0 = f->log_n0;
            a.lo = rt->lo; a.hi = rt->hi;
            a.tr = tr_dev;
            a.roots_out = roots_dev + 32 * (tail_base + 1);
            a.first_root_out = roots_dev + 32 * tail_base;
            a.last_out = last_dev;
            a.status = status_dev;
            a.absorb_first_root = pending ? 1 : 0;
            if (sc) { a.m = sc->matrix; a.d = sc->delta; a.height = sc->height; a.prev = prev_dev; a.sc_out = sc_dev + 2 * (k - k_start); }
            int i = 1;
            for (size_t m = half_n; m > 2; m >>= 1, i++) {  // committed tail layers: sizes half_n .. 4
                fe* code;
                MLB_TRY(pmalloc((void**)&code, m * 16, s));
                int st = fri_push_layer(f, code, m, true, s, false);
                if (st != ML_OK) { pfree(code, s); return st; }
                a.codes[i] = code;
                a.digests[i] = f->layers.back().tree->digests;
            }
            MLB_TRY(chain_tail_launch(a, s));
            if (sc) { size_t rounds = ilog2(n) - 1; sc->height >>= rounds; }
            pending = false;
            used_tail = true;
            k = total_steps;
            break;
        }
        // ---- challenge (absorbing the pending root first)
        const uint8_t* absorb = pending ? layer_root_ptr(f->layers.back()) : nullptr;
        uint8_t* copy_out = pending ? roots_dev + 32 * (f->layers.size() - 1) : nullptr;
        if (sc) {
            if (!have_partials) MLB_TRY(sumcheck_sums_partials_launch(sc->matrix, sc->delta, sc->height, partials, &sc_nb, s));
            MLB_TRY(chain_sumcheck_finish_launch(partials, sc_nb, prev_dev, tr_dev, absorb, pending ? 32 : 0, copy_out, sc_dev + 2 * (k - k_start), r_dev, s));
            // the next round's sums are fused into this fold whenever that round runs as separate kernels again
            // (the tail kernel computes its own sums)
            have_partials = half_n > ((size_t)1 << TAIL_LOG) && sc->height >= 4 && k + 1 < total_steps;
            if (have_partials) MLB_TRY(sumcheck_fold_sums_launch(sc->matrix, sc->delta, sc->height, r_dev, partials, &sc_nb, s));
            else MLB_TRY(sumcheck_fold_launch(sc->matrix, sc->delta, sc->height, 0, r_dev, s));
            sc->height >>= 1;
        } else {
            MLB_TRY(chain_challenge_launch(tr_dev, absorb, pending ? 32 : 0, copy_out, r_dev, true, s));
        }
        pending = false;
        // ---- fold
        fe* next = nullptr;
        bool owns_next = true;
        if (batched_round) {
            if (!hooks || !hooks->first_fold) { set_error("fold chain: empty FriProverData without a first-fold hook"); return ML_ERR_ARG; }
            MLB_TRY(hooks->first_fold(r_dev, &next, &owns_next));
        } else {
            MLB_TRY(pmalloc((void**)&next, half_n * 16, s));
            int st = fri_fold_launch(ctx, f->layers.back().code, n, next, 0, r_dev, k, f->log_n0, s);
            if (st != ML_OK) { pfree(next, s); return st; }
        }
        if (half_n == ((size_t)1 << ML_LOG_BLOWUP)) {  // only reachable from a batched first fold of a 4-element domain
            int st = chain_last_launch(next, tr_dev, last_dev, status_dev, s);
            if (owns_next) pfree(next, s);
            MLB_TRY(st);
            used_tail = true;
            k = total_steps;
            break;
        }
        int st = fri_push_layer(f, next, half_n, owns_next, s, true);
        if (st != ML_OK) { if (owns_next) pfree(next, s); return st; }
        pending = true;
    }
    if (pending) {  // chain ended on a committed layer (cannot happen for well-formed sizes, kept for safety)
        MLB_TRY(chain_challenge_launch(tr_dev, layer_root_ptr(f->layers.back()), 32, roots_dev + 32 * (f->layers.size() - 1), r_dev, false, s));
    }
    // ---- single synchronisation point: roots, last element, status, coefficients, transcript
    trace("enqueued");
    std::vector<uint8_t> host(off_part);
    MLB_TRY(d2h_sync(host.data(), base, off_part, s));
    int status = 0;
    memcpy(&status, host.data() + off_status, sizeof status);
    if (status != 0) { set_error("not an RS code"); return status; }
    for (size_t j = first_new_layer; j < f->layers.size(); j++) memcpy(f->layers[j].tree->root, host.data() + off_roots + 32 * j, 32);
    if (used_tail) {
        f->last = hfe_load(host.data() + off_last);
        f->has_last = true;
    }
    if (sc && sc_out)
        for (size_t i = 0; i < 2 * (total_steps - k_start); i++) sc_out[i] = hfe_load(host.data() + off_sc + 16 * i);
    memcpy(&t->sha, host.data() + off_tr, sizeof(DevTranscript));
    if (!f->has_last) { set_error("fold: last_element is None"); return ML_ERR_SIZE; }
    return ML_OK;
}

// ------------------------------------------------------------------ host verifiers (O(128 log n) work)
void hash_node_host(const uint8_t* l, const uint8_t* r, uint8_t* out) {
    HostSha256 h;
    h.update(l, 32);
    h.update(r, 32);
    h.digest(out);
}
int path_verify(const PathH& p, const uint8_t* root, size_t index) {  // merkle_tree/mod.rs:216-246
    uint8_t h[32], nx[32];
    HostSha256 hs;
    hs.update(p.value.data(), p.value.size());
    hs.digest(h);
    size_t computed = 0;
    for (size_t i = 0; i < p.dirs.size(); i++) {
        if (p.dirs[i] == 0) { computed += (size_t)1 << i; hash_node_host(&p.digests[32 * i], h, nx); }
        else hash_node_host(h, &p.digests[32 * i], nx);
        memcpy(h, nx, 32);
    }
    if (memcmp(h, root, 32) != 0) return ML_V_INCLUSION_HASH;
    if (computed != index) return ML_V_INCLUSION_INDEX;
    return ML_V_OK;
}
int query_verify(const QueryH& q, const uint8_t* commitments, size_t n_commitments, hfe last_element, size_t n, size_t index, hfe gen,
                 const hfe* rs) {  // fri/mod.rs:184-236
    if (q.paths.size() != n_commitments) return ML_V_WRONG_NUM_PATHS;
    size_t cur_n = n, cur_idx = index;
    hfe cur_gen = gen, two = 2;
    for (size_t i = 0; i < q.paths.size(); i++) {
        const PathH& p = q.paths[i];
        int st = path_verify(p, commitments + 32 * i, cur_idx);
        if (st != ML_V_OK) return st;
        hfe value = hfe_load(p.value.data()), minus_value = hfe_load(p.value.data() + 16);
        hfe gp = hfe_pow(cur_gen, (hfe)cur_idx);
        hfe even = hfe_div(hfe_add(value, minus_value), two);
        hfe odd = hfe_div(hfe_sub(value, minus_value), hfe_mul(two, gp));
        hfe expect = hfe_add(even, hfe_mul(rs[i], odd));
        if (i == q.paths.size() - 1) return last_element == expect ? ML_V_OK : ML_V_QUERY_MISMATCH;
        size_t next_idx = cur_idx % (cur_n / 2);
        const PathH& np = q.paths[i + 1];
        hfe next_value = next_idx == cur_idx ? hfe_load(np.value.data()) : hfe_load(np.value.data() + 16);
        if (next_value != expect) return ML_V_QUERY_MISMATCH;
        cur_gen = hfe_mul(cur_gen, cur_gen);
        cur_n /= 2;
        cur_idx = next_idx;
    }
    return ML_V_OK;
}
int fri_verify_queries(const ml_fri_proof* p, ml_transcript* t, const hfe* rs) {  // fri/mod.rs:311-340
    const size_t nc = p->commitments.size() / 32;
    const size_t log_domain = nc + ML_LOG_BLOWUP, domain = (size_t)1 << log_domain;
    hfe gen;
    if (!hfe_pow2_generator(log_domain, &gen)) return ML_V_QUERY_MISMATCH;
    for (const QueryH& q : p->queries) {
        size_t idx = next_query_index(t, domain);
        absorb_index(t, idx);
        int st = query_verify(q, p->commitments.data(), nc, p->last_elem, domain / 2, idx, gen, rs);
        if (st != ML_V_OK) return st;
    }
    uint8_t lr[32];
    t->sha.digest(lr);
    return memcmp(lr, p->last_random, 32) == 0 ? ML_V_OK : ML_V_LAST_RANDOM;
}
hfe delta_evaluate(const hfe* data, const hfe* points, size_t n) {  // evaluation.rs:80-90
    hfe prod = 1;
    for (size_t i = 0; i < n; i++) {
        hfe a = data[i], b = points[i];
        prod = hfe_mul(prod, hfe_add(hfe_mul(a, b), hfe_mul(hfe_sub(1, a), hfe_sub(1, b))));
    }
    return prod;
}
void to_polynomial(const hfe* nonzero, hfe sum, hfe pol[3]) {  // sumcheck.rs:269-276 (degree 2)
    pol[0] = hfe_div(hfe_sub(sum, hfe_add(nonzero[0], nonzero[1])), 2);
    pol[1] = nonzero[0];
    pol[2] = nonzero[1];
}
hfe eval3(const hfe pol[3], hfe x) { return hfe_add(hfe_mul(hfe_add(hfe_mul(pol[2], x), pol[1]), x), pol[0]); }
int sumcheck_replay(const std::vector<hfe>& sc, hfe sum, const std::vector<hfe>& inputs, const std::vector<hfe>& rs, hfe last_elem) {
    const size_t n = rs.size();
    hfe pol[3];
    to_polynomial(&sc[0], sum, pol);
    for (size_t i = 1; i < n; i++) to_polynomial(&sc[2 * i], eval3(pol, rs[i - 1]), pol);
    hfe delta = delta_evaluate(inputs.data(), rs.data(), n);
    return hfe_mul(delta, last_elem) == eval3(pol, rs[n - 1]) ? ML_V_OK : ML_V_SUMCHECK;
}
hfe fingerprint_host(hfe r, const hfe* c, size_t n) {  // batched_fri.rs:30-38
    hfe acc = 0;
    for (size_t i = 0; i < n; i++) acc = hfe_add(hfe_mul(acc, r), c[i]);
    return acc;
}

// ------------------------------------------------------------------ wire format (bincode fixed-int LE via serde, fri/mod.rs:367-369)
struct Writer {
    uint8_t* p;
    size_t n = 0;
    explicit Writer(uint8_t* out) : p(out) {}
    void bytes(const void* b, size_t len) { if (p) memcpy(p + n, b, len); n += len; }
    void u64(uint64_t v) { bytes(&v, 8); }
    void u32(uint32_t v) { bytes(&v, 4); }
    void febytes(const uint8_t* b) { u64(16); bytes(b, 16); }  // Field128::serialize -> serialize_bytes (field.rs:40-48)
    void pair(const uint8_t* v) { febytes(v); febytes(v + 16); }
    void path_tail(const PathH& q) {
        u64(q.dirs.size());
        for (size_t i = 0; i < q.dirs.size(); i++) { bytes(&q.digests[32 * i], 32); u32(q.dirs[i]); }
    }
    void query(const QueryH& q) {
        u64(q.paths.size());
        for (const PathH& ph : q.paths) { pair(ph.value.data()); path_tail(ph); }
    }
};
void write_fri_proof(const ml_fri_proof* p, Writer& w) {
    w.u64(p->commitments.size() / 32);
    w.bytes(p->commitments.data(), p->commitments.size());
    w.u64(p->queries.size());
    for (const QueryH& q : p->queries) w.query(q);
    uint8_t le[16];
    hfe_store(le, p->last_elem);
    w.febytes(le);
    w.bytes(p->last_random, 32);
}
// inverse of write_fri_proof (the crate's serde/bincode derives, fri/mod.rs:239-249): false on malformed input
struct Reader {
    const uint8_t* p;
    size_t n, o = 0;
    bool ok = true;
    Reader(const uint8_t* b, size_t len) : p(b), n(len) {}
    bool take(void* dst, size_t len) {
        if (!ok || len > n - o) { ok = false; return false; }
        memcpy(dst, p + o, len);
        o += len;
        return true;
    }
    uint64_t u64() { uint64_t v = 0; take(&v, 8); return v; }
    uint32_t u32() { uint32_t v = 0; take(&v, 4); return v; }
    bool febytes(uint8_t* out) { return u64() == 16 && take(out, 16); }
};
bool read_fri_proof(Reader& r, ml_fri_proof* p) {
    const uint64_t nc = r.u64();
    if (!r.ok || nc > 64) return false;
    p->commitments.resize(32 * nc);
    r.take(p->commitments.data(), 32 * nc);
    const uint64_t nq = r.u64();
    if (!r.ok || nq > 4096) return false;
    p->queries.resize(nq);
    for (QueryH& q : p->queries) {
        const uint64_t np = r.u64();
        if (!r.ok || np > 64) return false;
        q.paths.resize(np);
        for (PathH& ph : q.paths) {
            ph.value.resize(32);
            if (!r.febytes(ph.value.data()) || !r.febytes(ph.value.data() + 16)) return false;
            const uint64_t len = r.u64();
            if (!r.ok || len > 64) return false;
            ph.digests.resize(32 * len);
            ph.dirs.resize(len);
            for (uint64_t i = 0; i < len; i++) {
                r.take(&ph.digests[32 * i], 32);
                const uint32_t d = r.u32();
                if (!r.ok || d > 1) return false;
                ph.dirs[i] = (uint8_t)d;
            }
        }
    }
    uint8_t le[16];
    if (!r.febytes(le)) return false;
    p->last_elem = hfe_load(le);
    if (p->last_elem >= HFE_M) return false;
    return r.take(p->last_random, 32);
}
void write_bfri_proof(const ml_bfri_proof* p, Writer& w) {
    w.bytes(p->batch_commitment, 32);
    w.u64(p->commitments.size() / 32);
    w.bytes(p->commitments.data(), p->commitments.size());
    w.u64(p->queries.size());
    for (const BQueryH& q : p->queries) {
        const size_t nb = q.batch_path.value.size() / 32;
        w.u64(nb);
        for (size_t j = 0; j < nb; j++) w.pair(&q.batch_path.value[32 * j]);
        w.path_tail(q.batch_path);
        w.query(q.query);
    }
    uint8_t le[16];
    hfe_store(le, p->last_elem);
    w.febytes(le);
    w.bytes(p->last_random, 32);
}

// ------------------------------------------------------------------ batched FRI prover data (batched_fri.rs:9-14)
struct BatchedFri {
    std::vector<fe*> codes;      // device, n elements each
    bool owns_codes = true;
    fe** codes_ptrs_dev = nullptr;
    size_t n = 0;
    ml_merkle* batch_layer = nullptr;
    hfe fingerprint_r = 0;
    ml_fri* fri = nullptr;
    cudaStream_t stream = nullptr;
    ~BatchedFri() {
        if (owns_codes)
            for (fe* c : codes) pfree(c, stream);
        pfree(codes_ptrs_dev, stream);
        if (batch_layer) { batch_layer->owns_data = false; free_merkle(batch_layer); }
        free_fri(fri);
    }
};
// BatchedFriProverData::init (batched_fri.rs:41-99)
int bfri_init(BatchedFri* b, ml_transcript* t, cudaStream_t s) {
    const size_t B = b->codes.size(), n = b->n;
    if (B == 0) { set_error("Codes must not be empty"); return ML_ERR_SIZE; }
    MLB_TRY(check_code_len(n));
    b->stream = s;
    MLB_TRY(pmalloc((void**)&b->codes_ptrs_dev, B * sizeof(fe*), s));
    MLB_TRY(h2d(b->codes_ptrs_dev, b->codes.data(), B * sizeof(fe*), s));
    MLB_TRY(new_merkle(n / 2, s, &b->batch_layer));
    b->batch_layer->kind = ml_merkle::RS_CODE;
    b->batch_layer->item_bytes = 32;
    b->batch_layer->n_batches = B;
    for (fe* c : b->codes) b->batch_layer->data.push_back(c);
    b->batch_layer->owns_data = false;
    MLB_TRY(merkle_batched_rs_launch(b->codes_ptrs_dev, B, n, b->batch_layer->digests, s));  // :77
    MLB_TRY(merkle_fetch_root(b->batch_layer, s));
    t->sha.update(b->batch_layer->root, 32);  // :80
    b->fingerprint_r = challenge(t);          // :83
    absorb_fe(t, b->fingerprint_r);           // :86
    b->fri = new ml_fri();                    // :89-92
    b->fri->log_n0 = (int)ilog2(n);
    b->fri->stream = s;
    return ML_OK;
}
// batched_fold_step (batched_fri.rs:101-181)
int bfri_batched_fold_step(Ctx* ctx, BatchedFri* b, hfe r, ml_transcript* t, cudaStream_t s) {
    const size_t n = b->n;
    if (n <= ((size_t)1 << ML_LOG_BLOWUP)) return ML_OK;
    const size_t half_n = n >> 1;
    fe* next;
    MLB_TRY(pmalloc((void**)&next, half_n * 16, s));
    int st = fri_batched_fold_launch(ctx, b->codes_ptrs_dev, b->codes.size(), n, next, b->fingerprint_r, r, nullptr, b->fri->log_n0, s);
    if (st != ML_OK) { pfree(next, s); return st; }
    return fold_finish(b->fri, next, half_n, t, s);
}
int bfri_first_fold_dev(Ctx* ctx, BatchedFri* b, const fe* r_dev, fe** next_out, size_t* half_n_out, cudaStream_t s) {
    const size_t half_n = b->n >> 1;
    fe* next;
    MLB_TRY(pmalloc((void**)&next, half_n * 16, s));
    int st = fri_batched_fold_launch(ctx, b->codes_ptrs_dev, b->codes.size(), b->n, next, b->fingerprint_r, 0, r_dev, b->fri->log_n0, s);
    if (st != ML_OK) { pfree(next, s); return st; }
    *next_out = next;
    *half_n_out = half_n;
    return ML_OK;
}
// BatchedFriProverData::open_query_at (batched_fri.rs:207-225) for many indices at once
int bfri_open_queries(BatchedFri* b, const std::vector<size_t>& idx, std::vector<BQueryH>& out, cudaStream_t s) {
    const size_t n = b->n, L = n / 2, B = b->codes.size();
    if (b->fri->layers.empty()) { set_error("open_query_at: no folded layer (domain too small)"); return ML_ERR_OUT_OF_RANGE; }
    const size_t nq = idx.size();
    // batch layer: values of all codes + path in the batch tree
    std::vector<PathJob> jobs(nq);
    const int depth = (int)ilog2(L);
    for (size_t q = 0; q < nq; q++) {
        jobs[q].digests = b->batch_layer->digests; jobs[q].code = nullptr; jobs[q].n_leaves = L; jobs[q].index = idx[q];
        jobs[q].depth = depth; jobs[q].dig_off = q * 32ull * depth; jobs[q].val_off = 0;
    }
    std::vector<unsigned long long> idx64(idx.begin(), idx.end());
    Scratch djobs(s), dpaths(s), didx(s), dvals(s);
    MLB_TRY(djobs.alloc(nq * sizeof(PathJob)));
    MLB_TRY(dpaths.alloc(nq * 32 * (size_t)(depth ? depth : 1)));
    MLB_TRY(didx.alloc(nq * 8));
    MLB_TRY(dvals.alloc(nq * B * 32));
    MLB_TRY(h2d(djobs.p, jobs.data(), nq * sizeof(PathJob), s));
    MLB_TRY(h2d(didx.p, idx64.data(), nq * 8, s));
    gather_paths_kernel<<<(unsigned)nq, 64, 0, s>>>(djobs.as<PathJob>(), dpaths.as<uint8_t>());
    MLB_KERNEL_CHECK();
    gather_batch_values_kernel<<<(unsigned)nq, 64, 0, s>>>(b->codes_ptrs_dev, (int)B, L, didx.as<unsigned long long>(), dvals.as<uint8_t>());
    MLB_KERNEL_CHECK();
    std::vector<uint8_t> hp(nq * 32 * (size_t)depth), hv(nq * B * 32);
    MLB_TRY(d2h_sync(hp.data(), dpaths.p, hp.size(), s));
    MLB_TRY(d2h_sync(hv.data(), dvals.p, hv.size(), s));
    std::vector<size_t> sub(nq);
    for (size_t q = 0; q < nq; q++) sub[q] = idx[q] % (L / 2);  // :217-218
    std::vector<QueryH> qs;
    MLB_TRY(fri_open_queries(b->fri, sub, qs, s));
    out.resize(nq);
    for (size_t q = 0; q < nq; q++) {
        PathH& bp = out[q].batch_path;
        bp.value.assign(hv.begin() + q * B * 32, hv.begin() + (q + 1) * B * 32);
        bp.digests.assign(hp.begin() + q * 32 * (size_t)depth, hp.begin() + (q + 1) * 32 * (size_t)depth);
        fill_dirs(bp, idx[q], depth);
        out[q].query = std::move(qs[q]);
    }
    return ML_OK;
}
// query phase of BatchedFriProof::prove / BatchedPCSProof::prove (batched_fri.rs:296-308)
int bfri_assemble(BatchedFri* b, ml_transcript* t, ml_bfri_proof* p, cudaStream_t s) {
    if (b->fri->layers.empty()) { set_error("open_query_at: no folded layer (domain too small)"); return ML_ERR_OUT_OF_RANGE; }
    std::vector<size_t> idx;
    derive_indices(t, b->n, idx);
    MLB_TRY(bfri_open_queries(b, idx, p->queries, s));
    memcpy(p->batch_commitment, b->batch_layer->root, 32);
    p->commitments.resize(32 * b->fri->layers.size());
    for (size_t j = 0; j < b->fri->layers.size(); j++) memcpy(&p->commitments[32 * j], b->fri->layers[j].tree->root, 32);
    p->last_elem = b->fri->last;
    t->sha.digest(p->last_random);
    return ML_OK;
}
int bquery_verify(const BQueryH& bq, const ml_bfri_proof* fp, size_t n, size_t index, hfe gen, const hfe* rs, hfe fr) {  // batched_fri.rs:228-282
    const size_t nc = fp->commitments.size() / 32;
    if (bq.query.paths.size() != nc) return ML_V_WRONG_NUM_PATHS;
    int st = path_verify(bq.batch_path, fp->batch_commitment, index);
    if (st != ML_V_OK) return st;
    const size_t nb = bq.batch_path.value.size() / 32;
    hfe value = 0, minus_value = 0, two = 2;
    for (size_t j = 0; j < nb; j++) {
        value = hfe_add(hfe_mul(value, fr), hfe_load(&bq.batch_path.value[32 * j]));
        minus_value = hfe_add(hfe_mul(minus_value, fr), hfe_load(&bq.batch_path.value[32 * j + 16]));
    }
    hfe gp = hfe_pow(gen, (hfe)index);
    hfe even = hfe_div(hfe_add(value, minus_value), two);
    hfe odd = hfe_div(hfe_sub(value, minus_value), hfe_mul(two, gp));
    hfe expect = hfe_add(even, hfe_mul(rs[0], odd));
    if (bq.query.paths.empty()) return fp->last_elem == expect ? ML_V_OK : ML_V_QUERY_MISMATCH;
    const size_t next_n = n / 2, next_index = index % next_n;
    const PathH& np = bq.query.paths[0];
    hfe next_value = next_index == index ? hfe_load(np.value.data()) : hfe_load(np.value.data() + 16);
    if (next_value != expect) return ML_V_QUERY_MISMATCH;
    return query_verify(bq.query, fp->commitments.data(), nc, fp->last_elem, next_n, next_index, hfe_mul(gen, gen), rs + 1);
}
int bfri_verify_queries(const ml_bfri_proof* p, ml_transcript* t, const hfe* rs, hfe fr) {  // batched_fri.rs:356-397
    if (p->queries.size() != ML_NUM_QUERIES) return ML_V_WRONG_NUM_QUERIES;
    const size_t nc = p->commitments.size() / 32;
    const size_t log_domain = nc + 1 + ML_LOG_BLOWUP, domain = (size_t)1 << log_domain;
    hfe gen;
    if (!hfe_pow2_generator(log_domain, &gen)) return ML_V_QUERY_MISMATCH;
    for (const BQueryH& q : p->queries) {
        size_t idx = next_query_index(t, domain);
        int st = bquery_verify(q, p, domain / 2, idx, gen, rs, fr);
        if (st != ML_V_OK) return st;
        absorb_index(t, idx);
    }
    uint8_t lr[32];
    t->sha.digest(lr);
    return memcmp(lr, p->last_random, 32) == 0 ? ML_V_OK : ML_V_LAST_RANDOM;
}

int wsumcheck_check_terms(size_t width, size_t n_terms, const uint32_t* term_lens, const uint32_t* term_cols, std::vector<uint32_t>& off, size_t* total) {
    if (n_terms > (size_t)wsumcheck_limits(1)) { set_error("at most %d composition terms", wsumcheck_limits(1)); return ML_ERR_ARG; }
    off.assign(n_terms ? n_terms : 1, 0);
    *total = 0;
    for (size_t t = 0; t < n_terms; t++) {
        off[t] = (uint32_t)*total;
        for (uint32_t k = 0; k < term_lens[t]; k++)
            if (term_cols[*total + k] >= width) { set_error("composition term %zu references column %u of a width-%zu trace", t, term_cols[*total + k], width); return ML_ERR_OUT_OF_RANGE; }
        *total += term_lens[t];
    }
    if (*total > (size_t)wsumcheck_limits(2)) { set_error("at most %d column references", wsumcheck_limits(2)); return ML_ERR_ARG; }
    return ML_OK;
}
int wsumcheck_lagrange(size_t td, std::vector<uint8_t>& lag) {
    const size_t n = td + 1;
    std::vector<uint8_t> unit(n * 16), col(n * 16);
    lag.assign(n * n * 16, 0);
    for (size_t j = 0; j < n; j++) {
        std::fill(unit.begin(), unit.end(), 0);
        unit[16 * j] = 1;
        MLB_TRY(ml_poly_interpolate(unit.data(), n, col.data()));
        for (size_t i = 0; i < n; i++) memcpy(&lag[(i * n + j) * 16], &col[16 * i], 16);
    }
    return ML_OK;
}

}  // namespace mlbp
using namespace mlbp;

extern "C" {
void ml_trace_dump(void) { trace_dump_impl(); }

// ================================================================== Merkle
int ml_merkle_commit(const uint8_t* data, size_t item_bytes, size_t n_items, ml_merkle** out) {
    const uint8_t* one[1] = {data};
    int st = ml_merkle_batch_commit(one, 1, item_bytes, n_items, out);
    if (st == ML_OK) (*out)->n_batches = 0;
    return st;
}
int ml_merkle_batch_commit(const uint8_t* const* data, size_t n_batches, size_t item_bytes, size_t n_items, ml_merkle** out) {
    API_BEGIN
    if (n_batches == 0) { set_error("Data must not be empty"); return ML_ERR_SIZE; }
    if (!is_pow2(n_items)) { set_error("Data length must be a power of two"); return ML_ERR_NOT_POW2; }
    cudaStream_t s = lib_stream(ctx);
    ml_merkle* m;
    MLB_TRY(new_merkle(n_items, s, &m));
    m->kind = ml_merkle::BYTES;
    m->item_bytes = item_bytes;
    m->n_batches = n_batches;
    int st = ML_OK;
    for (size_t b = 0; b < n_batches && st == ML_OK; b++) {
        void* d = nullptr;
        if (pmalloc(&d, n_items * item_bytes + 16, s) != ML_OK) { st = ML_ERR_ALLOC; break; }
        m->data.push_back(d);
        st = h2d(d, data[b], n_items * item_bytes, s);
    }
    if (st == ML_OK) st = merkle_set_ptrs(m, s);
    if (st == ML_OK) st = merkle_bytes_launch((const uint8_t* const*)m->data_ptrs_dev, n_batches, item_bytes, n_items, m->digests, s);
    if (st == ML_OK) st = merkle_fetch_root(m, s);
    if (st != ML_OK) { free_merkle(m); return st; }
    *out = m;
    return ML_OK;
}
int ml_merkle_commit_rs_code_dev(const void* code_dev, size_t n, void* stream, ml_merkle** out) {
    API_BEGIN
    (void)ctx;
    MLB_TRY(check_code_len(n));
    cudaStream_t s = ST(stream);
    ml_merkle* m;
    MLB_TRY(new_merkle(n / 2, s, &m));
    m->kind = ml_merkle::RS_CODE;
    m->item_bytes = 32;
    m->data.push_back((void*)code_dev);
    m->owns_data = false;
    int st = merkle_rs_launch((const fe*)code_dev, n, m->digests, s);
    if (st == ML_OK) st = merkle_fetch_root(m, s);
    if (st != ML_OK) { free_merkle(m); return st; }
    *out = m;
    return ML_OK;
}
void ml_merkle_free(ml_merkle* m) { free_merkle(m); }
int ml_merkle_root(const ml_merkle* m, uint8_t out[32]) { memcpy(out, m->root, 32); return ML_OK; }
size_t ml_merkle_num_layers(const ml_merkle* m) { return ilog2(m->n_leaves) + 1; }
size_t ml_merkle_layer_len(const ml_merkle* m, size_t layer) { return m->n_leaves >> layer; }
int ml_merkle_layer(const ml_merkle* m, size_t layer, uint8_t* out) {
    API_BEGIN
    if (layer > ilog2(m->n_leaves)) return ML_ERR_OUT_OF_RANGE;
    return d2h_sync(out, m->digests + 32 * merkle_layer_offset(m->n_leaves, layer), (m->n_leaves >> layer) * 32, lib_stream(ctx));
}
int ml_merkle_open(const ml_merkle* m, size_t index, uint8_t* value, uint8_t* digests, uint8_t* dirs, size_t* path_len) {
    API_BEGIN
    if (index >= m->n_leaves) { set_error("open(%zu): None", index); return ML_ERR_OUT_OF_RANGE; }
    cudaStream_t s = lib_stream(ctx);
    const int depth = (int)ilog2(m->n_leaves);
    const size_t nb = m->n_batches ? m->n_batches : 1;
    const size_t vbytes = nb * m->item_bytes;
    Scratch dj(s), dout(s);
    MLB_TRY(dj.alloc(sizeof(PathJob)));
    MLB_TRY(dout.alloc(32 * (size_t)(depth + 1) + vbytes + 32));
    PathJob pj;
    pj.digests = m->digests; pj.code = nullptr; pj.n_leaves = m->n_leaves; pj.index = index; pj.depth = depth; pj.dig_off = 0; pj.val_off = 0;
    MLB_TRY(h2d(dj.p, &pj, sizeof pj, s));
    gather_paths_kernel<<<1, 64, 0, s>>>(dj.as<PathJob>(), dout.as<uint8_t>());
    MLB_KERNEL_CHECK();
    uint8_t* dval = dout.as<uint8_t>() + 32 * (size_t)(depth + 1);
    if (m->kind == ml_merkle::BYTES) {
        gather_bytes_kernel<<<1, 128, 0, s>>>((const uint8_t* const*)m->data_ptrs_dev, (int)nb, m->item_bytes, index, dval);
        MLB_KERNEL_CHECK();
    } else {
        for (size_t b = 0; b < nb; b++) {
            const fe* c = (const fe*)m->data[b];
            MLB_CUDA(cudaMemcpyAsync(dval + 32 * b, c + index, 16, cudaMemcpyDeviceToDevice, s));
            MLB_CUDA(cudaMemcpyAsync(dval + 32 * b + 16, c + index + m->n_leaves, 16, cudaMemcpyDeviceToDevice, s));
        }
    }
    std::vector<uint8_t> host(32 * (size_t)(depth + 1) + vbytes);
    MLB_TRY(d2h_sync(host.data(), dout.p, host.size(), s));
    memcpy(digests, host.data(), 32 * (size_t)depth);
    memcpy(value, host.data() + 32 * (size_t)(depth + 1), vbytes);
    for (int l = 0; l < depth; l++) dirs[l] = ((index >> l) & 1) ? 0 : 1;
    *path_len = (size_t)depth;
    return ML_OK;
}
int ml_merkle_path_verify(const uint8_t* value, size_t value_bytes, const uint8_t* digests, const uint8_t* dirs, size_t path_len,
                          const uint8_t root[32], size_t index) {
    PathH p;
    p.value.assign(value, value + value_bytes);
    p.digests.assign(digests, digests + 32 * path_len);
    p.dirs.assign(dirs, dirs + path_len);
    return path_verify(p, root, index);
}

// ================================================================== FRI
int ml_fri_init_dev(const void* code_dev, size_t n, ml_transcript* t, void* stream, ml_fri** out) {
    API_BEGIN
    (void)ctx;
    MLB_TRY(check_code_len(n));
    cudaStream_t s = ST(stream);
    fe* code;
    MLB_TRY(pmalloc((void**)&code, n * 16, s));
    cudaError_t e = cudaMemcpyAsync(code, code_dev, n * 16, cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) { pfree(code, s); set_error("copy failed: %s", cudaGetErrorString(e)); return ML_ERR_CUDA; }
    return fri_init_owned(out, code, n, true, t, s);
}
int ml_fri_init(const uint8_t* code_host, size_t n, ml_transcript* t, ml_fri** out) {
    API_BEGIN
    MLB_TRY(check_code_len(n));
    cudaStream_t s = lib_stream(ctx);
    fe* code;
    MLB_TRY(pmalloc((void**)&code, n * 16, s));
    int st = h2d(code, code_host, n * 16, s);
    if (st != ML_OK) { pfree(code, s); return st; }
    return fri_init_owned(out, code, n, true, t, s);
}
static int check_gen_pows(const ml_fri* f, const uint8_t* gen_pows, size_t gen_pows_len) {
    if (!gen_pows) return ML_OK;
    if (gen_pows_len != ((size_t)1 << f->log_n0)) { set_error("gen_pows.len() must equal the domain size"); return ML_ERR_SIZE; }
    // The kernels read their own root tables (powers of pow_2_generator(log2 domain)), not this array, so a caller-supplied table is
    // only accepted if it IS that table.  Checked at [0], [1], [2], [len/2], [len-1] and 16 spread positions (host scalar pow): a table
    // of the right length that disagrees anywhere else would be a table the reference's own callers never build (they all pass
    // pow_2_generator_powers, src/fri/mod.rs:352, multilinear_pcs.rs:98); the restriction is stated in the header.
    hfe w;
    hfe_pow2_generator((uint64_t)f->log_n0, &w);
    size_t probe[21] = {0, 1, 2, gen_pows_len / 2, gen_pows_len - 1};
    for (int i = 0; i < 16; i++) probe[5 + i] = (size_t)(((unsigned __int128)gen_pows_len * (2 * i + 1)) / 33) ^ (size_t)(i * 2654435761u % 97);
    for (size_t idx : probe) {
        if (idx >= gen_pows_len) continue;
        if (hfe_load(gen_pows + 16 * idx) != hfe_pow(w, (hfe)idx)) {
            set_error("gen_pows[%zu] is not pow_2_generator(%d)^%zu: only the domain's own power table is supported", idx, f->log_n0, idx);
            return ML_ERR_GENERATOR;
        }
    }
    return ML_OK;
}
int ml_fri_fold_step(ml_fri* f, const uint8_t* gen_pows, size_t gen_pows_len, size_t k, const uint8_t r[16], ml_transcript* t) {
    API_BEGIN
    MLB_TRY(check_gen_pows(f, gen_pows, gen_pows_len));
    return fri_fold_step_impl(ctx, f, k, hfe_load(r), t, lib_stream(ctx));
}
static int fri_from_copy(const void* src, size_t n, bool src_on_device, cudaStream_t s, ml_fri** out) {
    MLB_TRY(check_code_len(n));
    fe* code;
    MLB_TRY(pmalloc((void**)&code, n * 16, s));
    cudaError_t e = cudaMemcpyAsync(code, src, n * 16, src_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) { pfree(code, s); set_error("copy failed: %s", cudaGetErrorString(e)); return ML_ERR_CUDA; }
    return fri_new_unabsorbed(out, code, n, true, s);
}
int ml_fri_fold_dev(const void* code_dev, size_t n, ml_transcript* t, void* stream, ml_fri** out) {
    API_BEGIN
    ml_fri* f;
    MLB_TRY(fri_from_copy(code_dev, n, true, ST(stream), &f));
    int st = fold_chain_dev(ctx, f, nullptr, nullptr, 0, nullptr, 0, true, t, ST(stream));
    if (st != ML_OK) { free_fri(f); return st; }
    *out = f;
    return ML_OK;
}
int ml_fri_fold(const uint8_t* gen_pows, size_t gen_pows_len, const uint8_t* code, size_t n, ml_transcript* t, ml_fri** out) {
    API_BEGIN
    ml_fri* f;
    MLB_TRY(fri_from_copy(code, n, false, lib_stream(ctx), &f));
    int st = check_gen_pows(f, gen_pows, gen_pows_len);
    if (st == ML_OK) st = fold_chain_dev(ctx, f, nullptr, nullptr, 0, nullptr, 0, true, t, lib_stream(ctx));
    if (st != ML_OK) { free_fri(f); return st; }
    *out = f;
    return ML_OK;
}
void ml_fri_free(ml_fri* f) { free_fri(f); }
size_t ml_fri_num_trees(const ml_fri* f) { return f->layers.size(); }
int ml_fri_tree(const ml_fri* f, size_t i, const ml_merkle** tree) {
    if (i >= f->layers.size()) return ML_ERR_OUT_OF_RANGE;
    *tree = f->layers[i].tree;
    return ML_OK;
}
__global__ void pairs_kernel(const fe* __restrict__ code, size_t half, uint4* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < half; i += stride) {
        out[2 * i] = *reinterpret_cast<const uint4*>(code + i);
        out[2 * i + 1] = *reinterpret_cast<const uint4*>(code + i + half);
    }
}
int ml_fri_tree_data(const ml_fri* f, size_t i, uint8_t* pairs_out) {
    API_BEGIN
    if (i >= f->layers.size()) return ML_ERR_OUT_OF_RANGE;
    cudaStream_t s = lib_stream(ctx);
    const ml_fri::Layer& L = f->layers[i];
    Scratch d(s);
    MLB_TRY(d.alloc(L.n * 16));
    size_t blocks = (L.n / 2 + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    pairs_kernel<<<(unsigned)blocks, 256, 0, s>>>(L.code, L.n / 2, d.as<uint4>());
    MLB_KERNEL_CHECK();
    return d2h_sync(pairs_out, d.p, L.n * 16, s);
}
int ml_fri_fold_roots(const ml_fri* f, uint8_t* out) {
    for (size_t j = 0; j < f->layers.size(); j++) memcpy(out + 32 * j, f->layers[j].tree->root, 32);
    return ML_OK;
}
int ml_fri_last_element(const ml_fri* f, uint8_t out[16], int* is_some) {
    *is_some = f->has_last ? 1 : 0;
    if (f->has_last) hfe_store(out, f->last);
    return ML_OK;
}
int ml_fri_open_query_at(const ml_fri* f, size_t index, uint8_t* values, uint8_t* digests, uint8_t* dirs, size_t* path_lens) {
    API_BEGIN
    if (f->layers.empty() || index >= f->layers[0].n / 2) { set_error("open_query_at: index out of range"); return ML_ERR_OUT_OF_RANGE; }
    std::vector<size_t> idx(1, index);
    std::vector<QueryH> q;
    MLB_TRY(fri_open_queries(f, idx, q, lib_stream(ctx)));
    size_t doff = 0;
    for (size_t j = 0; j < q[0].paths.size(); j++) {
        const PathH& p = q[0].paths[j];
        memcpy(values + 32 * j, p.value.data(), 32);
        memcpy(digests + 32 * doff, p.digests.data(), p.digests.size());
        memcpy(dirs + doff, p.dirs.data(), p.dirs.size());
        path_lens[j] = p.dirs.size();
        doff += p.dirs.size();
    }
    return ML_OK;
}
static int fri_prove_from(Ctx* ctx, ml_fri* f, size_t n, ml_transcript* t, cudaStream_t s, ml_fri_proof** out) {
    trace("chain_begin");
    int st = fold_chain_dev(ctx, f, nullptr, nullptr, 0, nullptr, 0, true, t, s);
    trace("chain_done");
    ml_fri_proof* p = nullptr;
    if (st == ML_OK) {
        p = new ml_fri_proof();
        st = assemble_fri_proof(f, n, t, p, s);
    }
    trace("queries_done");
    free_fri(f);
    trace("freed");
    if (st != ML_OK) { delete p; return st; }
    *out = p;
    return ML_OK;
}
int ml_fri_prove_dev(const void* code_dev, size_t n, ml_transcript* t, void* stream, ml_fri_proof** out) {
    API_BEGIN
    ml_fri* f;
    MLB_TRY(fri_from_copy(code_dev, n, true, ST(stream), &f));
    return fri_prove_from(ctx, f, n, t, ST(stream), out);
}
int ml_fri_prove(const uint8_t* code, size_t n, const uint8_t* gen_pows, size_t gen_pows_len, ml_transcript* t, ml_fri_proof** out) {
    API_BEGIN
    ml_fri* f;
    MLB_TRY(fri_from_copy(code, n, false, lib_stream(ctx), &f));
    int st = check_gen_pows(f, gen_pows, gen_pows_len);
    if (st != ML_OK) { free_fri(f); return st; }
    return fri_prove_from(ctx, f, n, t, lib_stream(ctx), out);
}
static int rs_encode_owned(Ctx* ctx, const void* coeffs_dev, size_t n, fe** code_out, cudaStream_t s) {
    const size_t N = n << ML_LOG_BLOWUP;
    MLB_TRY(check_code_len(N));
    fe* code;
    MLB_TRY(pmalloc((void**)&code, N * 16, s));
    int st = ntt_launch(ctx, (const fe*)coeffs_dev, code, (int)ilog2(N), false, true, s);
    if (st != ML_OK) { pfree(code, s); return st; }
    *code_out = code;
    return ML_OK;
}
int ml_rs_fri_fold_dev(const void* coeffs_dev, size_t n, ml_transcript* t, void* stream, ml_fri** out) {
    API_BEGIN
    cudaStream_t s = ST(stream);
    fe* code;
    MLB_TRY(rs_encode_owned(ctx, coeffs_dev, n, &code, s));
    ml_fri* f;
    MLB_TRY(fri_new_unabsorbed(&f, code, n << ML_LOG_BLOWUP, true, s));
    int st = fold_chain_dev(ctx, f, nullptr, nullptr, 0, nullptr, 0, true, t, s);
    if (st != ML_OK) { free_fri(f); return st; }
    *out = f;
    return ML_OK;
}
int ml_rs_fri_prove_dev(const void* coeffs_dev, size_t n, ml_transcript* t, void* stream, ml_fri_proof** out) {
    API_BEGIN
    cudaStream_t s = ST(stream);
    fe* code;
    MLB_TRY(rs_encode_owned(ctx, coeffs_dev, n, &code, s));
    ml_fri* f;
    MLB_TRY(fri_new_unabsorbed(&f, code, n << ML_LOG_BLOWUP, true, s));
    return fri_prove_from(ctx, f, n << ML_LOG_BLOWUP, t, s, out);
}
int ml_rs_fri_prove(const uint8_t* coeffs, size_t n, ml_transcript* t, ml_fri_proof** out) {
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    trace("call");
    Scratch d(s);
    MLB_TRY(d.alloc(n * 16));
    MLB_TRY(h2d(d.p, coeffs, n * 16, s));
    int st = ml_rs_fri_prove_dev(d.p, n, t, s, out);
    trace("return");
    return st;
}
int ml_fri_verify(const ml_fri_proof* p) {  // fri/mod.rs:287-309
    if (p->queries.size() != ML_NUM_QUERIES) return ML_V_WRONG_NUM_QUERIES;
    ml_transcript t;
    const size_t nc = p->commitments.size() / 32;
    std::vector<hfe> rs(nc + 1);
    for (size_t i = 0; i < nc; i++) {
        t.sha.update(&p->commitments[32 * i], 32);
        rs[i] = challenge(&t);
    }
    absorb_fe(&t, p->last_elem);
    return fri_verify_queries(p, &t, rs.data());
}
void ml_fri_proof_free(ml_fri_proof* p) { delete p; }
size_t ml_fri_proof_num_commitments(const ml_fri_proof* p) { return p->commitments.size() / 32; }
int ml_fri_proof_commitments(const ml_fri_proof* p, uint8_t* out) { memcpy(out, p->commitments.data(), p->commitments.size()); return ML_OK; }
int ml_fri_proof_last(const ml_fri_proof* p, uint8_t last_elem[16], uint8_t last_random[32]) {
    hfe_store(last_elem, p->last_elem);
    memcpy(last_random, p->last_random, 32);
    return ML_OK;
}
size_t ml_fri_proof_serialized_len(const ml_fri_proof* p) { Writer w(nullptr); write_fri_proof(p, w); return w.n; }
int ml_fri_proof_serialize(const ml_fri_proof* p, uint8_t* out) { Writer w(out); write_fri_proof(p, w); return ML_OK; }
int ml_fri_proof_deserialize(const uint8_t* blob, size_t len, ml_fri_proof** out) {
    ml_fri_proof* p = new ml_fri_proof();
    Reader r(blob, len);
    if (!read_fri_proof(r, p) || r.o != len) { delete p; set_error("FriProof blob is malformed"); return ML_ERR_ARG; }
    *out = p;
    return ML_OK;
}

// ================================================================== sumcheck
int ml_sumcheck_build_tables_for_pcs(const uint8_t* inputs, size_t n_vars, const uint8_t* evals, size_t height, ml_sumcheck** out) {
    API_BEGIN
    return sumcheck_build(ctx, inputs, n_vars, evals, false, height, lib_stream(ctx), out);
}
int ml_sumcheck_build_tables_for_pcs_dev(const uint8_t* inputs, size_t n_vars, const void* evals_dev, size_t height, void* stream,
                                         ml_sumcheck** out) {
    API_BEGIN
    return sumcheck_build(ctx, inputs, n_vars, evals_dev, true, height, ST(stream), out);
}
void ml_sumcheck_free(ml_sumcheck* s) { free_sumcheck(s); }
size_t ml_sumcheck_height(const ml_sumcheck* s) { return s->height; }
int ml_sumcheck_tables(const ml_sumcheck* sc, uint8_t* matrix_out, uint8_t* delta_out) {
    API_BEGIN
    MLB_TRY(d2h_sync(matrix_out, sc->matrix, sc->height * 16, lib_stream(ctx)));
    return d2h_sync(delta_out, sc->delta, sc->height * 16, lib_stream(ctx));
}
int ml_sumcheck_partial_sum(const ml_sumcheck* sc, const uint8_t r[16], uint8_t out[16]) {
    API_BEGIN
    hfe o;
    MLB_TRY(sumcheck_partial_sum_launch(ctx, sc->matrix, sc->delta, sc->height, hfe_load(r), &o, lib_stream(ctx)));
    hfe_store(out, o);
    return ML_OK;
}
int ml_sumcheck_fold(ml_sumcheck* sc, const uint8_t r[16]) {
    API_BEGIN
    MLB_TRY(sumcheck_fold_launch(sc->matrix, sc->delta, sc->height, hfe_load(r), nullptr, lib_stream(ctx)));
    sc->height >>= 1;
    MLB_CUDA(cudaStreamSynchronize(lib_stream(ctx)));
    return ML_OK;
}
int ml_sumcheck_compute_polynomial(ml_sumcheck* sc, size_t total_degree, uint8_t previous_sum[16], ml_transcript* t,
                                   uint8_t* nonzero_coeffs_out, uint8_t r_out[16]) {
    API_BEGIN
    // total_degree 0: the reference reads evals[1] of a one-point round (:188) and panics
    if (total_degree < 1 || total_degree > 16) { set_error("total_degree must be 1..16"); return ML_ERR_ARG; }
    hfe prev = hfe_load(previous_sum), r;
    std::vector<hfe> nz(total_degree);
    MLB_TRY(sumcheck_round(ctx, sc, total_degree, &prev, t, nz.data(), &r, lib_stream(ctx)));
    for (size_t i = 0; i < total_degree; i++) hfe_store(nonzero_coeffs_out + 16 * i, nz[i]);
    hfe_store(previous_sum, prev);
    hfe_store(r_out, r);
    return ML_OK;
}
int ml_sumcheck_compute_polynomials(ml_sumcheck* sc, size_t composition_degree, ml_transcript* t, const uint8_t sum[16],
                                    uint8_t* coeffs_out, uint8_t* randoms_out) {
    API_BEGIN
    const size_t td = composition_degree + 1;  // :159
    if (td > 16) { set_error("composition_degree too large"); return ML_ERR_ARG; }
    cudaStream_t s = lib_stream(ctx);
    const size_t rounds = sc->height ? ilog2(sc->height) : 0;  // :160
    if (td != 2) {  // general degree: host transcript, one partial_sum launch per evaluation point
        hfe prev = hfe_load(sum);
        std::vector<hfe> nz(td);
        for (size_t k = 0; k < rounds; k++) {
            hfe r;
            MLB_TRY(sumcheck_round(ctx, sc, td, &prev, t, nz.data(), &r, s));
            for (size_t i = 0; i < td; i++) hfe_store(coeffs_out + 16 * (k * td + i), nz[i]);
            hfe_store(randoms_out + 16 * k, r);
        }
        MLB_CUDA(cudaStreamSynchronize(s));
        return ML_OK;
    }
    // the PCS degree: every round on the device (transcript in HBM), one synchronisation at the end
    if (rounds == 0) return ML_OK;
    const int max_nb = sumcheck_max_blocks();
    Scratch blk(s);
    const size_t off_tr = 0, off_r = 128, off_prev = 160, off_sc = 192, off_rs = off_sc + 2 * 64 * 16, off_part = off_rs + 64 * 16,
                 total = off_part + (size_t)(2 * max_nb + 2) * 16;
    MLB_TRY(blk.alloc(total));
    uint8_t* base = blk.as<uint8_t>();
    DevTranscript* tr_dev = (DevTranscript*)(base + off_tr);
    fe *r_dev = (fe*)(base + off_r), *prev_dev = (fe*)(base + off_prev), *sc_dev = (fe*)(base + off_sc), *rs_dev = (fe*)(base + off_rs),
       *partials = (fe*)(base + off_part);
    MLB_CUDA(cudaMemsetAsync(base, 0, off_part, s));
    MLB_TRY(h2d(tr_dev, &t->sha, sizeof(DevTranscript), s));
    MLB_TRY(h2d(prev_dev, sum, 16, s));
    size_t k = 0;
    bool have_partials = false;
    int nb = 0;
    for (; k < rounds && sc->height > ((size_t)1 << TAIL_LOG); k++) {
        if (!have_partials) MLB_TRY(sumcheck_sums_partials_launch(sc->matrix, sc->delta, sc->height, partials, &nb, s));
        MLB_TRY(chain_sumcheck_finish_launch(partials, nb, prev_dev, tr_dev, nullptr, 0, nullptr, sc_dev + 2 * k, r_dev, s));
        MLB_CUDA(cudaMemcpyAsync(rs_dev + k, r_dev, 16, cudaMemcpyDeviceToDevice, s));
        // round k+1 runs as separate kernels again iff its height is still above the tail size: fuse its sums into this fold
        have_partials = (sc->height >> 1) > ((size_t)1 << TAIL_LOG) && k + 1 < rounds;
        if (have_partials) MLB_TRY(sumcheck_fold_sums_launch(sc->matrix, sc->delta, sc->height, r_dev, partials, &nb, s));
        else MLB_TRY(sumcheck_fold_launch(sc->matrix, sc->delta, sc->height, 0, r_dev, s));
        sc->height >>= 1;
    }
    if (k < rounds) {
        MLB_TRY(chain_sumcheck_tail_launch(sc->matrix, sc->delta, sc->height, prev_dev, tr_dev, sc_dev + 2 * k, rs_dev + k, s));
        sc->height = 1;
    }
    std::vector<uint8_t> host(off_part);
    MLB_TRY(d2h_sync(host.data(), base, off_part, s));
    memcpy(coeffs_out, host.data() + off_sc, rounds * 32);
    memcpy(randoms_out, host.data() + off_rs, rounds * 16);
    memcpy(&t->sha, host.data() + off_tr, sizeof(DevTranscript));
    return ML_OK;
}
// ---- width-w tables (System path): System::build_tables sumcheck.rs:22-38, partial_sum :204-232, fold :234-247,
// compute_sumcheck_polynomials :147-202 with the composition given as a sparse polynomial over the row
void free_wsumcheck(ml_wsumcheck* w) {
    if (!w) return;
    pfree(w->matrix, w->stream); pfree(w->delta, w->stream); pfree(w->coef, w->stream);
    pfree(w->len, w->stream); pfree(w->off, w->stream); pfree(w->cols, w->stream);
    delete w;
}
static int wsumcheck_build(Ctx* ctx, const uint8_t* row_point, size_t n_vars, const void* matrix, bool on_device, size_t width, size_t height,
                           cudaStream_t s, ml_wsumcheck** out) {
    if (n_vars >= 40 || ((size_t)1 << n_vars) != height) { set_error("trace height must be 2^n_vars"); return ML_ERR_SIZE; }
    if (width == 0 || width > (size_t)wsumcheck_limits(0)) { set_error("trace width must be 1..%d", wsumcheck_limits(0)); return ML_ERR_ARG; }
    ml_wsumcheck* w = new ml_wsumcheck();
    w->width = width; w->height = height; w->stream = s;
    if (pmalloc((void**)&w->matrix, height * width * 16, s) != ML_OK || pmalloc((void**)&w->delta, height * 16, s) != ML_OK) {
        free_wsumcheck(w);
        return ML_ERR_ALLOC;
    }
    cudaError_t e = cudaMemcpyAsync(w->matrix, matrix, height * width * 16, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) { free_wsumcheck(w); set_error("copy failed: %s", cudaGetErrorString(e)); return ML_ERR_CUDA; }
    std::vector<hfe> pts(n_vars);
    for (size_t i = 0; i < n_vars; i++) pts[i] = hfe_load(row_point + 16 * i);
    int st = eq_table_launch(ctx, pts.data(), n_vars, w->delta, s);  // Mask::evaluate over every index (:26-31)
    if (st == ML_OK && cudaStreamSynchronize(s) != cudaSuccess) st = ML_ERR_CUDA;
    if (st != ML_OK) { free_wsumcheck(w); return st; }
    *out = w;
    return ML_OK;
}
int ml_wsumcheck_build(const uint8_t* row_point, size_t n_vars, const uint8_t* matrix, size_t width, size_t height, ml_wsumcheck** out) {
    API_BEGIN
    return wsumcheck_build(ctx, row_point, n_vars, matrix, false, width, height, lib_stream(ctx), out);
}
int ml_wsumcheck_build_dev(const uint8_t* row_point, size_t n_vars, const void* matrix_dev, size_t width, size_t height, void* stream,
                           ml_wsumcheck** out) {
    API_BEGIN
    return wsumcheck_build(ctx, row_point, n_vars, matrix_dev, true, width, height, ST(stream), out);
}
void ml_wsumcheck_free(ml_wsumcheck* w) { free_wsumcheck(w); }
size_t ml_wsumcheck_height(const ml_wsumcheck* w) { return w->height; }
size_t ml_wsumcheck_width(const ml_wsumcheck* w) { return w->width; }
int ml_wsumcheck_set_composition(ml_wsumcheck* w, size_t n_terms, const uint8_t* coefs, const uint32_t* term_lens, const uint32_t* term_cols) {
    API_BEGIN
    (void)ctx;
    std::vector<uint32_t> off;
    size_t total = 0;
    MLB_TRY(wsumcheck_check_terms(w->width, n_terms, term_lens, term_cols, off, &total));
    cudaStream_t s = w->stream;
    pfree(w->coef, s); pfree(w->len, s); pfree(w->off, s); pfree(w->cols, s);
    w->coef = nullptr; w->len = w->off = w->cols = nullptr;
    MLB_TRY(pmalloc((void**)&w->coef, (n_terms ? n_terms : 1) * 16, s));
    MLB_TRY(pmalloc((void**)&w->len, (n_terms ? n_terms : 1) * 4, s));
    MLB_TRY(pmalloc((void**)&w->off, (n_terms ? n_terms : 1) * 4, s));
    MLB_TRY(pmalloc((void**)&w->cols, (total ? total : 1) * 4, s));
    MLB_TRY(h2d(w->coef, coefs, n_terms * 16, s));
    MLB_TRY(h2d(w->len, term_lens, n_terms * 4, s));
    MLB_TRY(h2d(w->off, off.data(), n_terms * 4, s));
    MLB_TRY(h2d(w->cols, term_cols, total * 4, s));
    MLB_CUDA(cudaStreamSynchronize(s));  // off is a host temporary
    w->n_terms = n_terms; w->n_cols = total;
    return ML_OK;
}
int ml_wsumcheck_tables(const ml_wsumcheck* w, uint8_t* matrix_out, uint8_t* delta_out) {
    API_BEGIN
    (void)ctx;
    MLB_TRY(d2h_sync(matrix_out, w->matrix, w->height * w->width * 16, w->stream));
    return d2h_sync(delta_out, w->delta, w->height * 16, w->stream);
}
static int wpartial(ml_wsumcheck* w, hfe r, hfe* out) {
    if (w->height < 2) { *out = 0; return ML_OK; }
    return wsumcheck_partial_sum_launch(w->matrix, w->delta, w->height, w->width, r, w->coef, w->len, w->off, w->cols, w->n_terms, w->n_cols, out, w->stream);
}
int ml_wsumcheck_partial_sum(ml_wsumcheck* w, const uint8_t r[16], uint8_t out[16]) {
    API_BEGIN
    (void)ctx;
    hfe o;
    MLB_TRY(wpartial(w, hfe_load(r), &o));
    hfe_store(out, o);
    return ML_OK;
}
int ml_wsumcheck_fold(ml_wsumcheck* w, const uint8_t r[16]) {
    API_BEGIN
    (void)ctx;
    MLB_TRY(wsumcheck_fold_launch(w->matrix, w->delta, w->height, w->width, hfe_load(r), w->stream));
    w->height >>= 1;
    return ML_OK;
}
int ml_wsumcheck_compute_polynomials(ml_wsumcheck* w, size_t composition_degree, ml_transcript* t, const uint8_t sum[16], uint8_t* coeffs_out,
                                     uint8_t* randoms_out) {
    API_BEGIN
    (void)ctx;
    const size_t td = composition_degree + 1;  // :159
    if (td > 16) { set_error("composition_degree too large"); return ML_ERR_ARG; }
    const size_t rounds = w->height ? ilog2(w->height) : 0;
    static const bool host_rounds = getenv("MLB_WSUMCHECK_HOST_ROUNDS") != nullptr;  // the round-1 path, kept for comparison
    if (td <= (size_t)W_MAX_TD && rounds > 0 && !host_rounds) {
        // every round on the device: points kernel -> one-CTA bookkeeping (Lagrange matrix, transcript in HBM, challenge) -> fold
        // reading the challenge from HBM; the last WTAIL_LOG rounds in one CTA; one synchronisation at the end
        cudaStream_t s = w->stream;
        std::vector<uint8_t> lag_h;
        MLB_TRY(wsumcheck_lagrange(td, lag_h));
        const int max_nb = sumcheck_max_blocks();
        Scratch blk(s);
        const size_t off_tr = 0, off_r = 128, off_prev = 144, off_lag = 160, off_co = off_lag + 32 * 16, off_rs = off_co + 64 * W_MAX_TD * 16,
                     off_part = off_rs + 64 * 16, total = off_part + ((size_t)max_nb + 1) * W_MAX_TD * 16;
        MLB_TRY(blk.alloc(total));
        uint8_t* base = blk.as<uint8_t>();
        DevTranscript* tr_dev = (DevTranscript*)(base + off_tr);
        fe *r_dev = (fe*)(base + off_r), *prev_dev = (fe*)(base + off_prev), *lag_dev = (fe*)(base + off_lag), *co_dev = (fe*)(base + off_co),
           *rs_dev = (fe*)(base + off_rs), *partials = (fe*)(base + off_part);
        MLB_TRY(h2d(tr_dev, &t->sha, sizeof(DevTranscript), s));
        MLB_TRY(h2d(prev_dev, sum, 16, s));
        MLB_TRY(h2d(lag_dev, lag_h.data(), lag_h.size(), s));
        const WTerms terms{w->coef, w->len, w->off, w->cols, (int)w->n_terms, (int)w->n_cols};
        size_t k = 0;
        for (; k < rounds && w->height > ((size_t)1 << WTAIL_LOG); k++) {
            int nb = 0;
            MLB_TRY(wsumcheck_points_partials_launch(w->matrix, w->delta, w->height, w->width, terms, (int)td, partials, &nb, s));
            MLB_TRY(wchain_finish_launch(partials, nb, (int)td, lag_dev, prev_dev, tr_dev, co_dev + k * td, rs_dev + k, r_dev, s));
            MLB_TRY(wsumcheck_fold_dev_launch(w->matrix, w->delta, w->height, w->width, r_dev, s));
            w->height >>= 1;
        }
        if (k < rounds) {
            MLB_TRY(wchain_tail_launch(w->matrix, w->delta, w->height, (int)w->width, terms, (int)td, lag_dev, prev_dev, tr_dev, co_dev + k * td,
                                       rs_dev + k, s));
            w->height = 1;
        }
        std::vector<uint8_t> host(off_part);
        MLB_TRY(d2h_sync(host.data(), base, off_part, s));  // also keeps lag_h alive until its upload has run
        memcpy(coeffs_out, host.data() + off_co, rounds * td * 16);
        memcpy(randoms_out, host.data() + off_rs, rounds * 16);
        memcpy(&t->sha, host.data() + off_tr, sizeof(DevTranscript));
        return ML_OK;
    }
    hfe prev = hfe_load(sum);
    std::vector<hfe> evals(td + 1), coeffs;
    for (size_t k = 0; k < rounds; k++) {
        // :185-187 — every point of the round in one pass when td <= 4, else one pass per point
        if (w->height >= 2 && td <= 4) {
            MLB_TRY(wsumcheck_points_launch(w->matrix, w->delta, w->height, w->width, w->coef, w->len, w->off, w->cols, w->n_terms, w->n_cols,
                                            (int)td, &evals[1], w->stream));
        } else {
            for (size_t i = 1; i <= td; i++) MLB_TRY(wpartial(w, hfe_new((hfe)i), &evals[i]));
        }
        evals[0] = hfe_sub(prev, evals[1]);                                                 // :188
        interpolate(evals, coeffs);                                                         // :189-192
        for (size_t i = 1; i <= td; i++) { hfe_store(coeffs_out + 16 * (k * td + i - 1), coeffs[i]); absorb_fe(t, coeffs[i]); }
        hfe r = challenge(t);                                                               // :198
        prev = poly_eval(coeffs, r);                                                        // :199
        MLB_TRY(wsumcheck_fold_launch(w->matrix, w->delta, w->height, w->width, r, w->stream));  // :200
        w->height >>= 1;
        hfe_store(randoms_out + 16 * k, r);
    }
    MLB_CUDA(cudaStreamSynchronize(w->stream));
    return ML_OK;
}
// PolynomialEvals::interpolate (src/polynomials.rs:51-86): coefficients of the degree < n polynomial through (i, evals[i]), i = 0..n-1.
// The reference builds every Lagrange basis polynomial with poly_mul (O(n^3)); the interpolant is unique, so the same coefficients come
// from the master polynomial P(x) = prod (x - m) divided synthetically by (x - j), O(n^2).  Host scalars: the reference only calls it
// with n = total_degree + 1 <= 4 (sumcheck.rs:189-192).
int ml_poly_interpolate(const uint8_t* evals, size_t n, uint8_t* coeffs_out) {
    if (n == 0) return ML_OK;
    if (n > ((size_t)1 << 14)) { set_error("interpolate: at most 2^14 points (host scalar routine)"); return ML_ERR_ARG; }
    std::vector<hfe> P(n + 1, 0), q(n), c(n, 0), fact(n, 1);
    P[0] = 1;  // P(x) = prod_{m<n} (x - m), ascending coefficients
    for (size_t m = 0; m < n; m++) {
        const hfe xm = hfe_new((hfe)m);
        for (size_t i = m + 1; i-- > 0;) P[i + 1] = hfe_add(P[i + 1], P[i]), P[i] = hfe_neg(hfe_mul(P[i], xm));
    }
    for (size_t i = 1; i < n; i++) fact[i] = hfe_mul(fact[i - 1], hfe_new((hfe)i));
    for (size_t j = 0; j < n; j++) {
        const hfe xj = hfe_new((hfe)j);
        // q = P / (x - j): q[n-1] = P[n], q[i-1] = P[i] + j * q[i]
        q[n - 1] = P[n];
        for (size_t i = n - 1; i >= 1; i--) q[i - 1] = hfe_add(P[i], hfe_mul(xj, q[i]));
        // denom = prod_{m != j} (j - m) = j! * (n-1-j)! * (-1)^(n-1-j)
        hfe denom = hfe_mul(fact[j], fact[n - 1 - j]);
        if ((n - 1 - j) & 1) denom = hfe_neg(denom);
        const hfe scale = hfe_div(hfe_load(evals + 16 * j), denom);
        for (size_t i = 0; i < n; i++) c[i] = hfe_add(c[i], hfe_mul(scale, q[i]));
    }
    for (size_t i = 0; i < n; i++) hfe_store(coeffs_out + 16 * i, c[i]);
    return ML_OK;
}
// Polynomial::evaluate_over_domain (src/polynomials.rs:16-28): evals[i] = p(i), i = 0..n-1; one thread per point, Horner
__global__ void poly_eval_domain_kernel(const fe* __restrict__ coeffs, size_t n, fe* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const fe x = fe{{(uint32_t)i, (uint32_t)(i >> 32), 0u, 0u}};
    fe acc = fe_zero();
    for (size_t k = n; k-- > 0;) acc = fe_add(fe_mul(acc, x), fe_load_nc(coeffs + k));
    fe_store(out + i, acc);
}
int ml_poly_evaluate_over_domain(const uint8_t* coeffs, size_t n, uint8_t* evals_out) {
    API_BEGIN
    if (n == 0) return ML_OK;
    cudaStream_t s = lib_stream(ctx);
    Scratch dc(s), de(s);
    MLB_TRY(dc.alloc(n * 16));
    MLB_TRY(de.alloc(n * 16));
    MLB_TRY(h2d(dc.p, coeffs, n * 16, s));
    poly_eval_domain_kernel<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(dc.as<fe>(), n, de.as<fe>());
    MLB_KERNEL_CHECK();
    return d2h_sync(evals_out, de.p, n * 16, s);
}
int ml_delta_evaluate(const uint8_t* data, const uint8_t* points, size_t n, uint8_t out[16]) {
    std::vector<hfe> a(n), b(n);
    for (size_t i = 0; i < n; i++) { a[i] = hfe_load(data + 16 * i); b[i] = hfe_load(points + 16 * i); }
    hfe_store(out, delta_evaluate(a.data(), b.data(), n));
    return ML_OK;
}

// ================================================================== multilinear PCS
int ml_pcs_prove_dev(const uint8_t* inputs, size_t n_vars, const uint8_t output[16], const void* evals_dev, size_t n, ml_transcript* t,
                     void* stream, ml_pcs_proof** out) {
    API_BEGIN
    cudaStream_t s = ST(stream);
    if (!is_pow2(n) || n < 2 || n_vars >= 40 || ((size_t)1 << n_vars) != n) { set_error("PCSProof::prove: need 2^n_vars == evals.len() >= 2"); return ML_ERR_SIZE; }
    const size_t domain = n << ML_LOG_BLOWUP;  // :97
    fe* code;
    MLB_TRY(encode_poly(ctx, (const fe*)evals_dev, n, &code, s));  // :101-107
    // PCSProverData::fold (:43-76)
    ml_fri* f;
    MLB_TRY(fri_new_unabsorbed(&f, code, domain, true, s));  // :30 (root absorbed on the device by the chain)
    ml_sumcheck* sc = nullptr;
    int st = sumcheck_build(ctx, inputs, n_vars, evals_dev, true, n, s, &sc);  // :31
    ml_pcs_proof* p = new ml_pcs_proof();
    const size_t num_steps = ilog2(domain) - ML_LOG_BLOWUP;  // :52
    p->sumcheck.resize(2 * num_steps);
    // rounds :58-73 — sumcheck polynomial, shared challenge, table fold, FRI fold, commit — without host round trips
    if (st == ML_OK) st = fold_chain_dev(ctx, f, nullptr, sc, hfe_load(output), p->sumcheck.data(), 0, true, t, s);
    if (st == ML_OK) st = assemble_fri_proof(f, domain, t, &p->fri, s);  // :113-129
    if (st == ML_OK) {
        p->inputs.resize(n_vars);
        for (size_t i = 0; i < n_vars; i++) p->inputs[i] = hfe_load(inputs + 16 * i);
        p->output = hfe_load(output);
    }
    free_fri(f);
    free_sumcheck(sc);
    if (st != ML_OK) { delete p; return st; }
    *out = p;
    return ML_OK;
}
int ml_pcs_prove(const uint8_t* inputs, size_t n_vars, const uint8_t output[16], const uint8_t* evals, size_t n, ml_transcript* t,
                 ml_pcs_proof** out) {
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    Scratch d(s);
    MLB_TRY(d.alloc(n * 16));
    MLB_TRY(h2d(d.p, evals, n * 16, s));
    return ml_pcs_prove_dev(inputs, n_vars, output, d.p, n, t, s, out);
}
int ml_pcs_verify(const ml_pcs_proof* p, ml_transcript* t) {  // multilinear_pcs.rs:138-190
    const ml_fri_proof* fp = &p->fri;
    if (fp->queries.size() != ML_NUM_QUERIES) return ML_V_WRONG_NUM_QUERIES;
    const size_t n = fp->commitments.size() / 32;
    if (n == 0 || 2 * n != p->sumcheck.size() || n != p->inputs.size()) { set_error("assert_eq!(n, ...) failed"); return ML_ERR_SIZE; }
    std::vector<hfe> rs(n);
    for (size_t i = 0; i < n; i++) {
        t->sha.update(&fp->commitments[32 * i], 32);
        absorb_fe(t, p->sumcheck[2 * i]);
        absorb_fe(t, p->sumcheck[2 * i + 1]);
        rs[i] = challenge(t);
    }
    absorb_fe(t, fp->last_elem);
    int st = sumcheck_replay(p->sumcheck, p->output, p->inputs, rs, fp->last_elem);
    if (st != ML_V_OK) return st;
    return fri_verify_queries(fp, t, rs.data());
}
void ml_pcs_proof_free(ml_pcs_proof* p) { delete p; }
const ml_fri_proof* ml_pcs_proof_fri(const ml_pcs_proof* p) { return &p->fri; }
size_t ml_pcs_proof_num_rounds(const ml_pcs_proof* p) { return p->sumcheck.size() / 2; }
int ml_pcs_proof_sumcheck_coeffs(const ml_pcs_proof* p, uint8_t* out) {
    for (size_t i = 0; i < p->sumcheck.size(); i++) hfe_store(out + 16 * i, p->sumcheck[i]);
    return ML_OK;
}

// ================================================================== batched FRI / PCS
int ml_fingerprint(const uint8_t r[16], const uint8_t* coeffs, size_t n, uint8_t out[16]) {
    std::vector<hfe> c(n);
    for (size_t i = 0; i < n; i++) c[i] = hfe_load(coeffs + 16 * i);
    hfe_store(out, fingerprint_host(hfe_load(r), c.data(), n));
    return ML_OK;
}
int ml_batched_fri_prove(const uint8_t* const* codes, size_t n_codes, size_t n, const uint8_t* gen_pows, size_t gen_pows_len,
                         ml_transcript* t, ml_bfri_proof** out) {
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    if (n_codes == 0) { set_error("Codes must not be empty"); return ML_ERR_SIZE; }
    MLB_TRY(check_code_len(n));
    if (gen_pows && gen_pows_len != n) { set_error("gen_pows.len() must equal the domain size"); return ML_ERR_SIZE; }
    BatchedFri b;
    b.n = n;
    for (size_t j = 0; j < n_codes; j++) {
        fe* c;
        b.stream = s;
        MLB_TRY(pmalloc((void**)&c, n * 16, s));
        b.codes.push_back(c);
        MLB_TRY(h2d(c, codes[j], n * 16, s));
    }
    MLB_TRY(bfri_init(&b, t, s));
    // batched first fold (:193-195) + the remaining fold steps (:198-201), transcript advanced on the device
    ChainHooks hooks;
    hooks.first_fold = [&](const fe* r_dev, fe** next, bool* owns) { *owns = true; size_t hn = 0; return bfri_first_fold_dev(ctx, &b, r_dev, next, &hn, s); };
    MLB_TRY(fold_chain_dev(ctx, b.fri, &hooks, nullptr, 0, nullptr, 0, false, t, s));
    ml_bfri_proof* p = new ml_bfri_proof();
    int st = bfri_assemble(&b, t, p, s);
    if (st != ML_OK) { delete p; return st; }
    *out = p;
    return ML_OK;
}
// ---- BatchedFriProverData step by step (batched_fri.rs:9-14, 41-225): the host-transcript mirror of the struct's own methods
}  // extern "C"
struct ml_bfri {
    mlbp::BatchedFri b;
};
static int bfri_upload_codes(ml_bfri* h, const uint8_t* const* codes, size_t n_codes, size_t n, cudaStream_t s) {
    if (n_codes == 0) { set_error("Codes must not be empty"); return ML_ERR_SIZE; }
    MLB_TRY(check_code_len(n));
    h->b.n = n;
    h->b.stream = s;
    for (size_t j = 0; j < n_codes; j++) {
        fe* c;
        MLB_TRY(pmalloc((void**)&c, n * 16, s));
        h->b.codes.push_back(c);
        MLB_TRY(h2d(c, codes[j], n * 16, s));
    }
    return ML_OK;
}
extern "C" {
int ml_bfri_init(const uint8_t* const* codes, size_t n_codes, size_t n, ml_transcript* t, ml_bfri** out) {  // init :41-99
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    ml_bfri* h = new ml_bfri();
    int st = bfri_upload_codes(h, codes, n_codes, n, s);
    if (st == ML_OK) st = bfri_init(&h->b, t, s);
    if (st != ML_OK) { delete h; return st; }
    *out = h;
    return ML_OK;
}
int ml_bfri_batched_fold_step(ml_bfri* h, const uint8_t* gen_pows, size_t gen_pows_len, const uint8_t r[16], ml_transcript* t) {  // :101-181
    API_BEGIN
    if (gen_pows) MLB_TRY(check_gen_pows(h->b.fri, gen_pows, gen_pows_len));
    return bfri_batched_fold_step(ctx, &h->b, hfe_load(r), t, lib_stream(ctx));
}
int ml_bfri_fold(const uint8_t* gen_pows, size_t gen_pows_len, const uint8_t* const* codes, size_t n_codes, size_t n, ml_transcript* t,
                 ml_bfri** out) {  // fold :183-205 — transcript advanced on the device, one synchronisation
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    if (gen_pows && gen_pows_len != n) { set_error("gen_pows.len() must equal the domain size"); return ML_ERR_SIZE; }
    ml_bfri* h = new ml_bfri();
    int st = bfri_upload_codes(h, codes, n_codes, n, s);
    if (st == ML_OK) st = bfri_init(&h->b, t, s);
    if (st == ML_OK && gen_pows) st = check_gen_pows(h->b.fri, gen_pows, gen_pows_len);
    if (st == ML_OK) {
        ChainHooks hooks;
        mlbp::BatchedFri* b = &h->b;
        hooks.first_fold = [=](const fe* r_dev, fe** next, bool* owns) { *owns = true; size_t hn = 0; return bfri_first_fold_dev(ctx, b, r_dev, next, &hn, s); };
        st = fold_chain_dev(ctx, h->b.fri, &hooks, nullptr, 0, nullptr, 0, false, t, s);
    }
    if (st != ML_OK) { delete h; return st; }
    *out = h;
    return ML_OK;
}
void ml_bfri_free(ml_bfri* h) { delete h; }
ml_fri* ml_bfri_fri_data(ml_bfri* h) { return h->b.fri; }                     // fri_data (:13), borrowed
const ml_merkle* ml_bfri_batch_layer(const ml_bfri* h) { return h->b.batch_layer; }       // batch_layer (:11), borrowed
size_t ml_bfri_num_codes(const ml_bfri* h) { return h->b.codes.size(); }
int ml_bfri_fingerprint_r(const ml_bfri* h, uint8_t out[16]) { hfe_store(out, h->b.fingerprint_r); return ML_OK; }  // fingerprint_r (:12)
// open_query_at (:207-225): batch_values n_codes x 32 B, batch path (log2(n/2) digests + dirs), then the FRI query as ml_fri_open_query_at
int ml_bfri_open_query_at(const ml_bfri* h, size_t index, uint8_t* batch_values, uint8_t* batch_digests, uint8_t* batch_dirs, size_t* batch_path_len,
                          uint8_t* values, uint8_t* digests, uint8_t* dirs, size_t* path_lens) {
    API_BEGIN
    if (index >= h->b.n / 2) { set_error("open_query_at: Index out of bounds"); return ML_ERR_OUT_OF_RANGE; }
    std::vector<size_t> idx(1, index);
    std::vector<BQueryH> q;
    MLB_TRY(bfri_open_queries(const_cast<mlbp::BatchedFri*>(&h->b), idx, q, lib_stream(ctx)));
    const PathH& bp = q[0].batch_path;
    memcpy(batch_values, bp.value.data(), bp.value.size());
    memcpy(batch_digests, bp.digests.data(), bp.digests.size());
    memcpy(batch_dirs, bp.dirs.data(), bp.dirs.size());
    *batch_path_len = bp.dirs.size();
    size_t doff = 0;
    for (size_t j = 0; j < q[0].query.paths.size(); j++) {
        const PathH& p = q[0].query.paths[j];
        memcpy(values + 32 * j, p.value.data(), 32);
        memcpy(digests + 32 * doff, p.digests.data(), p.digests.size());
        memcpy(dirs + doff, p.dirs.data(), p.dirs.size());
        path_lens[j] = p.dirs.size();
        doff += p.dirs.size();
    }
    return ML_OK;
}
int ml_batched_fri_verify(const ml_bfri_proof* p) {  // batched_fri.rs:320-354
    ml_transcript t;
    t.sha.update(p->batch_commitment, 32);
    hfe fr = challenge(&t);
    absorb_fe(&t, fr);
    const size_t nc = p->commitments.size() / 32;
    std::vector<hfe> rs(nc + 1);
    rs[0] = challenge(&t);
    for (size_t i = 0; i < nc; i++) {
        t.sha.update(&p->commitments[32 * i], 32);
        rs[i + 1] = challenge(&t);
    }
    absorb_fe(&t, p->last_elem);
    return bfri_verify_queries(p, &t, rs.data(), fr);
}
void ml_bfri_proof_free(ml_bfri_proof* p) { delete p; }
int ml_bfri_proof_batch_commitment(const ml_bfri_proof* p, uint8_t out[32]) { memcpy(out, p->batch_commitment, 32); return ML_OK; }
size_t ml_bfri_proof_num_commitments(const ml_bfri_proof* p) { return p->commitments.size() / 32; }
int ml_bfri_proof_commitments(const ml_bfri_proof* p, uint8_t* out) { memcpy(out, p->commitments.data(), p->commitments.size()); return ML_OK; }
int ml_bfri_proof_last(const ml_bfri_proof* p, uint8_t last_elem[16], uint8_t last_random[32]) {
    hfe_store(last_elem, p->last_elem);
    memcpy(last_random, p->last_random, 32);
    return ML_OK;
}
size_t ml_bfri_proof_serialized_len(const ml_bfri_proof* p) { Writer w(nullptr); write_bfri_proof(p, w); return w.n; }
int ml_bfri_proof_serialize(const ml_bfri_proof* p, uint8_t* out) { Writer w(out); write_bfri_proof(p, w); return ML_OK; }

int ml_batched_pcs_prove_dev(const uint8_t* inputs, size_t n_vars, const uint8_t* outputs, size_t n_polys, const void* const* evals_dev,
                             size_t n, ml_transcript* t, void* stream, ml_bpcs_proof** out) {
    API_BEGIN
    cudaStream_t s = ST(stream);
    if (n_polys == 0 || !is_pow2(n) || n < 2 || n_vars >= 40 || ((size_t)1 << n_vars) != n) { set_error("BatchedPCSProof::prove: bad sizes"); return ML_ERR_SIZE; }
    const size_t domain = n << ML_LOG_BLOWUP;  // batched_pcs.rs:136
    BatchedFri b;
    b.n = domain;
    b.stream = s;
    for (size_t j = 0; j < n_polys; j++) {  // :144-149
        fe* code;
        MLB_TRY(encode_poly(ctx, (const fe*)evals_dev[j], n, &code, s));
        b.codes.push_back(code);
    }
    // BatchedPCSProverData::init (:37-77)
    t->sha.update(inputs, n_vars * 16);    // :44-46
    t->sha.update(outputs, n_polys * 16);  // :47-49
    MLB_TRY(bfri_init(&b, t, s));
    const hfe fr = b.fingerprint_r;
    // fingerprinted evaluation table (:55-63) straight into the sumcheck matrix
    ml_sumcheck* sc = new ml_sumcheck();
    sc->height = n;
    sc->stream = s;
    Scratch dptrs(s);
    int st = ML_OK;
    if (pmalloc((void**)&sc->matrix, n * 16, s) != ML_OK || pmalloc((void**)&sc->delta, n * 16, s) != ML_OK) st = ML_ERR_ALLOC;
    if (st == ML_OK) st = dptrs.alloc(n_polys * sizeof(void*));
    if (st == ML_OK) st = h2d(dptrs.p, evals_dev, n_polys * sizeof(void*), s);
    if (st == ML_OK) st = fingerprint_rows_launch((const fe* const*)dptrs.p, n_polys, n, fr, sc->matrix, s);
    std::vector<hfe> pts(n_vars), outs(n_polys);
    for (size_t i = 0; i < n_vars; i++) pts[i] = hfe_load(inputs + 16 * i);
    for (size_t i = 0; i < n_polys; i++) outs[i] = hfe_load(outputs + 16 * i);
    if (st == ML_OK) st = eq_table_launch(ctx, pts.data(), n_vars, sc->delta, s);  // :66-67
    if (st == ML_OK && cudaStreamSynchronize(s) != cudaSuccess) st = ML_ERR_CUDA;
    ml_bpcs_proof* p = new ml_bpcs_proof();
    const size_t num_steps = ilog2(domain) - ML_LOG_BLOWUP;  // :90
    p->sumcheck.resize(2 * num_steps);
    hfe prev = fingerprint_host(fr, outs.data(), n_polys);   // :92-94
    ChainHooks hooks;
    hooks.first_fold = [&](const fe* r_dev, fe** next, bool* owns) { *owns = true; size_t hn = 0; return bfri_first_fold_dev(ctx, &b, r_dev, next, &hn, s); };
    if (st == ML_OK) st = fold_chain_dev(ctx, b.fri, &hooks, sc, prev, p->sumcheck.data(), 0, false, t, s);  // :100-123
    if (st == ML_OK) st = bfri_assemble(&b, t, &p->fri, s);  // :155-173
    free_sumcheck(sc);
    if (st != ML_OK) { delete p; return st; }
    p->inputs = pts;
    p->outputs = outs;
    *out = p;
    return ML_OK;
}
int ml_batched_pcs_prove(const uint8_t* inputs, size_t n_vars, const uint8_t* outputs, size_t n_polys, const uint8_t* const* evals, size_t n,
                         ml_transcript* t, ml_bpcs_proof** out) {
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    std::vector<void*> dev(n_polys, nullptr);
    int st = ML_OK;
    for (size_t j = 0; j < n_polys && st == ML_OK; j++) {
        if (pmalloc(&dev[j], n * 16 + 16, s) != ML_OK) { st = ML_ERR_ALLOC; break; }
        st = h2d(dev[j], evals[j], n * 16, s);
    }
    if (st == ML_OK) st = ml_batched_pcs_prove_dev(inputs, n_vars, outputs, n_polys, dev.data(), n, t, s, out);
    cudaStreamSynchronize(s);
    for (void* d : dev) pfree(d, s);
    return st;
}
int ml_batched_pcs_verify(const ml_bpcs_proof* p, ml_transcript* t) {  // batched_pcs.rs:182-253
    const ml_bfri_proof* fp = &p->fri;
    if (fp->queries.size() != ML_NUM_QUERIES) return ML_V_WRONG_NUM_QUERIES;
    const size_t n = fp->commitments.size() / 32 + 1;
    if (2 * n != p->sumcheck.size() || n != p->inputs.size()) { set_error("assert_eq!(n, ...) failed"); return ML_ERR_SIZE; }
    std::vector<hfe> rs(n);
    for (hfe x : p->inputs) absorb_fe(t, x);
    for (hfe x : p->outputs) absorb_fe(t, x);
    hfe fr = 0;
    for (size_t i = 0; i < n; i++) {
        if (i == 0) {
            t->sha.update(fp->batch_commitment, 32);
            fr = challenge(t);
            absorb_fe(t, fr);
        } else t->sha.update(&fp->commitments[32 * (i - 1)], 32);
        absorb_fe(t, p->sumcheck[2 * i]);
        absorb_fe(t, p->sumcheck[2 * i + 1]);
        rs[i] = challenge(t);
    }
    absorb_fe(t, fp->last_elem);
    hfe sum = fingerprint_host(fr, p->outputs.data(), p->outputs.size());
    int st = sumcheck_replay(p->sumcheck, sum, p->inputs, rs, fp->last_elem);
    if (st != ML_V_OK) return st;
    return bfri_verify_queries(fp, t, rs.data(), fr);
}
void ml_bpcs_proof_free(ml_bpcs_proof* p) { delete p; }
const ml_bfri_proof* ml_bpcs_proof_fri(const ml_bpcs_proof* p) { return &p->fri; }
size_t ml_bpcs_proof_num_rounds(const ml_bpcs_proof* p) { return p->sumcheck.size() / 2; }
int ml_bpcs_proof_sumcheck_coeffs(const ml_bpcs_proof* p, uint8_t* out) {
    for (size_t i = 0; i < p->sumcheck.size(); i++) hfe_store(out + 16 * i, p->sumcheck[i]);
    return ML_OK;
}

// ================================================================== sharded batched commit (config 5)
int ml_batched_leaf_subtree_dev(const void* const* pairs_dev, size_t n_codes, size_t leaf_count, void* stream, uint8_t root_out[32]) {
    API_BEGIN
    (void)ctx;
    cudaStream_t s = ST(stream);
    if (!is_pow2(leaf_count) || n_codes == 0) { set_error("leaf_count must be a power of two"); return ML_ERR_NOT_POW2; }
    Scratch dig(s), ptrs(s);
    MLB_TRY(dig.alloc(2 * leaf_count * 32));
    MLB_TRY(ptrs.alloc(n_codes * sizeof(void*)));
    MLB_TRY(h2d(ptrs.p, pairs_dev, n_codes * sizeof(void*), s));
    MLB_TRY(merkle_batched_pairs_launch((const uint8_t* const*)ptrs.p, n_codes, leaf_count, dig.as<uint8_t>(), s));
    const int top = (int)ilog2(leaf_count);
    return d2h_sync(root_out, dig.as<uint8_t>() + 32 * merkle_layer_offset(leaf_count, top), 32, s);
}
// ReedSolomonPairs of a code, laid out for the leaf-range exchange: pair i of local polynomial `pl` goes to
// out[((dest * n_local + pl) * rows + i % rows) * 32], dest = i / rows, rows = (n_code / 2) / n_ranks
__global__ void pack_pairs_kernel(const fe* __restrict__ code, size_t half, size_t rows, size_t n_local, size_t pl, uint4* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < half; i += stride) {
        const size_t dest = i / rows, r = i - dest * rows;
        uint4* o = out + 2 * ((dest * n_local + pl) * rows + r);
        o[0] = *reinterpret_cast<const uint4*>(code + i);
        o[1] = *reinterpret_cast<const uint4*>(code + i + half);
    }
}
int ml_pack_pairs_dev(const void* code_dev, size_t n_code, size_t n_ranks, size_t n_local_polys, size_t local_index, void* out_dev,
                      void* stream) {
    API_BEGIN
    (void)ctx;
    const size_t half = n_code / 2;
    if (!is_pow2(n_code) || n_ranks == 0 || half % n_ranks != 0 || local_index >= n_local_polys) { set_error("ml_pack_pairs_dev: bad partition"); return ML_ERR_SIZE; }
    size_t blocks = (half + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    pack_pairs_kernel<<<(unsigned)blocks, 256, 0, ST(stream)>>>((const fe*)code_dev, half, half / n_ranks, n_local_polys, local_index, (uint4*)out_dev);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
// Same pairs written straight into the leaf-range owners' receive buffers over NVLink (peer-mapped pointers): the
// exchange is fused into the pack pass, no send buffer and no collective.  Pair i goes to rank dest = i / rows at
// peers.base[dest] + ((poly * rows) + i % rows) * 32, i.e. every rank's buffer is [global poly][row][32 B].
// Warps walk contiguous 32-byte pairs of one destination, so the NVLink writes are full 128-byte lines.
struct PeerBases {
    uint4* base[ML_MAX_PEERS];
};
__global__ void __launch_bounds__(256) pack_pairs_peer_kernel(const fe* __restrict__ code, size_t half, size_t rows, size_t poly, PeerBases peers) {
    // four pairs (128 bytes) in flight per thread: the store pass runs on a small grid, so each thread has to cover the
    // NVLink write latency with its own independent stores
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < half; i += 4 * stride) {
        uint4 x[4], y[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            x[u] = __ldg(reinterpret_cast<const uint4*>(code + i + u * stride));
            y[u] = __ldg(reinterpret_cast<const uint4*>(code + i + u * stride + half));
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const size_t k = i + u * stride, dest = k / rows, r = k - dest * rows;
            uint4* o = peers.base[dest] + 2 * (poly * rows + r);
            o[0] = x[u];
            o[1] = y[u];
        }
    }
    for (; i < half; i += stride) {
        const size_t dest = i / rows, r = i - dest * rows;
        uint4* o = peers.base[dest] + 2 * (poly * rows + r);
        o[0] = __ldg(reinterpret_cast<const uint4*>(code + i));
        o[1] = __ldg(reinterpret_cast<const uint4*>(code + i + half));
    }
}
int ml_pack_pairs_peer_dev(const void* code_dev, size_t n_code, size_t n_ranks, size_t global_poly, void* const* peer_bases, unsigned max_ctas,
                           void* stream) {
    API_BEGIN
    (void)ctx;
    const size_t half = n_code / 2;
    if (!is_pow2(n_code) || n_ranks == 0 || n_ranks > ML_MAX_PEERS || half % n_ranks != 0) { set_error("ml_pack_pairs_peer_dev: bad partition"); return ML_ERR_SIZE; }
    PeerBases pb;
    for (size_t g = 0; g < ML_MAX_PEERS; g++) pb.base[g] = g < n_ranks ? (uint4*)peer_bases[g] : nullptr;
    size_t blocks = (half + 255) / 256;
    const size_t cap = max_ctas ? max_ctas : 148 * 8;
    if (blocks > cap) blocks = cap;
    pack_pairs_peer_kernel<<<(unsigned)blocks, 256, 0, ST(stream)>>>((const fe*)code_dev, half, half / n_ranks, global_poly, pb);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
// Peer-visible device buffers (CUDA IPC): the owner allocates and publishes a 64-byte handle, peers map it.
int ml_ipc_alloc(size_t bytes, void** dev_out, uint8_t handle_out[64]) {
    API_BEGIN
    (void)ctx;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    void* p = nullptr;
    MLB_CUDA(cudaMalloc(&p, bytes));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); set_error("cudaIpcGetMemHandle: %s", cudaGetErrorString(e)); cudaGetLastError(); return ML_ERR_CUDA; }
    memcpy(handle_out, &h, 64);
    *dev_out = p;
    return ML_OK;
}
int ml_ipc_open(const uint8_t handle[64], void** dev_out) {
    API_BEGIN
    (void)ctx;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    MLB_CUDA(cudaIpcOpenMemHandle(dev_out, h, cudaIpcMemLazyEnablePeerAccess));
    return ML_OK;
}
int ml_ipc_close(void* dev) {
    API_BEGIN
    (void)ctx;
    MLB_CUDA(cudaIpcCloseMemHandle(dev));
    return ML_OK;
}
int ml_ipc_free(void* dev) {
    API_BEGIN
    (void)ctx;
    MLB_CUDA(cudaFree(dev));
    return ML_OK;
}
// device-to-device variant of ml_batched_leaf_subtree_dev: the 32-byte subtree root stays in HBM (root_dev) so it can
// feed the NCCL all-gather without a host round trip
int ml_batched_leaf_subtree_root_dev(const void* const* pairs_dev, size_t n_codes, size_t leaf_count, void* root_dev, void* stream) {
    API_BEGIN
    (void)ctx;
    cudaStream_t s = ST(stream);
    if (!is_pow2(leaf_count) || n_codes == 0) { set_error("leaf_count must be a power of two"); return ML_ERR_NOT_POW2; }
    Scratch dig(s), ptrs(s);
    MLB_TRY(dig.alloc(2 * leaf_count * 32));
    MLB_TRY(ptrs.alloc(n_codes * sizeof(void*)));
    MLB_TRY(h2d(ptrs.p, pairs_dev, n_codes * sizeof(void*), s));
    MLB_TRY(merkle_batched_pairs_launch((const uint8_t* const*)ptrs.p, n_codes, leaf_count, dig.as<uint8_t>(), s));
    const int top = (int)ilog2(leaf_count);
    MLB_CUDA(cudaMemcpyAsync(root_dev, dig.as<uint8_t>() + 32 * merkle_layer_offset(leaf_count, top), 32, cudaMemcpyDeviceToDevice, s));
    return ML_OK;
}
// evals -> to_coefficient -> bit_reverse -> reed_solomon into a caller-provided code buffer (batched_pcs.rs:144-149)
int ml_pcs_encode_dev(const void* evals_dev, size_t n, void* code_dev, void* stream) {
    API_BEGIN
    if (!is_pow2(n)) { set_error("evals length must be a power of two"); return ML_ERR_NOT_POW2; }
    return encode_into(ctx, (const fe*)evals_dev, n, (fe*)code_dev, ST(stream));
}
int ml_merkle_top_from_roots(const uint8_t* roots, size_t n_roots, uint8_t root_out[32]) {
    if (!is_pow2(n_roots)) { set_error("n_roots must be a power of two"); return ML_ERR_NOT_POW2; }
    std::vector<uint8_t> cur(roots, roots + 32 * n_roots), nxt;
    while (cur.size() > 32) {  // O(n_roots) host hashing of the subtree roots gathered over NCCL
        nxt.resize(cur.size() / 2);
        for (size_t i = 0; i < nxt.size() / 32; i++) hash_node_host(&cur[64 * i], &cur[64 * i + 32], &nxt[32 * i]);
        cur.swap(nxt);
    }
    memcpy(root_out, cur.data(), 32);
    return ML_OK;
}

}  // extern "C"
