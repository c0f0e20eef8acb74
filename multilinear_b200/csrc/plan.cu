// Stream-ordered provers (include/multilinear_b200.h, "stream-ordered provers"): FriProof::prove (src/fri/mod.rs:261-285), with or
// without reed_solomon first, and PCSProof::prove (src/fri/multilinear_pcs.rs:90-136) enqueued on a caller's stream with no host
// work in between.
//
// A plan owns every device buffer one prove of its domain size needs, allocated once at creation, and creation builds the root
// and pass tables the kernels read.  An enqueue call then only launches kernels and device-to-device copies:
//   encode (RS NTT, or Moebius + NTT)  ->  layer-0 tree  ->  fold chain (fold_chain_enqueue, the same chain the blocking
//   provers run, with its layers in the plan)  ->  fri_query_indices_kernel  ->  fri_proof_write_kernel  ->  status copy.
// The blocking provers read the chain's state back and open the queries on the host (assemble_fri_proof); here the query indices
// are derived on the device and the proof writer gathers the openings straight into the bincode blob.
#include "plan.h"

using namespace mlb;
using namespace mlbp;

namespace {

const int MAX_LAYERS = PLAN_MAX_LAYERS;

// the FriProof wire format: plan.h
size_t proof_bytes(int D) { return header_bytes(D) + (size_t)ML_NUM_QUERIES * query_bytes(D) + 56; }

struct WriteArgs {
    const fe* code[MAX_LAYERS];          // layer j: N >> j elements
    const uint8_t* digests[MAX_LAYERS];  // layer j: every Merkle layer of its tree (merkle_layer_offset)
    const unsigned long long* indices;   // 128 query indices in [0, N/2)
    const uint8_t* roots;                // nc x 32 B
    const fe* last;
    const uint8_t* last_random;
    uint8_t* out;
    int log_domain;
};
// CTA q < 128 writes query q (write_fri_query, plan.h), CTA 128 writes the rest.
__global__ void __launch_bounds__(256) fri_proof_write_kernel(WriteArgs a) {
    const int D = a.log_domain, nc = D - 1;
    const size_t qbytes = query_bytes(D), header = header_bytes(D);
    const int tid = threadIdx.x;
    if (blockIdx.x == ML_NUM_QUERIES) {
        if (tid == 0) { put64(a.out, (unsigned long long)nc); put64(a.out + 8 + 32 * (size_t)nc, ML_NUM_QUERIES); }
        for (int w = tid; w < 8 * nc; w += blockDim.x) put32(a.out + 8 + 4 * (size_t)w, word(a.roots, w));
        uint8_t* tail = a.out + header + (size_t)ML_NUM_QUERIES * qbytes;
        if (tid == 0) put64(tail, 16);
        if (tid < 4) put32(tail + 8 + 4 * tid, word(a.last, tid));
        if (tid >= 32 && tid < 40) put32(tail + 24 + 4 * (tid - 32), word(a.last_random, tid - 32));
        return;
    }
    write_fri_query(a.out + header + (size_t)blockIdx.x * qbytes, a.code, a.digests, D, a.indices[blockIdx.x]);
}

size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace

int mlbp::plan_check_bufs(const PlanBuf* b, size_t n) {
    char name[64];
    auto label = [&](const PlanBuf& x) -> const char* {
        if (x.index < 0) return x.name;
        snprintf(name, sizeof name, "%s[%ld]", x.name, x.index);
        return name;
    };
    for (size_t i = 0; i < n; i++) {
        if (!b[i].p) { set_error("prove plan: %s is NULL", label(b[i])); return ML_ERR_ARG; }
        if ((uintptr_t)b[i].p & 15) { set_error("prove plan: %s is not 16-byte aligned", label(b[i])); return ML_ERR_ARG; }
    }
    // outputs are few: compare each with every other buffer (inputs may overlap each other)
    for (size_t i = 0; i < n; i++) {
        if (!b[i].out) continue;
        const uintptr_t a0 = (uintptr_t)b[i].p, a1 = a0 + b[i].bytes;
        for (size_t j = 0; j < n; j++) {
            if (j == i || (b[j].out && j < i)) continue;
            const uintptr_t c0 = (uintptr_t)b[j].p, c1 = c0 + b[j].bytes;
            if (a0 < c1 && c0 < a1) {
                char other[64];
                snprintf(other, sizeof other, "%s", label(b[j]));
                set_error("prove plan: %s overlaps %s", b[i].name, other);
                return ML_ERR_ARG;
            }
        }
    }
    return ML_OK;
}

struct ml_prove_plan {
    int device = -1;
    int log_domain = 0;
    bool pcs = false;
    void* mem = nullptr;  // one cudaMalloc holding everything below
    size_t bytes = 0;
    fe* code[MAX_LAYERS] = {nullptr};           // layer j: N >> j elements (layer 0: the encoded code)
    uint8_t* digests[MAX_LAYERS] = {nullptr};   // layer j: (N >> j) digests; layer 0's also serves as the encode's scratch
    uint8_t* chain = nullptr;                   // the fold chain's scratch block
    unsigned long long* indices = nullptr;      // 128 query indices
    uint8_t* last_random = nullptr;             // 32 B
    fe* matrix = nullptr;                       // PCS: the sumcheck tables (N/2 each) and the eq-weight scratch
    fe* delta = nullptr;
    fe* weights = nullptr;
};

namespace {

int check_plan(const ml_prove_plan* p, Ctx** ctx) {
    if (!p) { set_error("prove plan: plan is NULL"); return ML_ERR_ARG; }
    int dev = -1;
    MLB_CUDA(cudaGetDevice(&dev));
    if (dev != p->device) { set_error("prove plan made on device %d used with device %d current", p->device, dev); return ML_ERR_ARG; }
    return get_ctx(ctx);
}

// layer 0 is in place (or its encode enqueued): tree, fold chain, query phase, proof blob, status
int enqueue_prove(Ctx* ctx, ml_prove_plan* p, const fe* layer0, ml_sumcheck* sc, const fe* output_dev, void* transcript_dev, void* proof_dev,
                  void* sumcheck_dev, int* status_dev, cudaStream_t s) {
    const int D = p->log_domain;
    const size_t N = (size_t)1 << D;
    ml_fri* f = new ml_fri();
    f->log_n0 = D;
    f->stream = s;
    int st = fri_push_layer(f, (fe*)layer0, N, false, s, true, p->digests[0]);
    ChainHooks hooks;
    hooks.tr_dev = (const DevTranscript*)transcript_dev;
    hooks.prev_dev = output_dev;
    hooks.layer_code = p->code;
    hooks.layer_digests = p->digests;
    ChainRun run;
    if (st == ML_OK) st = fold_chain_enqueue(ctx, f, &hooks, sc, 0, 0, true, nullptr, p->chain, &run, s);
    const size_t nc = f->layers.size();
    if (st == ML_OK && nc != (size_t)D - 1) { set_error("prove plan: %zu layers for a domain of 2^%d", nc, D); st = ML_ERR_SIZE; }
    free_fri(f);  // host bookkeeping only: the layers' buffers belong to the plan (or the caller)
    MLB_TRY(st);
    MLB_TRY(fri_query_indices_launch((const DevTranscript*)(p->chain + CHAIN_OFF_TR), (DevTranscript*)transcript_dev, D - 1, p->indices,
                                     p->last_random, s));
    WriteArgs a;
    memset(&a, 0, sizeof a);
    for (int j = 0; j < D - 1; j++) { a.code[j] = j == 0 ? layer0 : p->code[j]; a.digests[j] = p->digests[j]; }
    a.indices = p->indices;
    a.roots = p->chain + CHAIN_OFF_ROOTS;
    a.last = (const fe*)(p->chain + CHAIN_OFF_LAST);
    a.last_random = p->last_random;
    a.out = (uint8_t*)proof_dev;
    a.log_domain = D;
    {
        ProfScope prof(PROF_GATHER, (double)proof_bytes(D), s);
        fri_proof_write_kernel<<<ML_NUM_QUERIES + 1, 256, 0, s>>>(a);
        MLB_KERNEL_CHECK();
    }
    if (sc) MLB_CUDA(cudaMemcpyAsync(sumcheck_dev, p->chain + CHAIN_OFF_SC, 2 * (size_t)(D - 1) * 16, cudaMemcpyDeviceToDevice, s));
    MLB_CUDA(cudaMemcpyAsync(status_dev, p->chain + CHAIN_OFF_STATUS, sizeof(int), cudaMemcpyDeviceToDevice, s));
    return ML_OK;
}

}  // namespace

extern "C" {

int ml_prove_plan_create(size_t log_domain, int pcs, ml_prove_plan** out) {
    if (!out) { set_error("ml_prove_plan_create: out is NULL"); return ML_ERR_ARG; }
    *out = nullptr;
    if (log_domain < 2 || log_domain > 40) { set_error("prove plan: log_domain %zu outside 2..40", log_domain); return ML_ERR_SIZE; }
    Ctx* ctx;
    MLB_TRY(get_ctx(&ctx));
    const int D = (int)log_domain;
    const size_t N = (size_t)1 << D;
    // carve every buffer out of one allocation: layers N .. 4 with their trees, chain scratch, query phase, PCS tables
    size_t off = 0, code_off[MAX_LAYERS], dig_off[MAX_LAYERS];
    for (int j = 0; j < D - 1; j++) {
        code_off[j] = off; off = align_up(off + 16 * (N >> j));
        dig_off[j] = off; off = align_up(off + 32 * (N >> j));
    }
    const size_t chain_off = off; off = align_up(off + chain_scratch_bytes());
    const size_t idx_off = off; off = align_up(off + 8 * ML_NUM_QUERIES);
    const size_t lr_off = off; off = align_up(off + 32);
    size_t m_off = 0, d_off = 0, w_off = 0;
    if (pcs) {
        m_off = off; off = align_up(off + 16 * (N / 2));
        d_off = off; off = align_up(off + 16 * (N / 2));
        w_off = off; off = align_up(off + 16 * eq_weights_elems((size_t)D - 1));
    }
    ml_prove_plan* p = new ml_prove_plan();
    p->log_domain = D;
    p->pcs = pcs != 0;
    p->bytes = off;
    MLB_CUDA(cudaGetDevice(&p->device));
    if (cudaMalloc(&p->mem, off) != cudaSuccess) {
        cudaGetLastError();
        delete p;
        set_error("prove plan for 2^%d: device allocation of %zu bytes failed", D, off);
        return ML_ERR_ALLOC;
    }
    uint8_t* base = (uint8_t*)p->mem;
    for (int j = 0; j < D - 1; j++) { p->code[j] = (fe*)(base + code_off[j]); p->digests[j] = base + dig_off[j]; }
    p->chain = base + chain_off;
    p->indices = (unsigned long long*)(base + idx_off);
    p->last_random = base + lr_off;
    if (pcs) { p->matrix = (fe*)(base + m_off); p->delta = (fe*)(base + d_off); p->weights = (fe*)(base + w_off); }
    // the tables every enqueue reads (the RS encode's NTT and the folds use those of 2^D), built and waited for now
    int st = ntt_prepare(ctx, D, lib_stream(ctx));
    if (st != ML_OK) { cudaFree(p->mem); delete p; return st; }
    *out = p;
    return ML_OK;
}

void ml_prove_plan_free(ml_prove_plan* p) {
    if (!p) return;
    int dev = -1;
    cudaGetDevice(&dev);
    if (dev != p->device) cudaSetDevice(p->device);
    cudaFree(p->mem);
    if (dev != p->device && dev >= 0) cudaSetDevice(dev);
    delete p;
}

size_t ml_prove_plan_device_bytes(const ml_prove_plan* p) { return p ? p->bytes : 0; }
size_t ml_prove_plan_proof_bytes(const ml_prove_plan* p) { return p ? proof_bytes(p->log_domain) : 0; }

int ml_rs_fri_prove_async(ml_prove_plan* p, const void* coeffs_dev, void* transcript_dev, void* proof_dev, int* status_dev, void* stream) {
    Ctx* ctx;
    MLB_TRY(check_plan(p, &ctx));
    const size_t N = (size_t)1 << p->log_domain;
    const PlanBuf b[] = {{coeffs_dev, 16 * (N / 2), false, "coeffs_dev"}, {transcript_dev, sizeof(DevTranscript), true, "transcript_dev"},
                     {proof_dev, proof_bytes(p->log_domain), true, "proof_dev"}, {status_dev, sizeof(int), true, "status_dev"}};
    MLB_TRY(plan_check_bufs(b, 4));
    cudaStream_t s = (cudaStream_t)stream;
    // reed_solomon (fri/mod.rs:19-28) into layer 0; the multi-pass NTT's temporary is layer 0's digest buffer, which the tree
    // of layer 0 overwrites only after the NTT
    MLB_TRY(ntt_launch(ctx, (const fe*)coeffs_dev, p->code[0], p->log_domain, false, true, s, false, (fe*)p->digests[0]));
    return enqueue_prove(ctx, p, p->code[0], nullptr, nullptr, transcript_dev, proof_dev, nullptr, status_dev, s);
}

int ml_fri_prove_async(ml_prove_plan* p, const void* code_dev, void* transcript_dev, void* proof_dev, int* status_dev, void* stream) {
    Ctx* ctx;
    MLB_TRY(check_plan(p, &ctx));
    const size_t N = (size_t)1 << p->log_domain;
    const PlanBuf b[] = {{code_dev, 16 * N, false, "code_dev"}, {transcript_dev, sizeof(DevTranscript), true, "transcript_dev"},
                     {proof_dev, proof_bytes(p->log_domain), true, "proof_dev"}, {status_dev, sizeof(int), true, "status_dev"}};
    MLB_TRY(plan_check_bufs(b, 4));
    // the caller's code is layer 0 itself: the kernels only read it
    return enqueue_prove(ctx, p, (const fe*)code_dev, nullptr, nullptr, transcript_dev, proof_dev, nullptr, status_dev, (cudaStream_t)stream);
}

int ml_pcs_prove_async(ml_prove_plan* p, const void* inputs_dev, const void* output_dev, const void* evals_dev, void* transcript_dev, void* proof_dev,
                       void* sumcheck_dev, int* status_dev, void* stream) {
    Ctx* ctx;
    MLB_TRY(check_plan(p, &ctx));
    if (!p->pcs) { set_error("ml_pcs_prove_async: the plan was made with pcs = 0"); return ML_ERR_ARG; }
    const int D = p->log_domain;
    const size_t N = (size_t)1 << D, n_vars = (size_t)D - 1;
    const PlanBuf b[] = {{inputs_dev, 16 * n_vars, false, "inputs_dev"}, {output_dev, 16, false, "output_dev"}, {evals_dev, 16 * (N / 2), false, "evals_dev"},
                     {transcript_dev, sizeof(DevTranscript), true, "transcript_dev"}, {proof_dev, proof_bytes(D), true, "proof_dev"},
                     {sumcheck_dev, 2 * 16 * n_vars, true, "sumcheck_dev"}, {status_dev, sizeof(int), true, "status_dev"}};
    MLB_TRY(plan_check_bufs(b, 7));
    cudaStream_t s = (cudaStream_t)stream;
    // encode (multilinear_pcs.rs:101-107) into layer 0, its scratch in layer 0's digest buffer as above
    MLB_TRY(encode_into(ctx, (const fe*)evals_dev, N / 2, p->code[0], s, (fe*)p->digests[0]));
    // SumcheckTables::build_tables_for_pcs (sumcheck.rs:128-145) from the points in HBM
    MLB_CUDA(cudaMemcpyAsync(p->matrix, evals_dev, 16 * (N / 2), cudaMemcpyDeviceToDevice, s));
    MLB_TRY(eq_table_launch(ctx, nullptr, n_vars, p->delta, s, (const fe*)inputs_dev, p->weights));
    ml_sumcheck sc;
    sc.matrix = p->matrix;
    sc.delta = p->delta;
    sc.height = N / 2;
    return enqueue_prove(ctx, p, p->code[0], &sc, (const fe*)output_dev, transcript_dev, proof_dev, sumcheck_dev, status_dev, s);
}

}  // extern "C"
