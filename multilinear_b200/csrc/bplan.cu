// Stream-ordered batched provers (include/multilinear_b200.h, "stream-ordered batched provers"): BatchedFriProof::prove
// (batched_fri.rs:286-318) of B codes, given as codes or as coefficients (reed_solomon of each first), and BatchedPCSProof::prove
// (batched_pcs.rs:130-180), enqueued on a caller's stream with no host work in between.
//
// A plan owns every device buffer one prove of B codes of 2^D elements needs, allocated once at creation.  An enqueue call only
// launches kernels and device-to-device copies:
//   [encode each polynomial into the plan's codes]  ->  batch tree over the B codes  ->  batch_root_kernel (claim, batch root,
//   rho, running claim)  ->  [PCS: fingerprinted table, eq table]  ->  fold chain (fold_chain_enqueue; its batched first fold
//   reads rho from HBM)  ->  fri_query_indices_kernel  ->  bfri_proof_write_kernel  ->  [sumcheck copy]  ->  status copy.
// The blocking provers read the batch root back to draw rho on the host, synchronise before the chain and once after it, and
// open the queries on the host (bfri_assemble); here all of that stays on the device.
#include <algorithm>

#include "plan.h"
#include "transcript.cuh"

using namespace mlb;
using namespace mlbp;

namespace {

const int MAX_LAYERS = PLAN_MAX_LAYERS;
const size_t MAX_CODES = (size_t)1 << 20;
const int PTR_CHUNK = 2048;  // pointers per table-writing launch: 16 KiB of kernel parameters

// The bincode wire format of a BatchedFriProof (batched_fri.rs:21-27; write_bfri_proof in prover.cu) at log_domain D, B codes:
//   32 B batch commitment | FriProof header at D - 1 (u64 nc | nc = D - 2 commitments | u64 128) | 128 batched queries |
//   Field128 last_element (u64 16 + 16 B) | 32 B last_random
// batched query = u64 B | B x (u64 16 | value 16 B | u64 16 | minus_value 16 B) | u64 (D - 1) | (D - 1) x (32 B sibling | u32
// direction) in the batch tree | a FriProof query at D - 1 (layers N/2 .. 4, index idx mod N/4)
__host__ __device__ inline size_t bquery_bytes(int D, size_t B) { return 16 + 48 * B + 36 * (size_t)(D - 1) + query_bytes(D - 1); }
size_t bproof_bytes(int D, size_t B) { return 32 + header_bytes(D - 1) + (size_t)ML_NUM_QUERIES * bquery_bytes(D, B) + 56; }

__global__ void __launch_bounds__(32) batch_root_kernel(const DevTranscript* tr_in, DevTranscript* tr_out, const uint8_t* __restrict__ root,
                                                        const fe* __restrict__ inputs, int n_inputs, const fe* __restrict__ outputs,
                                                        int n_outputs, int absorb_claim, fe* rho_out, fe* prev_out, fe* r_out) {
    if (threadIdx.x != 0) return;
    DevTranscript t = *tr_in;
    if (absorb_claim) {  // batched_pcs.rs:44-49
        dt_absorb(&t, reinterpret_cast<const uint8_t*>(inputs), 16 * n_inputs);
        dt_absorb(&t, reinterpret_cast<const uint8_t*>(outputs), 16 * n_outputs);
    }
    fe rho;
    const fe acc = dt_batch_root(&t, root, outputs, n_outputs, &rho);
    fe_store(rho_out, rho);
    if (prev_out) fe_store(prev_out, acc);
    if (r_out) {
        const fe r = dt_challenge(&t);
        fe_store(r_out, r);
        fe_store(r_out + 1, fe_half(r));
    }
    *tr_out = t;
}

// a caller's host array of device pointers into a device table, through kernel parameters (a graph-capturable enqueue cannot copy
// from host memory)
struct PtrChunk {
    const void* p[PTR_CHUNK];
};
__global__ void __launch_bounds__(256) ptr_table_kernel(PtrChunk c, int n, const void** dst) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = c.p[i];
}
int ptr_table_write(const void* const* src, size_t n, const void** dst, cudaStream_t s) {
    for (size_t o = 0; o < n; o += PTR_CHUNK) {
        const int k = (int)std::min((size_t)PTR_CHUNK, n - o);
        PtrChunk c;
        memcpy(c.p, src + o, (size_t)k * sizeof(void*));
        ptr_table_kernel<<<1, 256, 0, s>>>(c, k, dst + o);
        MLB_KERNEL_CHECK();
    }
    return ML_OK;
}

struct BWriteArgs {
    const fe* code[MAX_LAYERS];          // FRI layer j: N/2 >> j elements
    const uint8_t* digests[MAX_LAYERS];  // its tree (merkle_layer_offset)
    const fe* const* codes;              // the B codes, N elements each
    const uint8_t* batch_digests;        // the batch tree, N/2 leaves
    const unsigned long long* indices;   // 128 query indices in [0, N/2)
    const uint8_t* roots;                // D - 2 commitments
    const fe* last;
    const uint8_t* last_random;
    uint8_t* out;
    int log_domain;
    int n_codes;
};
// CTA q < 128 writes batched query q (open_query_at, batched_fri.rs:207-225): the B value pairs at idx and idx + N/2, the path in
// the batch tree, then the FriProof query of layers N/2 .. 4 (write_fri_query).  CTA 128 writes the rest.
__global__ void __launch_bounds__(256) bfri_proof_write_kernel(BWriteArgs a) {
    const int D = a.log_domain, nc = D - 2, B = a.n_codes, tid = threadIdx.x;
    const size_t half = (size_t)1 << (D - 1), header = 32 + header_bytes(D - 1), qbytes = bquery_bytes(D, (size_t)B);
    if (blockIdx.x == ML_NUM_QUERIES) {
        const uint8_t* root = a.batch_digests + 32 * (2 * half - 2);
        if (tid < 8) put32(a.out + 4 * tid, word(root, tid));
        if (tid == 0) { put64(a.out + 32, (unsigned long long)nc); put64(a.out + 40 + 32 * (size_t)nc, ML_NUM_QUERIES); }
        for (int w = tid; w < 8 * nc; w += blockDim.x) put32(a.out + 40 + 4 * (size_t)w, word(a.roots, w));
        uint8_t* tail = a.out + header + (size_t)ML_NUM_QUERIES * qbytes;
        if (tid == 0) put64(tail, 16);
        if (tid < 4) put32(tail + 8 + 4 * tid, word(a.last, tid));
        if (tid >= 32 && tid < 40) put32(tail + 24 + 4 * (tid - 32), word(a.last_random, tid - 32));
        return;
    }
    uint8_t* qo = a.out + header + (size_t)blockIdx.x * qbytes;
    const unsigned long long idx = a.indices[blockIdx.x];
    if (tid == 0) put64(qo, (unsigned long long)B);
    for (int c = tid; c < B; c += blockDim.x) { put64(qo + 8 + 48 * (size_t)c, 16); put64(qo + 32 + 48 * (size_t)c, 16); }
    for (int e = tid; e < 8 * B; e += blockDim.x) {
        const int c = e >> 3, w = e & 7;
        const fe* src = a.codes[c] + idx + (w >= 4 ? half : 0);
        put32(qo + 48 * (size_t)c + (w < 4 ? 16 + 4 * w : 24 + 4 * w), word(src, w & 3));
    }
    uint8_t* bp = qo + 8 + 48 * (size_t)B;
    if (tid == 0) put64(bp, (unsigned long long)(D - 1));
    write_path_tail(bp + 8, a.batch_digests, half, idx, D - 1, tid, blockDim.x);
    write_fri_query(bp + 8 + 36 * (size_t)(D - 1), a.code, a.digests, D - 1, idx);
}

size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace

int mlbp::batch_root_launch(const DevTranscript* tr_in, DevTranscript* tr_out, const uint8_t* root, const fe* inputs, int n_inputs, const fe* outputs,
                            int n_outputs, bool absorb_claim, fe* rho_out, fe* prev_out, fe* r_out, cudaStream_t s) {
    ProfScope prof(PROF_TRANSCRIPT, 0.0, s);
    batch_root_kernel<<<1, 32, 0, s>>>(tr_in, tr_out, root, inputs, n_inputs, outputs, n_outputs, absorb_claim ? 1 : 0, rho_out, prev_out, r_out);
    MLB_KERNEL_CHECK();
    return ML_OK;
}

struct ml_batched_prove_plan {
    int device = -1;
    int log_domain = 0;
    int kind = ML_BPLAN_CODES;
    size_t n_codes = 0;
    void* mem = nullptr;  // one cudaMalloc holding everything below
    size_t bytes = 0;
    uint8_t* batch_digests = nullptr;          // the batch tree (N/2 leaves); before it is built, the encodes' scratch
    fe* code[MAX_LAYERS] = {nullptr};          // FRI layer j: N/2 >> j elements
    uint8_t* digests[MAX_LAYERS] = {nullptr};  // its tree
    fe* codes = nullptr;                       // RS / PCS: the B codes, N elements each
    const fe** codes_table = nullptr;          // RS / PCS: pointers to them, written at creation
    const void** in_table = nullptr;           // CODES: the caller's codes; PCS: the caller's evaluations
    fe* matrix = nullptr;                      // PCS: the sumcheck tables (N/2 each) and the eq-weight scratch
    fe* delta = nullptr;
    fe* weights = nullptr;
    uint8_t* chain = nullptr;                  // the fold chain's scratch block
    DevTranscript* tr = nullptr;               // the transcript after the batch root
    fe* rho = nullptr;
    fe* prev = nullptr;                        // PCS: the running claim fingerprint(rho, outputs)
    unsigned long long* indices = nullptr;     // 128 query indices
    uint8_t* last_random = nullptr;            // 32 B
};

namespace {

int check_bplan(const ml_batched_prove_plan* p, int kind, const char* who, Ctx** ctx) {
    if (!p) { set_error("%s: plan is NULL", who); return ML_ERR_ARG; }
    int dev = -1;
    MLB_CUDA(cudaGetDevice(&dev));
    if (dev != p->device) { set_error("batched prove plan made on device %d used with device %d current", p->device, dev); return ML_ERR_ARG; }
    if (kind != p->kind) { set_error("%s: the plan was made for kind %d", who, p->kind); return ML_ERR_ARG; }
    return get_ctx(ctx);
}

// the checks of one call: `ptrs` (n_codes device buffers of elems elements each) plus the fixed buffers in `fixed`
int check_call(const ml_batched_prove_plan* p, const void* const* ptrs, const char* ptrs_name, size_t elems, std::vector<PlanBuf>& bufs) {
    if (!ptrs) { set_error("prove plan: %s is NULL", ptrs_name); return ML_ERR_ARG; }
    for (size_t j = 0; j < p->n_codes; j++) {
        PlanBuf b{ptrs[j], 16 * elems, false, ptrs_name};
        b.index = (long)j;
        bufs.push_back(b);
    }
    return plan_check_bufs(bufs.data(), bufs.size());
}

// the B codes are in place (or their encodes enqueued), `table` points to them: batch tree, root kernel, PCS tables, fold chain,
// query phase, proof blob, copies
int benqueue(Ctx* ctx, ml_batched_prove_plan* p, const fe* const* table, const fe* inputs_dev, const fe* outputs_dev, void* transcript_dev,
             void* proof_dev, void* sumcheck_dev, int* status_dev, cudaStream_t s) {
    const int D = p->log_domain;
    const size_t N = (size_t)1 << D, B = p->n_codes, n_vars = (size_t)D - 1;
    const bool pcs = p->kind == ML_BPLAN_PCS;
    MLB_TRY(merkle_batched_rs_launch(table, B, N, p->batch_digests, s));  // batched_fri.rs:77
    MLB_TRY(batch_root_launch((const DevTranscript*)transcript_dev, p->tr, p->batch_digests + 32 * (N - 2), inputs_dev, (int)n_vars, outputs_dev,
                              pcs ? (int)B : 0, pcs, p->rho, pcs ? p->prev : nullptr, nullptr, s));
    ml_sumcheck sc;
    if (pcs) {  // batched_pcs.rs:55-67: the fingerprinted evaluation table and the eq table
        MLB_TRY(fingerprint_rows_launch((const fe* const*)p->in_table, B, N / 2, 0, p->matrix, s, p->rho));
        MLB_TRY(eq_table_launch(ctx, nullptr, n_vars, p->delta, s, inputs_dev, p->weights));
        sc.matrix = p->matrix;
        sc.delta = p->delta;
        sc.height = N / 2;
    }
    ml_fri* f = new ml_fri();
    f->log_n0 = D;
    f->stream = s;
    ChainHooks hooks;
    hooks.tr_dev = p->tr;
    hooks.prev_dev = pcs ? p->prev : nullptr;
    hooks.layer_code = p->code;
    hooks.layer_digests = p->digests;
    hooks.first_fold = [&](const fe* r_dev, fe** next, bool* owns) {  // batched_fri.rs:193-195, rho from HBM
        *owns = false;
        *next = p->code[0];
        return fri_batched_fold_launch(ctx, table, B, N, p->code[0], 0, 0, r_dev, D, s, p->rho);
    };
    ChainRun run;
    int st = fold_chain_enqueue(ctx, f, &hooks, pcs ? &sc : nullptr, 0, 0, false, nullptr, p->chain, &run, s);
    const size_t nc = f->layers.size();
    if (st == ML_OK && nc != (size_t)D - 2) { set_error("batched prove plan: %zu layers for a domain of 2^%d", nc, D); st = ML_ERR_SIZE; }
    free_fri(f);  // host bookkeeping only: the layers' buffers belong to the plan
    MLB_TRY(st);
    // BatchedFriProof::prove's query phase (batched_fri.rs:296-308): indices in [0, N/2), as FriProof's at 2^D
    MLB_TRY(fri_query_indices_launch((const DevTranscript*)(p->chain + CHAIN_OFF_TR), (DevTranscript*)transcript_dev, D - 1, p->indices,
                                     p->last_random, s));
    BWriteArgs a;
    memset(&a, 0, sizeof a);
    for (int j = 0; j < D - 2; j++) { a.code[j] = p->code[j]; a.digests[j] = p->digests[j]; }
    a.codes = table;
    a.batch_digests = p->batch_digests;
    a.indices = p->indices;
    a.roots = p->chain + CHAIN_OFF_ROOTS;
    a.last = (const fe*)(p->chain + CHAIN_OFF_LAST);
    a.last_random = p->last_random;
    a.out = (uint8_t*)proof_dev;
    a.log_domain = D;
    a.n_codes = (int)B;
    {
        ProfScope prof(PROF_GATHER, (double)bproof_bytes(D, B), s);
        bfri_proof_write_kernel<<<ML_NUM_QUERIES + 1, 256, 0, s>>>(a);
        MLB_KERNEL_CHECK();
    }
    if (pcs) MLB_CUDA(cudaMemcpyAsync(sumcheck_dev, p->chain + CHAIN_OFF_SC, 2 * n_vars * 16, cudaMemcpyDeviceToDevice, s));
    MLB_CUDA(cudaMemcpyAsync(status_dev, p->chain + CHAIN_OFF_STATUS, sizeof(int), cudaMemcpyDeviceToDevice, s));
    return ML_OK;
}

}  // namespace

extern "C" {

int ml_batched_prove_plan_create(size_t log_domain, size_t n_codes, int kind, ml_batched_prove_plan** out) {
    if (!out) { set_error("ml_batched_prove_plan_create: out is NULL"); return ML_ERR_ARG; }
    *out = nullptr;
    if (log_domain < 3 || log_domain > 40) { set_error("batched prove plan: log_domain %zu outside 3..40", log_domain); return ML_ERR_SIZE; }
    if (n_codes < 1 || n_codes > MAX_CODES) { set_error("batched prove plan: n_codes %zu outside 1..2^20", n_codes); return ML_ERR_SIZE; }
    if (kind != ML_BPLAN_CODES && kind != ML_BPLAN_RS && kind != ML_BPLAN_PCS) { set_error("batched prove plan: unknown kind %d", kind); return ML_ERR_ARG; }
    Ctx* ctx;
    MLB_TRY(get_ctx(&ctx));
    const int D = (int)log_domain;
    const size_t N = (size_t)1 << D, B = n_codes;
    const bool encodes = kind != ML_BPLAN_CODES, pcs = kind == ML_BPLAN_PCS;
    if (encodes && B > (SIZE_MAX / 32) / N) { set_error("batched prove plan: %zu codes of 2^%d do not fit", B, D); return ML_ERR_ALLOC; }
    // carve every buffer out of one allocation: batch tree, layers N/2 .. 4 with their trees, codes, tables, chain scratch, query phase
    size_t off = 0, code_off[MAX_LAYERS], dig_off[MAX_LAYERS];
    const size_t batch_off = off; off = align_up(off + 32 * N);  // >= the RS NTT's 16 N and encode_into's 24 N bytes of scratch
    for (int j = 0; j < D - 2; j++) {
        code_off[j] = off; off = align_up(off + 16 * ((N / 2) >> j));
        dig_off[j] = off; off = align_up(off + 32 * ((N / 2) >> j));
    }
    size_t codes_off = 0, ctab_off = 0, in_off = 0, m_off = 0, d_off = 0, w_off = 0;
    if (encodes) {
        codes_off = off; off = align_up(off + 16 * N * B);
        ctab_off = off; off = align_up(off + sizeof(void*) * B);
    }
    if (!encodes || pcs) { in_off = off; off = align_up(off + sizeof(void*) * B); }
    if (pcs) {
        m_off = off; off = align_up(off + 16 * (N / 2));
        d_off = off; off = align_up(off + 16 * (N / 2));
        w_off = off; off = align_up(off + 16 * eq_weights_elems((size_t)D - 1));
    }
    const size_t chain_off = off; off = align_up(off + chain_scratch_bytes());
    const size_t tr_off = off; off = align_up(off + sizeof(DevTranscript));
    const size_t rho_off = off; off = align_up(off + 16);
    const size_t prev_off = off; off = align_up(off + 16);
    const size_t idx_off = off; off = align_up(off + 8 * ML_NUM_QUERIES);
    const size_t lr_off = off; off = align_up(off + 32);
    ml_batched_prove_plan* p = new ml_batched_prove_plan();
    p->log_domain = D;
    p->kind = kind;
    p->n_codes = B;
    p->bytes = off;
    MLB_CUDA(cudaGetDevice(&p->device));
    if (cudaMalloc(&p->mem, off) != cudaSuccess) {
        cudaGetLastError();
        delete p;
        set_error("batched prove plan for %zu x 2^%d: device allocation of %zu bytes failed", B, D, off);
        return ML_ERR_ALLOC;
    }
    uint8_t* base = (uint8_t*)p->mem;
    p->batch_digests = base + batch_off;
    for (int j = 0; j < D - 2; j++) { p->code[j] = (fe*)(base + code_off[j]); p->digests[j] = base + dig_off[j]; }
    if (encodes) { p->codes = (fe*)(base + codes_off); p->codes_table = (const fe**)(base + ctab_off); }
    if (!encodes || pcs) p->in_table = (const void**)(base + in_off);
    if (pcs) { p->matrix = (fe*)(base + m_off); p->delta = (fe*)(base + d_off); p->weights = (fe*)(base + w_off); }
    p->chain = base + chain_off;
    p->tr = (DevTranscript*)(base + tr_off);
    p->rho = (fe*)(base + rho_off);
    p->prev = (fe*)(base + prev_off);
    p->indices = (unsigned long long*)(base + idx_off);
    p->last_random = base + lr_off;
    int st = ML_OK;
    if (encodes) {  // the table of the plan's own codes never changes: written once, now
        std::vector<const fe*> t(B);
        for (size_t j = 0; j < B; j++) t[j] = p->codes + j * N;
        if (cudaMemcpy(p->codes_table, t.data(), sizeof(void*) * B, cudaMemcpyHostToDevice) != cudaSuccess) {
            set_error("batched prove plan: writing the code table failed");
            st = ML_ERR_CUDA;
        }
    }
    // the tables every enqueue reads (the encodes' NTT and the folds use those of 2^D), built and waited for now
    if (st == ML_OK) st = ntt_prepare(ctx, D, lib_stream(ctx));
    if (st == ML_OK && cudaStreamSynchronize(lib_stream(ctx)) != cudaSuccess) { set_error("batched prove plan: table build failed"); st = ML_ERR_CUDA; }
    if (st != ML_OK) { cudaFree(p->mem); delete p; return st; }
    *out = p;
    return ML_OK;
}

void ml_batched_prove_plan_free(ml_batched_prove_plan* p) {
    if (!p) return;
    int dev = -1;
    cudaGetDevice(&dev);
    if (dev != p->device) cudaSetDevice(p->device);
    cudaFree(p->mem);
    if (dev != p->device && dev >= 0) cudaSetDevice(dev);
    delete p;
}

size_t ml_batched_prove_plan_device_bytes(const ml_batched_prove_plan* p) { return p ? p->bytes : 0; }
size_t ml_batched_prove_plan_proof_bytes(const ml_batched_prove_plan* p) { return p ? bproof_bytes(p->log_domain, p->n_codes) : 0; }

int ml_batched_fri_prove_async(ml_batched_prove_plan* p, const void* const* codes_dev, void* transcript_dev, void* proof_dev, int* status_dev,
                               void* stream) {
    Ctx* ctx;
    MLB_TRY(check_bplan(p, ML_BPLAN_CODES, "ml_batched_fri_prove_async", &ctx));
    const int D = p->log_domain;
    const size_t N = (size_t)1 << D;
    std::vector<PlanBuf> b = {{transcript_dev, sizeof(DevTranscript), true, "transcript_dev"},
                              {proof_dev, bproof_bytes(D, p->n_codes), true, "proof_dev"},
                              {status_dev, sizeof(int), true, "status_dev"}};
    MLB_TRY(check_call(p, codes_dev, "codes_dev", N, b));
    cudaStream_t s = (cudaStream_t)stream;
    // the caller's codes are read in place through the plan's input table
    MLB_TRY(ptr_table_write(codes_dev, p->n_codes, p->in_table, s));
    return benqueue(ctx, p, (const fe* const*)p->in_table, nullptr, nullptr, transcript_dev, proof_dev, nullptr, status_dev, s);
}

int ml_batched_rs_fri_prove_async(ml_batched_prove_plan* p, const void* const* coeffs_dev, void* transcript_dev, void* proof_dev, int* status_dev,
                                  void* stream) {
    Ctx* ctx;
    MLB_TRY(check_bplan(p, ML_BPLAN_RS, "ml_batched_rs_fri_prove_async", &ctx));
    const int D = p->log_domain;
    const size_t N = (size_t)1 << D;
    std::vector<PlanBuf> b = {{transcript_dev, sizeof(DevTranscript), true, "transcript_dev"},
                              {proof_dev, bproof_bytes(D, p->n_codes), true, "proof_dev"},
                              {status_dev, sizeof(int), true, "status_dev"}};
    MLB_TRY(check_call(p, coeffs_dev, "coeffs_dev", N / 2, b));
    cudaStream_t s = (cudaStream_t)stream;
    // reed_solomon (fri/mod.rs:19-28) of each into the plan's codes; the multi-pass NTT's temporary is the batch tree's buffer,
    // which the tree overwrites only after the last encode
    for (size_t j = 0; j < p->n_codes; j++)
        MLB_TRY(ntt_launch(ctx, (const fe*)coeffs_dev[j], p->codes + j * N, D, false, true, s, false, (fe*)p->batch_digests));
    return benqueue(ctx, p, p->codes_table, nullptr, nullptr, transcript_dev, proof_dev, nullptr, status_dev, s);
}

int ml_batched_pcs_prove_async(ml_batched_prove_plan* p, const void* inputs_dev, const void* outputs_dev, const void* const* evals_dev,
                               void* transcript_dev, void* proof_dev, void* sumcheck_dev, int* status_dev, void* stream) {
    Ctx* ctx;
    MLB_TRY(check_bplan(p, ML_BPLAN_PCS, "ml_batched_pcs_prove_async", &ctx));
    const int D = p->log_domain;
    const size_t N = (size_t)1 << D, n_vars = (size_t)D - 1;
    std::vector<PlanBuf> b = {{inputs_dev, 16 * n_vars, false, "inputs_dev"},
                              {outputs_dev, 16 * p->n_codes, false, "outputs_dev"},
                              {transcript_dev, sizeof(DevTranscript), true, "transcript_dev"},
                              {proof_dev, bproof_bytes(D, p->n_codes), true, "proof_dev"},
                              {sumcheck_dev, 2 * 16 * n_vars, true, "sumcheck_dev"},
                              {status_dev, sizeof(int), true, "status_dev"}};
    MLB_TRY(check_call(p, evals_dev, "evals_dev", N / 2, b));
    cudaStream_t s = (cudaStream_t)stream;
    // encode (batched_pcs.rs:144-149) of each into the plan's codes, the scratch in the batch tree's buffer as above
    for (size_t j = 0; j < p->n_codes; j++)
        MLB_TRY(encode_into(ctx, (const fe*)evals_dev[j], N / 2, p->codes + j * N, s, (fe*)p->batch_digests));
    MLB_TRY(ptr_table_write(evals_dev, p->n_codes, p->in_table, s));
    return benqueue(ctx, p, p->codes_table, (const fe*)inputs_dev, (const fe*)outputs_dev, transcript_dev, proof_dev, sumcheck_dev, status_dev, s);
}

}  // extern "C"
