// Context, memory and the array-level C ABI (field vectors, NTT, Reed-Solomon, multilinear transforms, transcript).
#include <cstdlib>
#include <utility>
#include <cstring>
#include <mutex>
#include <map>
#include "field.cuh"
#include "handles.h"
#include "internal.h"

namespace mlb {

static thread_local char g_err[512] = "";
std::atomic<unsigned long long> g_kernel_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

// ---- per-kernel timing registry
bool g_prof_on = false;
struct ProfRec { int id; double bytes; cudaEvent_t e0, e1; bool closed; };
static std::vector<ProfRec> g_prof;
static std::vector<cudaEvent_t> g_event_pool;
static std::mutex g_prof_mu;
static cudaEvent_t prof_event() {
    if (!g_event_pool.empty()) { cudaEvent_t e = g_event_pool.back(); g_event_pool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}
long prof_begin(int id, double alg_bytes, cudaStream_t s) {
    std::lock_guard<std::mutex> lock(g_prof_mu);
    ProfRec r{id, alg_bytes, prof_event(), prof_event(), false};
    cudaEventRecord(r.e0, s);
    g_prof.push_back(r);
    return (long)g_prof.size() - 1;
}
void prof_end(long rec, cudaStream_t s) {
    std::lock_guard<std::mutex> lock(g_prof_mu);
    if (rec < 0 || (size_t)rec >= g_prof.size()) return;
    cudaEventRecord(g_prof[rec].e1, s);
    g_prof[rec].closed = true;
}
static thread_local cudaStream_t tl_stream = nullptr;
static thread_local bool tl_stream_set = false;
cudaStream_t lib_stream(Ctx* ctx) { return tl_stream_set ? tl_stream : ctx->stream; }

static std::mutex g_ctx_mu;
static std::map<int, Ctx*> g_ctx;
static unsigned long long g_release_threshold_init();

int get_ctx(Ctx** out) {
    int dev = 0;
    MLB_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_ctx_mu);
    auto it = g_ctx.find(dev);
    if (it == g_ctx.end()) {
        cudaDeviceProp prop;
        MLB_CUDA(cudaGetDeviceProperties(&prop, dev));
        if (prop.major < 10) {
            set_error("device %d (%s, sm_%d%d) is not a Blackwell GPU; this library ships sm_100a code only", dev, prop.name, prop.major, prop.minor);
            return ML_ERR_CUDA;
        }
        Ctx* c = new Ctx();
        c->device = dev;
        c->sm_count = prop.multiProcessorCount;
        MLB_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        cudaMemPool_t pool;
        MLB_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
        unsigned long long thr = g_release_threshold_init();  // keep freed scratch cached in the pool (ml_set_pool_release_threshold bounds it)
        MLB_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
        // default pool (only used for the legacy stream now, see pool_for): never satisfy an allocation on one stream with a
        // block whose free is still queued on another stream — the driver does that by making the allocating stream wait
        // for the other stream's pending work, which silently serialises concurrent commits
        int off = 0;
        if (!getenv("MLB_POOL_INTERNAL_DEPS")) MLB_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolReuseAllowInternalDependencies, &off));
        it = g_ctx.emplace(dev, c).first;
    }
    *out = it->second;
    return ML_OK;
}
// One memory pool per (device, LIBRARY-OWNED stream).  Concurrent commits run on their own streams and make ~100 stream-ordered
// allocations each, up to 512 MB.  In the shared default pool a block freed on stream A and requested on stream B either makes B
// wait for A's pending work (internal dependencies) or forces the pool to grow with slow virtual-memory calls under a driver-wide
// lock; both showed up as erratic end-to-end times (75 ms to > 1 s per step with 8 commits in flight, tools/e2e_probe.py traces).
// With a private pool per stream every block is recycled on the stream that freed it: no cross-stream waits, no growth after the
// first commit.  Only streams made by ml_stream_create get a private pool (it dies with ml_stream_destroy); streams the caller owns
// (torch streams, the legacy stream) allocate from the device's default pool, so the library never keeps memory keyed to a handle
// whose lifetime it does not control.  Cached blocks are returned to the driver by ml_trim_pools / ml_release_pools, and the amount
// a pool may keep cached is bounded by ml_set_pool_release_threshold (default: keep everything, the point of the pool).
static std::mutex g_pool_mu;
static std::map<std::pair<int, cudaStream_t>, cudaMemPool_t> g_pools;  // library streams only; nullptr = creation failed, use default
static std::atomic<unsigned long long> g_release_threshold{~0ull};
static void register_stream_pool(int dev, cudaStream_t s) {
    static const bool shared = getenv("MLB_SHARED_POOL") != nullptr;
    cudaMemPool_t pool = nullptr;
    if (!shared) {
        cudaMemPoolProps props;
        memset(&props, 0, sizeof props);
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = dev;
        cudaError_t e = cudaMemPoolCreate(&pool, &props);
        if (e != cudaSuccess) {
            cudaGetLastError();
            pool = nullptr;
            fprintf(stderr, "multilinear_b200: cudaMemPoolCreate failed (%s); stream %p allocates from the device default pool\n",
                    cudaGetErrorString(e), (void*)s);
        } else {
            unsigned long long thr = g_release_threshold.load();
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
    }
    std::lock_guard<std::mutex> lock(g_pool_mu);
    g_pools[std::make_pair(dev, s)] = pool;
}
static unsigned long long g_release_threshold_init() { return g_release_threshold.load(); }
static cudaMemPool_t pool_for(cudaStream_t s) {
    if (s == nullptr) return nullptr;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    std::lock_guard<std::mutex> lock(g_pool_mu);
    auto it = g_pools.find(std::make_pair(dev, s));
    return it == g_pools.end() ? nullptr : it->second;  // not a library stream: default pool
}
int dev_alloc_async(void** p, size_t bytes, cudaStream_t s) {
    if (bytes == 0) bytes = 16;
    cudaMemPool_t pool = pool_for(s);
    cudaError_t e = pool ? cudaMallocFromPoolAsync(p, bytes, pool, s) : cudaMallocAsync(p, bytes, s);
    if (e != cudaSuccess) { set_error("device allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e)); return ML_ERR_ALLOC; }
    return ML_OK;
}
int dev_free_async(void* p, cudaStream_t s) {
    if (p) MLB_CUDA(cudaFreeAsync(p, s));
    return ML_OK;
}

// RAII scratch buffer on a stream
struct Scratch {
    void* p = nullptr;
    cudaStream_t s;
    explicit Scratch(cudaStream_t st) : s(st) {}
    int alloc(size_t bytes) { return dev_alloc_async(&p, bytes, s); }
    ~Scratch() { if (p) cudaFreeAsync(p, s); }
    template <class T> T* as() { return (T*)p; }
};

}  // namespace mlb

using namespace mlb;

#define API_BEGIN   \
    Ctx* ctx;       \
    MLB_TRY(get_ctx(&ctx));
#define ST(stream_arg) ((cudaStream_t)(stream_arg))

extern "C" {

const char* ml_last_error(void) { return g_err; }
const char* ml_version(void) { return "multilinear_b200 0.1 (sm_100a)"; }
int ml_device_count(int* count) { MLB_CUDA(cudaGetDeviceCount(count)); return ML_OK; }
int ml_set_device(int device) { MLB_CUDA(cudaSetDevice(device)); return ML_OK; }
int ml_device_name(char* out, size_t cap) {
    int dev;
    MLB_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    MLB_CUDA(cudaGetDeviceProperties(&prop, dev));
    snprintf(out, cap, "%s", prop.name);
    return ML_OK;
}
int ml_synchronize(void) { MLB_CUDA(cudaDeviceSynchronize()); return ML_OK; }
uint64_t ml_kernel_launches(void) { return g_kernel_launches; }

int ml_profile_enable(int on) { g_prof_on = on != 0; return ML_OK; }
int ml_profile_reset(void) {
    std::lock_guard<std::mutex> lock(g_prof_mu);
    for (auto& r : g_prof) { g_event_pool.push_back(r.e0); g_event_pool.push_back(r.e1); }
    g_prof.clear();
    return ML_OK;
}
int ml_profile_get(int id, double* total_ms, uint64_t* launches, double* alg_bytes) {
    MLB_CUDA(cudaDeviceSynchronize());
    std::lock_guard<std::mutex> lock(g_prof_mu);
    double ms = 0, bytes = 0;
    uint64_t n = 0;
    for (auto& r : g_prof) {
        if (r.id != id || !r.closed) continue;
        float t = 0;
        if (cudaEventElapsedTime(&t, r.e0, r.e1) == cudaSuccess) { ms += t; bytes += r.bytes; n++; }
    }
    *total_ms = ms; *launches = n; *alg_bytes = bytes;
    return ML_OK;
}

// the largest launches of a group (records whose algorithmic bytes equal the group's maximum): mean device time
int ml_profile_get_max(int id, double* mean_ms, uint64_t* launches, double* alg_bytes) {
    MLB_CUDA(cudaDeviceSynchronize());
    std::lock_guard<std::mutex> lock(g_prof_mu);
    double mx = -1;
    for (auto& r : g_prof)
        if (r.id == id && r.closed && r.bytes > mx) mx = r.bytes;
    double ms = 0;
    uint64_t n = 0;
    for (auto& r : g_prof) {
        if (r.id != id || !r.closed || r.bytes != mx) continue;
        float t = 0;
        if (cudaEventElapsedTime(&t, r.e0, r.e1) == cudaSuccess) { ms += t; n++; }
    }
    *mean_ms = n ? ms / n : 0; *launches = n; *alg_bytes = mx < 0 ? 0 : mx;
    return ML_OK;
}
int ml_stream_create(void** out) {
    cudaStream_t s;
    MLB_TRY(lib_stream_create(&s, false));  // blocking stream: ordered against the legacy default stream (event timing in bench.py)
    *out = (void*)s;
    return ML_OK;
}
// cached (free) blocks of every pool the library allocates from on the current device go back to the driver, down to
// `keep_bytes` per pool; blocks in use are untouched.  Call between phases when another allocator (e.g. PyTorch's) needs the HBM.
int ml_trim_pools(size_t keep_bytes) {
    int dev = 0;
    MLB_CUDA(cudaGetDevice(&dev));
    cudaMemPool_t def = nullptr;
    MLB_CUDA(cudaDeviceGetDefaultMemPool(&def, dev));
    MLB_CUDA(cudaMemPoolTrimTo(def, keep_bytes));
    std::lock_guard<std::mutex> lock(g_pool_mu);
    for (auto& kv : g_pools)
        if (kv.first.first == dev && kv.second) MLB_CUDA(cudaMemPoolTrimTo(kv.second, keep_bytes));
    return ML_OK;
}
int ml_release_pools(void) {
    MLB_CUDA(cudaDeviceSynchronize());
    return ml_trim_pools(0);
}
// upper bound on what a pool keeps cached after a free reaches a synchronisation point (cudaMemPoolAttrReleaseThreshold);
// applies to existing pools of the current device and to every pool created later.  ~0 (default) keeps everything.
int ml_set_pool_release_threshold(uint64_t bytes) {
    g_release_threshold.store(bytes);
    int dev = 0;
    MLB_CUDA(cudaGetDevice(&dev));
    unsigned long long thr = bytes;
    cudaMemPool_t def = nullptr;
    MLB_CUDA(cudaDeviceGetDefaultMemPool(&def, dev));
    MLB_CUDA(cudaMemPoolSetAttribute(def, cudaMemPoolAttrReleaseThreshold, &thr));
    std::lock_guard<std::mutex> lock(g_pool_mu);
    for (auto& kv : g_pools)
        if (kv.first.first == dev && kv.second) MLB_CUDA(cudaMemPoolSetAttribute(kv.second, cudaMemPoolAttrReleaseThreshold, &thr));
    return ML_OK;
}
int ml_pool_stats(uint64_t* reserved_bytes, uint64_t* used_bytes) {
    int dev = 0;
    MLB_CUDA(cudaGetDevice(&dev));
    unsigned long long res = 0, used = 0, v = 0;
    cudaMemPool_t def = nullptr;
    MLB_CUDA(cudaDeviceGetDefaultMemPool(&def, dev));
    MLB_CUDA(cudaMemPoolGetAttribute(def, cudaMemPoolAttrReservedMemCurrent, &v)); res += v;
    MLB_CUDA(cudaMemPoolGetAttribute(def, cudaMemPoolAttrUsedMemCurrent, &v)); used += v;
    std::lock_guard<std::mutex> lock(g_pool_mu);
    for (auto& kv : g_pools) {
        if (kv.first.first != dev || !kv.second) continue;
        MLB_CUDA(cudaMemPoolGetAttribute(kv.second, cudaMemPoolAttrReservedMemCurrent, &v)); res += v;
        MLB_CUDA(cudaMemPoolGetAttribute(kv.second, cudaMemPoolAttrUsedMemCurrent, &v)); used += v;
    }
    *reserved_bytes = res; *used_bytes = used;
    return ML_OK;
}
int ml_stream_destroy(void* stream) { return lib_stream_destroy((cudaStream_t)stream); }
}  // extern "C"
namespace mlb {
int lib_stream_create(cudaStream_t* out, bool non_blocking) {
    Ctx* ctx;
    MLB_TRY(get_ctx(&ctx));  // sets the default pool's attributes before the first allocation on this device
    cudaStream_t s;
    if (non_blocking) MLB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    else MLB_CUDA(cudaStreamCreate(&s));
    register_stream_pool(ctx->device, s);
    *out = s;
    return ML_OK;
}
int lib_stream_destroy(cudaStream_t s) {
    MLB_CUDA(cudaStreamSynchronize(s));
    {   // drop the stream's private pool (the driver defers the release until its last allocation is freed)
        int dev = 0;
        cudaGetDevice(&dev);
        std::lock_guard<std::mutex> lock(g_pool_mu);
        auto it = g_pools.find(std::make_pair(dev, s));
        if (it != g_pools.end()) {
            if (it->second) cudaMemPoolDestroy(it->second);
            g_pools.erase(it);
        }
    }
    MLB_CUDA(cudaStreamDestroy(s));
    return ML_OK;
}
}  // namespace mlb
extern "C" {
int ml_stream_synchronize(void* stream) { MLB_CUDA(cudaStreamSynchronize((cudaStream_t)stream)); return ML_OK; }
int ml_set_thread_stream(void* stream, int enable) {
    tl_stream = (cudaStream_t)stream;
    tl_stream_set = enable != 0;
    return ML_OK;
}

int ml_dev_alloc(size_t bytes, void** out) { MLB_CUDA(cudaMalloc(out, bytes ? bytes : 16)); return ML_OK; }
int ml_dev_free(void* p) { MLB_CUDA(cudaFree(p)); return ML_OK; }
int ml_dev_upload(void* dst, const void* src, size_t bytes) { MLB_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice)); return ML_OK; }
int ml_dev_download(void* dst, const void* src, size_t bytes) { MLB_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost)); return ML_OK; }
int ml_host_alloc_pinned(size_t bytes, void** out) { MLB_CUDA(cudaMallocHost(out, bytes ? bytes : 16)); return ML_OK; }
int ml_host_free_pinned(void* p) { MLB_CUDA(cudaFreeHost(p)); return ML_OK; }
// page-lock memory the caller allocated itself (a Vec<Field128>, a numpy array): uploads from it then run at pinned-memory speed.
// The caller must unregister before freeing the memory.
int ml_host_register(void* p, size_t bytes) { MLB_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterDefault)); return ML_OK; }
int ml_host_unregister(void* p) { MLB_CUDA(cudaHostUnregister(p)); return ML_OK; }

// ------------------------------------------------------------------ helpers for host-pointer entry points
static int upload(Scratch& sc, const void* host, size_t bytes, cudaStream_t s) {
    MLB_TRY(sc.alloc(bytes));
    if (bytes) MLB_CUDA(cudaMemcpyAsync(sc.p, host, bytes, cudaMemcpyHostToDevice, s));
    return ML_OK;
}
static int download(void* host, const void* dev, size_t bytes, cudaStream_t s) {
    if (bytes) MLB_CUDA(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, s));
    MLB_CUDA(cudaStreamSynchronize(s));
    return ML_OK;
}

// ------------------------------------------------------------------ field vectors
static int vec2(int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) {
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    Scratch da(s), db(s), dout(s);
    MLB_TRY(upload(da, a, n * 16, s));
    if (b) MLB_TRY(upload(db, b, n * 16, s));
    MLB_TRY(dout.alloc(n * 16));
    MLB_TRY(fe_vec_launch(op, da.as<fe>(), db.as<fe>(), n, dout.as<fe>(), s));
    return download(out, dout.p, n * 16, s);
}
int ml_fe_add_vec(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) { return vec2(0, a, b, n, out); }
int ml_fe_sub_vec(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) { return vec2(1, a, b, n, out); }
int ml_fe_mul_vec(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) { return vec2(2, a, b, n, out); }
int ml_fe_inv_vec(const uint8_t* a, size_t n, uint8_t* out) { return vec2(3, a, nullptr, n, out); }
int ml_fe_pow_vec(const uint8_t* a, const uint8_t exp_le[16], size_t n, uint8_t* out) {
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    Scratch da(s), dout(s);
    MLB_TRY(upload(da, a, n * 16, s));
    MLB_TRY(dout.alloc(n * 16));
    MLB_TRY(fe_pow_vec_launch(da.as<fe>(), hfe_load(exp_le), n, dout.as<fe>(), s));
    return download(out, dout.p, n * 16, s);
}
int ml_fe_from_i64_vec(const int64_t* v, size_t n, uint8_t* out) {
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    Scratch dv(s), dout(s);
    MLB_TRY(upload(dv, v, n * 8, s));
    MLB_TRY(dout.alloc(n * 16));
    MLB_TRY(fe_from_i64_launch(dv.as<int64_t>(), n, dout.as<fe>(), s));
    return download(out, dout.p, n * 16, s);
}
int ml_fe_from_wide_vec(const uint8_t* v, size_t n, int variant, uint8_t* out) {
    API_BEGIN
    if (variant != 1 && variant != 2) { set_error("reduction variant must be 1 or 2"); return ML_ERR_ARG; }
    cudaStream_t s = lib_stream(ctx);
    Scratch dv(s), dout(s);
    MLB_TRY(upload(dv, v, n * 32, s));
    MLB_TRY(dout.alloc(n * 16));
    MLB_TRY(fe_from_wide_launch(dv.p, n, variant, dout.as<fe>(), s));
    return download(out, dout.p, n * 16, s);
}
int ml_synthetic_elements_dev(uint64_t seed, size_t n, void* out_dev, void* stream) {
    API_BEGIN
    (void)ctx;
    return synthetic_launch(seed, n, (fe*)out_dev, ST(stream));
}

// ------------------------------------------------------------------ NTT
int ml_pow2_generator(uint64_t log_size, uint8_t out[16]) {
    hfe g;
    if (!hfe_pow2_generator(log_size, &g)) { set_error("pow_2_generator(%llu): None", (unsigned long long)log_size); return ML_ERR_OUT_OF_RANGE; }
    hfe_store(out, g);
    return ML_OK;
}
int ml_pow2_generator_powers_dev(uint64_t log_size, void* out_dev, void* stream) {
    API_BEGIN
    if (log_size > 40) { set_error("pow_2_generator_powers(%llu): None", (unsigned long long)log_size); return ML_ERR_OUT_OF_RANGE; }
    return powers_launch(ctx, (int)log_size, (fe*)out_dev, ST(stream));
}
int ml_pow2_generator_powers(uint64_t log_size, uint8_t* out) {
    API_BEGIN
    if (log_size > 40) { set_error("pow_2_generator_powers(%llu): None", (unsigned long long)log_size); return ML_ERR_OUT_OF_RANGE; }
    cudaStream_t s = lib_stream(ctx);
    Scratch d(s);
    const size_t bytes = ((size_t)16) << log_size;
    MLB_TRY(d.alloc(bytes));
    MLB_TRY(powers_launch(ctx, (int)log_size, d.as<fe>(), s));
    return download(out, d.p, bytes, s);
}
int ml_bit_reverse_permutation(uint8_t* values, size_t n, size_t elem_bytes) {
    API_BEGIN
    if (n == 0) return ML_OK;
    if (elem_bytes != 16) { set_error("bit_reverse_permutation: only 16-byte (Field128) elements are supported"); return ML_ERR_ARG; }
    cudaStream_t s = lib_stream(ctx);
    Scratch din(s), dout(s);
    MLB_TRY(upload(din, values, n * 16, s));
    MLB_TRY(dout.alloc(n * 16));
    MLB_TRY(bit_reverse_launch(din.p, dout.p, n, 16, s));
    return download(values, dout.p, n * 16, s);
}

// gen must be the primitive n-th root the reference's callers pass (pow_2_generator(log2 n)) or its inverse
static int classify_gen(size_t n, const uint8_t gen[16], bool* use_inverse_tables) {
    const unsigned log_n = ilog2(n);
    hfe g = hfe_load(gen), w;
    if (log_n > 40 || !hfe_pow2_generator(log_n, &w)) { set_error("no root of unity of order 2^%u", log_n); return ML_ERR_OUT_OF_RANGE; }
    if (g == w) { *use_inverse_tables = false; return ML_OK; }
    if (n > 1 && g == hfe_inv(w)) { *use_inverse_tables = true; return ML_OK; }
    set_error("ntt: gen is not pow_2_generator(%u) or its inverse", log_n);
    return ML_ERR_GENERATOR;
}
static int ntt_dev_impl(Ctx* ctx, const void* in, size_t n, const uint8_t gen[16], void* out, bool is_intt, bool rs, cudaStream_t s) {
    const size_t N = rs ? n << ML_LOG_BLOWUP : n;
    if (!is_pow2(N)) { set_error("The number of coeffs must be a power of 2"); return ML_ERR_NOT_POW2; }
    bool inv_tables;
    MLB_TRY(classify_gen(N, gen, &inv_tables));
    // intt(gen) runs the network with 1/gen and scales by 1/n; with gen = w^-1 that is the forward tables plus scaling
    if (!is_intt) {
        if (!inv_tables) return ntt_launch(ctx, (const fe*)in, (fe*)out, (int)ilog2(N), false, rs, s);
        // forward network with the inverse root = unscaled inverse transform: run inverse tables then multiply by N
        MLB_TRY(ntt_launch(ctx, (const fe*)in, (fe*)out, (int)ilog2(N), true, rs, s));
        // scale back by N: out[i] *= N  (rare path: callers normally pass the forward generator)
        hfe Nf = hfe_new((hfe)N);
        Scratch tmp(s);
        MLB_TRY(tmp.alloc(16));
        uint8_t nb[16];
        hfe_store(nb, Nf);
        MLB_CUDA(cudaMemcpyAsync(tmp.p, nb, 16, cudaMemcpyHostToDevice, s));
        return fe_vec_launch(4, (const fe*)out, tmp.as<fe>(), N, (fe*)out, s);
    }
    if (!inv_tables) return ntt_launch(ctx, (const fe*)in, (fe*)out, (int)ilog2(N), true, false, s);
    // intt with gen = w^-1: network runs with w, then 1/n scaling
    MLB_TRY(ntt_launch(ctx, (const fe*)in, (fe*)out, (int)ilog2(N), false, false, s));
    hfe ninv = hfe_inv(hfe_new((hfe)N));
    Scratch tmp(s);
    MLB_TRY(tmp.alloc(16));
    uint8_t nb[16];
    hfe_store(nb, ninv);
    MLB_CUDA(cudaMemcpyAsync(tmp.p, nb, 16, cudaMemcpyHostToDevice, s));
    return fe_vec_launch(4, (const fe*)out, tmp.as<fe>(), N, (fe*)out, s);
}
int ml_ntt_dev(const void* c, size_t n, const uint8_t gen[16], void* e, void* stream) {
    API_BEGIN
    return ntt_dev_impl(ctx, c, n, gen, e, false, false, ST(stream));
}
int ml_intt_dev(const void* e, size_t n, const uint8_t gen[16], void* c, void* stream) {
    API_BEGIN
    return ntt_dev_impl(ctx, e, n, gen, c, true, false, ST(stream));
}
int ml_reed_solomon_dev(const void* c, size_t n, const uint8_t gen[16], void* code, void* stream) {
    API_BEGIN
    return ntt_dev_impl(ctx, c, n, gen, code, false, true, ST(stream));
}
static int ntt_host(const uint8_t* in, size_t n, const uint8_t gen[16], uint8_t* out, bool is_intt, bool rs) {
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    const size_t N = rs ? n << ML_LOG_BLOWUP : n;
    if (!is_pow2(N)) { set_error("The number of coeffs must be a power of 2"); return ML_ERR_NOT_POW2; }
    Scratch din(s), dout(s);
    MLB_TRY(upload(din, in, n * 16, s));
    MLB_TRY(dout.alloc(N * 16));
    MLB_TRY(ntt_dev_impl(ctx, din.p, n, gen, dout.p, is_intt, rs, s));
    return download(out, dout.p, N * 16, s);
}
int ml_ntt(const uint8_t* c, size_t n, const uint8_t gen[16], uint8_t* e) { return ntt_host(c, n, gen, e, false, false); }
int ml_intt(const uint8_t* e, size_t n, const uint8_t gen[16], uint8_t* c) { return ntt_host(e, n, gen, c, true, false); }
int ml_reed_solomon(const uint8_t* c, size_t n, const uint8_t gen[16], uint8_t* code) { return ntt_host(c, n, gen, code, false, true); }
int ml_poly_evaluate(const uint8_t* coeffs, size_t n, const uint8_t x[16], uint8_t out[16]) {
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    Scratch d(s);
    MLB_TRY(upload(d, coeffs, n * 16, s));
    hfe r;
    MLB_TRY(poly_eval_launch(ctx, d.as<fe>(), n, hfe_load(x), &r, s));
    hfe_store(out, r);
    return ML_OK;
}

// ------------------------------------------------------------------ multilinear polynomials
int ml_mle_to_coefficient_dev(const void* e, size_t len, void* c, void* stream) {
    API_BEGIN
    (void)ctx;
    return mobius_launch((const fe*)e, (fe*)c, len, true, ST(stream));
}
int ml_mle_to_evaluation_dev(const void* c, size_t len, void* e, void* stream) {
    API_BEGIN
    (void)ctx;
    return mobius_launch((const fe*)c, (fe*)e, len, false, ST(stream));
}
static int mobius_host(const uint8_t* in, size_t len, uint8_t* out, bool sub) {
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    Scratch d(s);
    MLB_TRY(upload(d, in, len * 16, s));
    MLB_TRY(mobius_launch(d.as<fe>(), d.as<fe>(), len, sub, s));
    return download(out, d.p, len * 16, s);
}
int ml_mle_to_coefficient(const uint8_t* e, size_t len, uint8_t* c) { return mobius_host(e, len, c, true); }
int ml_mle_to_evaluation(const uint8_t* c, size_t len, uint8_t* e) { return mobius_host(c, len, e, false); }
static int load_args(const uint8_t* args, size_t n, std::vector<hfe>& v) {
    v.resize(n);
    for (size_t i = 0; i < n; i++) v[i] = hfe_load(args + 16 * i);
    return ML_OK;
}
int ml_mle_evals_evaluate_dev(const void* evals, size_t len, const uint8_t* args, size_t n_args, uint8_t out[16], void* stream) {
    API_BEGIN
    std::vector<hfe> a;
    load_args(args, n_args, a);
    hfe r;
    MLB_TRY(mle_evals_evaluate_launch(ctx, (const fe*)evals, len, a.data(), n_args, &r, ST(stream)));
    hfe_store(out, r);
    return ML_OK;
}
int ml_mle_evals_evaluate(const uint8_t* evals, size_t len, const uint8_t* args, size_t n_args, uint8_t out[16]) {
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    Scratch d(s);
    MLB_TRY(upload(d, evals, len * 16, s));
    return ml_mle_evals_evaluate_dev(d.p, len, args, n_args, out, s);
}
int ml_mle_coeffs_evaluate(const uint8_t* coeffs, size_t len, const uint8_t* args, size_t n_args, uint8_t out[16]) {
    API_BEGIN
    cudaStream_t s = lib_stream(ctx);
    Scratch d(s);
    MLB_TRY(upload(d, coeffs, len * 16, s));
    std::vector<hfe> a;
    load_args(args, n_args, a);
    hfe r;
    MLB_TRY(mle_coeffs_evaluate_launch(ctx, d.as<fe>(), len, a.data(), n_args, &r, s));
    hfe_store(out, r);
    return ML_OK;
}

// ------------------------------------------------------------------ transcript (host; src/transcript.rs)
int ml_transcript_new(ml_transcript** out) { *out = new ml_transcript(); return ML_OK; }
int ml_transcript_clone(const ml_transcript* t, ml_transcript** out) { *out = new ml_transcript(*t); return ML_OK; }
void ml_transcript_free(ml_transcript* t) { delete t; }
int ml_transcript_absorb(ml_transcript* t, const uint8_t* bytes, size_t len) { t->sha.update(bytes, len); return ML_OK; }
int ml_transcript_random(const ml_transcript* t, uint8_t out[32]) { t->sha.digest(out); return ML_OK; }
int ml_transcript_next_challenge(ml_transcript* t, uint8_t out[16]) {
    uint8_t d[32];
    t->sha.digest(d);
    hfe_store(out, hfe_new(hfe_load(d)));
    return ML_OK;
}
size_t ml_transcript_state_bytes(void) { return sizeof(HostSha256); }
int ml_transcript_export(const ml_transcript* t, uint8_t* state_out) {
    if (!t || !state_out) { set_error("ml_transcript_export: null pointer"); return ML_ERR_ARG; }
    memcpy(state_out, &t->sha, sizeof(HostSha256));
    return ML_OK;
}
int ml_transcript_import(const uint8_t* state, ml_transcript** out) {
    if (!state || !out) { set_error("ml_transcript_import: null pointer"); return ML_ERR_ARG; }
    ml_transcript* t = new ml_transcript();
    memcpy(&t->sha, state, sizeof(HostSha256));
    *out = t;
    return ML_OK;
}

}  // extern "C"
