// Peer plumbing shared by the sharded handles: arenas, flags, push / wait kernels, IPC records, the handle core (peer.h).
#include <cstdlib>
#include <string>

#include "peer.h"
#include "prover_internal.h"

namespace mlb {

// thread g sets flag[phase][rank] = epoch in rank g's arena (only: a single target, or -1 for all ranks)
__global__ void peer_signal_kernel(PeerPtrs peers, size_t off_flags, int world, int phase, int rank, unsigned long long epoch, int only) {
    const int g = threadIdx.x;
    if (g >= world || (only >= 0 && g != only)) return;
    __threadfence_system();  // everything this rank's earlier kernels stored (stream order) is visible before the flag
    flag_store_release(reinterpret_cast<unsigned long long*>(peers.base[g] + off_flags) + phase * PEER_MAXR + rank, epoch);
}
__global__ void peer_wait_kernel(const unsigned long long* flags, int world, int only_from, unsigned long long epoch,
                                 unsigned long long timeout_ns, int* status) {
    wait_flags(flags, world, only_from, epoch, timeout_ns, status);
}
__global__ void peer_push_kernel(const uint8_t* __restrict__ src, int nbytes, PeerPtrs peers, size_t dst_off, size_t off_flags, int world,
                                 int phase, int rank, unsigned long long epoch, int only) {
    const int g = threadIdx.x;
    if (g >= world || (only >= 0 && g != only)) return;
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* d4 = reinterpret_cast<uint4*>(peers.base[g] + dst_off);
    for (int i = 0; i < nbytes / 16; i++) d4[i] = s4[i];
    __threadfence_system();
    flag_store_release(reinterpret_cast<unsigned long long*>(peers.base[g] + off_flags) + phase * PEER_MAXR + rank, epoch);
}

unsigned peer_grid(size_t n, size_t cap) {
    size_t b = (n + 255) / 256;
    if (b > cap) b = cap;
    if (b == 0) b = 1;
    return (unsigned)b;
}

int peer_check_world(const char* who, int world, int n_local) {
    if (world < 1 || world > PEER_MAXR || (world & (world - 1)) || n_local < 1 || n_local > world) { set_error("%s: world must be a power of two <= %d", who, PEER_MAXR); return ML_ERR_ARG; }
    if (n_local != 1 && n_local != world) { set_error("%s: a process hosts either one rank or all of them", who); return ML_ERR_ARG; }
    return ML_OK;
}

int peer_rank_init(PeerGroup& g, PeerRank& r, const char* who, size_t zero_bytes) {
    if (r.rank < 0 || r.rank >= g.world) { set_error("%s: rank out of range", who); return ML_ERR_ARG; }
    if (cudaSetDevice(r.device) != cudaSuccess) { cudaGetLastError(); set_error("%s: no CUDA device %d", who, r.device); return ML_ERR_CUDA; }
    MLB_TRY(get_ctx(&r.ctx));
    auto it = g.streams.find(r.device);
    if (it == g.streams.end()) {
        DevStreams ds;
        if (lib_stream_create(&ds.main, true) != ML_OK || lib_stream_create(&ds.enc2, true) != ML_OK || lib_stream_create(&ds.side, true) != ML_OK) return ML_ERR_CUDA;
        it = g.streams.emplace(r.device, ds).first;
    }
    r.st = it->second;
    if (cudaMalloc((void**)&r.arena, g.arena_bytes) != cudaSuccess || cudaMemset(r.arena, 0, zero_bytes) != cudaSuccess) {
        cudaGetLastError();
        set_error("%s: allocation of %zu bytes on device %d failed", who, g.arena_bytes, r.device);
        return ML_ERR_ALLOC;
    }
    return ML_OK;
}

int peer_link_local(PeerGroup& g, const std::vector<PeerRank*>& ranks, const char* who) {
    int st = ML_OK;
    for (PeerRank* r : ranks) g.base[r->rank] = r->arena;
    for (PeerRank* a : ranks)
        for (PeerRank* b : ranks) {
            if (a->device == b->device) continue;
            cudaSetDevice(a->device);
            cudaError_t e = cudaDeviceEnablePeerAccess(b->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { set_error("no peer access from device %d to %d: %s", a->device, b->device, cudaGetErrorString(e)); st = ML_ERR_PEER; }
            cudaGetLastError();
        }
    for (int r = 0; r < g.world; r++)
        if (!g.base[r]) { set_error("%s: rank %d is missing from local_ranks", who, r); st = ML_ERR_ARG; }
    g.connected = st == ML_OK;
    return st;
}

int peer_export(const std::vector<PeerRank*>& ranks, uint8_t* records_out) {
    DeviceGuard guard;
    for (size_t i = 0; i < ranks.size(); i++) {
        const PeerRank& r = *ranks[i];
        MLB_CUDA(cudaSetDevice(r.device));
        int32_t hdr[2] = {r.rank, 0};
        cudaIpcMemHandle_t h;
        MLB_CUDA(cudaIpcGetMemHandle(&h, r.arena));
        memcpy(records_out + PEER_RECORD_BYTES * i, hdr, 8);
        memcpy(records_out + PEER_RECORD_BYTES * i + 8, &h, 64);
    }
    return ML_OK;
}

int peer_connect(PeerGroup& g, PeerRank& me, const uint8_t* records, size_t n_records, const char* who) {
    DeviceGuard guard;
    MLB_CUDA(cudaSetDevice(me.device));
    for (size_t i = 0; i < n_records; i++) {
        int32_t hdr[2];
        memcpy(hdr, records + PEER_RECORD_BYTES * i, 8);
        const int r = hdr[0];
        if (r < 0 || r >= g.world) { set_error("%s: record with rank %d", who, r); return ML_ERR_ARG; }
        if (r == me.rank) { g.base[r] = me.arena; continue; }
        if (g.base[r]) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, records + PEER_RECORD_BYTES * i + 8, 64);
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) { cudaGetLastError(); set_error("%s: cannot map the arena of rank %d: %s", who, r, cudaGetErrorString(e)); return ML_ERR_PEER; }
        g.base[r] = (uint8_t*)p;
        g.mapped[r] = true;
    }
    for (int r = 0; r < g.world; r++)
        if (!g.base[r]) { set_error("%s: no record for rank %d", who, r); return ML_ERR_ARG; }
    g.connected = true;
    return ML_OK;
}

void peer_rank_free(PeerRank& r) {
    if (r.arena) cudaFree(r.arena);
    r.arena = nullptr;
}

void peer_group_release(PeerGroup& g, int device) {
    cudaSetDevice(device);
    for (int r = 0; r < PEER_MAXR; r++)
        if (g.mapped[r]) cudaIpcCloseMemHandle(g.base[r]);
    for (auto& kv : g.streams) {
        cudaSetDevice(kv.first);
        lib_stream_destroy(kv.second.main);
        lib_stream_destroy(kv.second.enc2);
        lib_stream_destroy(kv.second.side);
    }
    g.streams.clear();
}

int peer_check_ready(const PeerGroup& g, const char* who) {
    if (!g.connected) { set_error("%s: arenas of the other ranks are not connected (%s_connect)", who, who); return ML_ERR_ARG; }
    return ML_OK;
}

int peer_signal(const PeerGroup& g, const PeerRank& r, int phase, int only, cudaStream_t s) {
    peer_signal_kernel<<<1, 32, 0, s>>>(g.peers(), g.off_flags, g.world, phase, r.rank, g.epoch, only);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
int peer_wait(const PeerGroup& g, const PeerRank& r, int phase, int only_from, cudaStream_t s) { return peer_wait_for(g, r, phase, only_from, g.epoch, s); }
int peer_wait_for(const PeerGroup& g, const PeerRank& r, int phase, int only_from, unsigned long long epoch, cudaStream_t s) {
    peer_wait_kernel<<<1, 32, 0, s>>>(g.flags(r, phase), g.world, only_from, epoch, g.timeout_ns, g.status(r));
    MLB_KERNEL_CHECK();
    return ML_OK;
}
int peer_push(const PeerGroup& g, const PeerRank& r, const void* src_dev, int nbytes, size_t dst_off, int phase, int only, cudaStream_t s) {
    peer_push_kernel<<<1, 32, 0, s>>>((const uint8_t*)src_dev, nbytes, g.peers(), dst_off, g.off_flags, g.world, phase, r.rank, g.epoch, only);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
int peer_read_status(const PeerGroup& g, const PeerRank& r, const char* who) {
    int st = 0;
    MLB_CUDA(cudaSetDevice(r.device));
    MLB_TRY(mlbp::d2h_sync(&st, g.status(r), sizeof st, r.st.main));
    if (st == 0) return ML_OK;
    if (st != ML_ERR_PEER) { set_error("%s: rank %d: rank 0 ended the call with status %d", who, r.rank, st); return st; }  // relayed (tail_fail)
    set_error("%s: rank %d timed out waiting for a peer rank (%.0f s)", who, r.rank, g.timeout_ns * 1e-9);
    return ML_ERR_PEER;
}


PeerHandle::~PeerHandle() {
    DeviceGuard guard;
    for (int i = 0; i < N_MARKS; i++)
        if (mark[i]) cudaEventDestroy(mark[i]);
    for (auto& r : local) {
        cudaSetDevice(r.device);
        cudaDeviceSynchronize();
        peer_rank_free(r);
    }
    peer_group_release(grp, local.empty() ? guard.prev : local[0].device);
}

int PeerHandle::init(int world_, int n_local, const int* local_ranks, const int* local_devices, size_t arena_bytes, size_t off_flags,
                     size_t off_status, size_t zero_bytes) {
    const std::string create = std::string(who) + "_create";
    world = world_;
    grp.world = world;
    grp.arena_bytes = arena_bytes;
    grp.off_flags = off_flags;
    grp.off_status = off_status;
    if (const char* e = getenv("MLB_SHARD_TIMEOUT_S")) grp.timeout_ns = (unsigned long long)(atof(e) * 1e9);
    int st = ML_OK;
    for (int i = 0; i < n_local && st == ML_OK; i++) {
        PeerRank r;
        r.rank = local_ranks[i];
        r.device = local_devices[i];
        st = peer_rank_init(grp, r, create.c_str(), zero_bytes);
        if (st == ML_OK || st == ML_ERR_ALLOC) local.push_back(r);
    }
    if (st == ML_OK && n_local == world) {
        std::vector<PeerRank*> ranks;
        for (auto& r : local) ranks.push_back(&r);
        st = peer_link_local(grp, ranks, create.c_str());
    }
    return st;
}

int PeerHandle::export_records(uint8_t* records_out) {
    std::vector<PeerRank*> ranks;
    for (auto& r : local) ranks.push_back(&r);
    return peer_export(ranks, records_out);
}
int PeerHandle::connect(const uint8_t* records, size_t n_records) {
    const std::string entry = std::string(who) + "_connect";
    if (local.size() != 1) { set_error("%s: only for handles that host one rank", entry.c_str()); return ML_ERR_ARG; }
    return peer_connect(grp, local[0], records, n_records, entry.c_str());
}
void* PeerHandle::stream(int local_index) const {
    if (local_index < 0 || (size_t)local_index >= local.size()) return nullptr;
    return (void*)local[local_index].st.main;
}
int PeerHandle::phase_ms(double* out, int cap) const {
    int n = 0;
    for (int i = 0; i + 1 < n_marks && n < cap; i++) {
        float ms = 0;
        if (!mark[i] || !mark[i + 1] || cudaEventElapsedTime(&ms, mark[i], mark[i + 1]) != cudaSuccess) { cudaGetLastError(); ms = -1.f; }
        out[n++] = ms;
    }
    return n;
}
void PeerHandle::mark_phase(int idx) {
    if (idx >= N_MARKS || local.empty()) return;
    PeerRank& r = local[0];
    cudaSetDevice(r.device);
    if (!mark[idx] && cudaEventCreate(&mark[idx]) != cudaSuccess) { cudaGetLastError(); return; }
    cudaEventRecord(mark[idx], r.st.main);
    if (idx + 1 > n_marks) n_marks = idx + 1;
}
PeerRank* PeerHandle::rank0() {
    for (auto& r : local)
        if (r.rank == 0) return &r;
    return nullptr;
}

int PeerHandle::host_call(const char* entry, size_t n_blocks, size_t bytes, const std::function<const uint8_t*(int rank, size_t j)>& src,
                          const std::function<int(const void* const* dev)>& run) {
    if ((int)local.size() != world) { set_error("%s: host-pointer entry needs a handle that hosts every rank", entry); return ML_ERR_ARG; }
    DeviceGuard guard;
    std::vector<void*> dev(local.size() * n_blocks, nullptr);
    int st = ML_OK;
    for (size_t i = 0; i < local.size() && st == ML_OK; i++) {
        PeerRank& r = local[i];
        if (cudaSetDevice(r.device) != cudaSuccess) { st = ML_ERR_CUDA; break; }
        for (size_t j = 0; j < n_blocks && st == ML_OK; j++) {
            void*& d = dev[i * n_blocks + j];
            st = mlbp::pmalloc(&d, bytes, r.st.main);
            if (st == ML_OK) st = mlbp::h2d(d, src(r.rank, j), bytes, r.st.main);
        }
        if (st == ML_OK && cudaStreamSynchronize(r.st.main) != cudaSuccess) st = ML_ERR_CUDA;
    }
    if (st == ML_OK) st = run(dev.data());
    for (size_t i = 0; i < local.size(); i++) {
        cudaSetDevice(local[i].device);
        cudaStreamSynchronize(local[i].st.main);
        for (size_t j = 0; j < n_blocks; j++) mlbp::pfree(dev[i * n_blocks + j], local[i].st.main);
    }
    return st;
}

}  // namespace mlb
