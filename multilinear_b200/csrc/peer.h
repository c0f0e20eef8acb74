// Peer plumbing shared by every sharded handle (ml_shard_*, ml_pcs_shard_*, ml_bpcs_shard_*, ml_fri_shard_*, ml_bfri_shard_*,
// ml_wsumcheck_shard_*): arenas, flags, push / wait kernels, IPC records, and the handle core PeerHandle.
//
// Every rank owns one peer-visible ARENA in HBM (cudaMalloc; mapped into the other ranks through CUDA IPC, or plain peer access
// when one process hosts all ranks).  The arena starts with a mailbox of flags: flag[phase][rank].  All data-path exchange is a
// kernel STORING into a peer's arena, followed by a flag store (release, system scope) into the consumers' arenas; consumers
// wait on their own flags with a tiny spin kernel (acquire, system scope, bounded by a timeout that raises ML_ERR_PEER in the
// arena's status word).  A flag holds the epoch of the call that raised it, so flags never need resetting.
//
// A handle hosts the ranks of ONE process: one rank (one process per GPU, arenas connected through records the caller
// all-gathers) or all of them (devices may repeat: virtual ranks on one GPU).  Ranks that share a device share its streams,
// and the host enqueues phase by phase over the local ranks, so on a shared device every wait is already satisfied when it is
// enqueued.
#pragma once
#include <functional>
#include <map>
#include <vector>

#include "internal.h"

namespace mlb {

static const int PEER_MAXR = ML_MAX_PEERS;
static const size_t PEER_RECORD_BYTES = 72;  // int32 rank | int32 reserved | 64-byte CUDA IPC handle of the arena

struct PeerPtrs {
    uint8_t* base[PEER_MAXR];
};

__device__ __forceinline__ void flag_store_release(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long flag_load_acquire(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// thread g waits until flags[g] >= epoch in the LOCAL arena (only_from: a single source, or -1 for all)
__device__ __forceinline__ void wait_flags(const unsigned long long* flags, int world, int only_from, unsigned long long epoch,
                                           unsigned long long timeout_ns, int* status) {
    const int g = threadIdx.x;
    if (g < world && (only_from < 0 || g == only_from)) {
        const unsigned long long t0 = global_ns();
        while (flag_load_acquire(flags + g) < epoch) {
            if (global_ns() - t0 > timeout_ns) { atomicExch(status, ML_ERR_PEER); break; }
            __nanosleep(200);
        }
    }
}

struct DevStreams {
    cudaStream_t main = nullptr, enc2 = nullptr, side = nullptr;
};
struct PeerRank {
    int rank = 0, device = 0;
    Ctx* ctx = nullptr;
    DevStreams st;
    uint8_t* arena = nullptr;
};

// the ranks' arenas as seen from this process, and the protocol state of one handle
struct PeerGroup {
    int world = 1;
    size_t arena_bytes = 0, off_flags = 0, off_status = 0;  // the arena layout's total and its mailbox words
    std::map<int, DevStreams> streams;                       // per device
    uint8_t* base[PEER_MAXR];
    bool mapped[PEER_MAXR];                                  // opened through IPC (must be closed)
    bool connected = false;
    unsigned long long epoch = 0;
    unsigned long long timeout_ns = 20ull * 1000 * 1000 * 1000;  // MLB_SHARD_TIMEOUT_S
    PeerGroup() {
        for (int g = 0; g < PEER_MAXR; g++) { base[g] = nullptr; mapped[g] = false; }
    }
    PeerPtrs peers() const {
        PeerPtrs p;
        for (int g = 0; g < PEER_MAXR; g++) p.base[g] = base[g];
        return p;
    }
    unsigned long long* flags(const PeerRank& r, int phase) const {
        return reinterpret_cast<unsigned long long*>(r.arena + off_flags) + (size_t)phase * PEER_MAXR;
    }
    int* status(const PeerRank& r) const { return reinterpret_cast<int*>(r.arena + off_status); }
};

struct DeviceGuard {
    int prev = 0;
    DeviceGuard() { cudaGetDevice(&prev); }
    ~DeviceGuard() { cudaSetDevice(prev); }
};

static inline size_t peer_align(size_t x) { return (x + 255) & ~(size_t)255; }
unsigned peer_grid(size_t n, size_t cap = 148 * 8);

// create-time argument checks shared by the handles (world a power of two <= ML_MAX_PEERS, one or all ranks local)
int peer_check_world(const char* who, int world, int n_local);
// device, context, the device's shared streams and the arena (first zero_bytes cleared) of one local rank
int peer_rank_init(PeerGroup& g, PeerRank& r, const char* who, size_t zero_bytes);
// every rank in this process: plain pointers; distinct devices get peer access in both directions
int peer_link_local(PeerGroup& g, const std::vector<PeerRank*>& ranks, const char* who);
int peer_export(const std::vector<PeerRank*>& ranks, uint8_t* records_out);
int peer_connect(PeerGroup& g, PeerRank& me, const uint8_t* records, size_t n_records, const char* who);
void peer_rank_free(PeerRank& r);      // arena
void peer_group_release(PeerGroup& g, int device);  // IPC mappings (closed on `device`) and streams
int peer_check_ready(const PeerGroup& g, const char* who);

// flag[phase][r.rank] = epoch in every rank's arena (only: a single target, or -1 for all)
int peer_signal(const PeerGroup& g, const PeerRank& r, int phase, int only, cudaStream_t s);
// wait for flag[phase][*] >= epoch in r's arena (only_from: a single source, or -1 for all)
int peer_wait(const PeerGroup& g, const PeerRank& r, int phase, int only_from, cudaStream_t s);
// the same for flags raised by an earlier call: flag[phase][*] >= epoch
int peer_wait_for(const PeerGroup& g, const PeerRank& r, int phase, int only_from, unsigned long long epoch, cudaStream_t s);
// copy nbytes (multiple of 16, <= 128) from src_dev to dst_off in the arenas of all ranks (or one), then raise the flag there
int peer_push(const PeerGroup& g, const PeerRank& r, const void* src_dev, int nbytes, size_t dst_off, int phase, int only, cudaStream_t s);
// ML_ERR_PEER if a wait of r's timed out, or the status rank 0 stored into r's status word (synchronises r's main stream)
int peer_read_status(const PeerGroup& g, const PeerRank& r, const char* who);

// The host side of a sharded handle: the ranks this process hosts, their group and the phase marks of the last call.  A handle
// type derives from it and adds its shape, arena layout and stages.
struct PeerHandle {
    int world = 1;
    const char* who = "";  // ABI prefix of the handle (ml_pcs_shard, ...), the prefix of its error messages
    std::vector<PeerRank> local;
    PeerGroup grp;
    // device-time marks of the last call on the first local rank's main stream (include/multilinear_b200_instr.h)
    static const int N_MARKS = 10;
    cudaEvent_t mark[N_MARKS] = {nullptr};
    int n_marks = 0;

    ~PeerHandle();  // marks, arenas (each device idle first), IPC mappings and streams
    // the group over an arena layout (timeout from MLB_SHARD_TIMEOUT_S), every local rank (first zero_bytes of its arena
    // cleared) and, when this process hosts every rank, the links between them (arguments checked by peer_check_world)
    int init(int world, int n_local, const int* local_ranks, const int* local_devices, size_t arena_bytes, size_t off_flags, size_t off_status,
             size_t zero_bytes);
    int export_records(uint8_t* records_out);
    int connect(const uint8_t* records, size_t n_records);  // a handle that hosts one rank
    void* stream(int local_index) const;
    int phase_ms(double* out, int cap) const;  // device time between consecutive marks
    void mark_phase(int idx);
    PeerRank* rank0();  // nullptr unless this process hosts rank 0
    int check_ready() const { return peer_check_ready(grp, who); }
    // host-pointer entry `entry` (a handle that hosts every rank): uploads n_blocks blocks of `bytes` to every local rank, block j of
    // rank r from src(r, j), runs run(dev) with block j of local rank i at dev[i * n_blocks + j], then frees the blocks
    int host_call(const char* entry, size_t n_blocks, size_t bytes, const std::function<const uint8_t*(int rank, size_t j)>& src,
                  const std::function<int(const void* const* dev)>& run);
};

}  // namespace mlb
