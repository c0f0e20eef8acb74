// The width-w System sumcheck (SumcheckTables::compute_sumcheck_polynomials, src/constraint_system/sumcheck.rs:147-202) sharded
// over G ranks, one GPU each; every round's coefficients, every challenge and the final transcript equal
// ml_wsumcheck_compute_polynomials'.  Notation: L = log2 G, h = 2^v rows, nloc = h/G, T = 2^WTAIL_LOG.
//
//   S0  h > T: rank b holds the row block [b*nloc, (b+1)*nloc) of the row-major [h][w] trace.  It stores every row into the
//       owner's table, which is CYCLIC: rank g owns global rows i = m*G + g at local row m.  The local eq table is
//       eq(row_point[0 .. v-L)) times prod_{b<L} (bit_b(g) ? p : 1-p), p = row_point[v-1-b] (local_eq_table).  Flag PX -> all.
//       h <= T: the block goes in natural order into every rank's tail tables; every rank builds the full eq table.
//   Round k (global height h >> k > T): every fold pair (i, i + h'/2) of the cyclic tables is local while h' >= 2G, and it is
//       the pair (m, m + h'/(2G)) of the local tables, so the single-GPU points, finish and fold kernels run unchanged on each
//       rank: wait PX (k = 0); points kernel -> CTA partials; the post kernel sums them into td values and stores them into
//       slot (k, g) of every rank's mailbox, flag PR0 + k -> all; wait for every post; wchain_finish_kernel reads the mailbox
//       as its partials with nb = G (its [block][td] layout is exactly [rank][td]); fold with the challenge in HBM.
//   All-gather (global height T): every rank stores its T/G rows of the matrix and of delta into every rank's tail tables at
//       natural index m*G + g; flag PG -> all.
//   Tail: wait PG; wchain_tail_kernel on T rows, identically on every rank; one D2H of the coefficients, randoms and transcript.
//   G = 1 takes no post or wait: the block is copied into the local tables and the rounds run exactly as the single-GPU path.
// Field sums are exact, so summing per rank first does not change any value.
#include "pcs_shard.h"
#include "reduce.cuh"

using namespace mlb;
using namespace mlbp;

namespace {

const char* WHO = "ml_wsumcheck_shard";
const size_t T_ROWS = (size_t)1 << WTAIL_LOG;
const int MAX_SR = 39 - WTAIL_LOG;  // sharded rounds: n_vars - WTAIL_LOG, n_vars < 40
// PD: the tail of the call is done (h <= T only: the next call's S0 stores into the peers' tail tables)
enum Phase { PX = 0, PG, PD, PR0, N_PHASES = PR0 + MAX_SR };
// the round-state block, as ml_wsumcheck_compute_polynomials lays it out: transcript | r | prev | Lagrange | coefficients | randoms
const size_t OFF_TR = 0, OFF_R = 128, OFF_PREV = 144, OFF_LAG = 160, OFF_CO = OFF_LAG + 32 * 16, OFF_RS = OFF_CO + 64 * W_MAX_TD * 16,
             HDR_BYTES = OFF_RS + 64 * 16;
const size_t SLOT_BYTES = (size_t)PEER_MAXR * W_MAX_TD * 16;  // one round's mailbox: td values per rank

struct WLayout {
    size_t flags, status, hdr, coef, len, off, cols, part, mail, m, d, tail_m, tail_d, total;
};

// block row o -> row (b*nloc + o) / G of rank o mod G (per = nloc / G rows per destination); a row is w * 16 contiguous bytes and
// a tile of consecutive rows for one destination is stored contiguously
__global__ void __launch_bounds__(256) wsc_transpose_kernel(const fe* __restrict__ block, size_t nloc, int width, int L, int log_per, int rank,
                                                            PeerPtrs peers, size_t off_m) {
    const int TR = 256;  // rows per tile
    const size_t per = (size_t)1 << log_per;
    const uint4* src = reinterpret_cast<const uint4*>(block);
    for (size_t base = (size_t)blockIdx.x * TR; base < nloc; base += (size_t)gridDim.x * TR) {
        for (int k = threadIdx.x; k < TR * width; k += blockDim.x) {
            const int rr = k / width, j = k - rr * width;
            const size_t x = base + rr;
            if (x >= nloc) break;
            const size_t dest = x >> log_per, ml = x & (per - 1);
            reinterpret_cast<uint4*>(peers.base[dest] + off_m)[((size_t)rank * per + ml) * width + j] = __ldg(src + ((ml << L) + dest) * width + j);
        }
    }
}
// rows local rows of the matrix (and of delta, if given) -> row m * stride + first of every rank's tail tables
__global__ void __launch_bounds__(256) wsc_gather_kernel(const fe* __restrict__ m, const fe* __restrict__ d, size_t rows, int width, size_t stride,
                                                         size_t first, int world, PeerPtrs peers, size_t off_tm, size_t off_td) {
    const size_t nm = rows * (size_t)width, total = nm + (d ? rows : 0), gs = (size_t)gridDim.x * blockDim.x;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gs) {
        size_t dst, off;
        uint4 v;
        if (e < nm) {
            const size_t row = e / width, j = e - row * width;
            v = __ldg(reinterpret_cast<const uint4*>(m) + e);
            dst = (row * stride + first) * width + j;
            off = off_tm;
        } else {
            const size_t row = e - nm;
            v = __ldg(reinterpret_cast<const uint4*>(d) + row);
            dst = row * stride + first;
            off = off_td;
        }
        for (int g = 0; g < world; g++) reinterpret_cast<uint4*>(peers.base[g] + off)[dst] = v;
    }
}
// this rank's td point sums (CTA partials [block][td]) -> slot `rank` of round k's mailbox in every rank's arena, then the flag there
__global__ void __launch_bounds__(256) wsc_post_kernel(const fe* __restrict__ part, int nb, int td, int rank, int world, PeerPtrs peers, size_t off_slot,
                                                       size_t off_flag, unsigned long long epoch) {
    __shared__ fe scratch[32];
    __shared__ fe sums[W_MAX_TD];
    for (int k = 0; k < td; k++) {
        fe a = fe_zero();
        for (int b = threadIdx.x; b < nb; b += blockDim.x) a = fe_add(a, part[(size_t)b * td + k]);
        a = block_sum(a, scratch);
        if (threadIdx.x == 0) sums[k] = a;
    }
    __syncthreads();
    const int g = threadIdx.x;
    if (g >= world) return;
    uint8_t* dst = peers.base[g];
    for (int k = 0; k < td; k++) fe_store(reinterpret_cast<fe*>(dst + off_slot) + (size_t)rank * td + k, sums[k]);
    __threadfence_system();
    flag_store_release(reinterpret_cast<unsigned long long*>(dst + off_flag) + rank, epoch);
}

}  // namespace

struct ml_wsumcheck_shard : PeerHandle {
    int L = 0;
    size_t n_vars = 0, h = 0, nloc = 0, width = 0, n_terms = 0, n_cols = 0;
    WLayout lay;
};

namespace {

inline fe* at(const PeerRank& r, size_t off) { return reinterpret_cast<fe*>(r.arena + off); }
bool sharded_rounds(const ml_wsumcheck_shard* sh) { return sh->h > T_ROWS; }
// the tables the tail runs on: the local tables at G = 1, else the all-gathered tail tables
fe* tail_m(const ml_wsumcheck_shard* sh, const PeerRank& r) { return at(r, sh->world == 1 ? sh->lay.m : sh->lay.tail_m); }
fe* tail_d(const ml_wsumcheck_shard* sh, const PeerRank& r) { return at(r, sh->world == 1 ? sh->lay.d : sh->lay.tail_d); }

WLayout make_layout(size_t h, size_t width, int G) {
    const size_t nloc = h / G, local_rows = G == 1 ? h : (h > T_ROWS ? nloc : 0), tail_rows = G == 1 ? 0 : (h < T_ROWS ? h : T_ROWS);
    WLayout a;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o = peer_align(o + bytes); return r; };
    a.flags = take((size_t)N_PHASES * PEER_MAXR * 8);
    a.status = take(16);
    a.hdr = take(HDR_BYTES);
    a.coef = take((size_t)W_MAX_TERMS * 16);
    a.len = take((size_t)W_MAX_TERMS * 4);
    a.off = take((size_t)W_MAX_TERMS * 4);
    a.cols = take((size_t)W_MAX_COLS * 4);
    a.part = take(((size_t)sumcheck_max_blocks() + 1) * W_MAX_TD * 16);
    a.mail = take(G > 1 ? (size_t)MAX_SR * SLOT_BYTES : 0);
    a.m = take(local_rows * width * 16);
    a.d = take(local_rows * 16);
    a.tail_m = take(tail_rows * width * 16);
    a.tail_d = take(tail_rows * 16);
    a.total = o;
    return a;
}

// S0 of one rank: round state, then the tables (module comment)
int stage_tables(ml_wsumcheck_shard* sh, PeerRank& r, const fe* block, const std::vector<hfe>& pts, const uint8_t* hdr_init) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    const WLayout& a = sh->lay;
    const int v = (int)sh->n_vars;
    MLB_TRY(h2d(r.arena + a.hdr, hdr_init, OFF_LAG + 25 * 16, s));
    MLB_CUDA(cudaMemsetAsync(sh->grp.status(r), 0, 16, s));
    if (sh->world == 1) {
        MLB_CUDA(cudaMemcpyAsync(at(r, a.m), block, sh->h * sh->width * 16, cudaMemcpyDeviceToDevice, s));
        return eq_table_launch(r.ctx, pts.data(), (size_t)v, at(r, a.d), s);
    }
    if (sharded_rounds(sh)) {
        wsc_transpose_kernel<<<peer_grid(sh->nloc), 256, 0, s>>>(block, sh->nloc, (int)sh->width, sh->L, (int)sh->n_vars - 2 * sh->L, r.rank,
                                                                        sh->grp.peers(), a.m);
        MLB_KERNEL_CHECK();
        MLB_TRY(mlbs::local_eq_table(r.ctx, pts, v, sh->L, r.rank, at(r, a.d), s));
    } else {
        if (sh->grp.epoch > 1) MLB_TRY(peer_wait_for(sh->grp, r, PD, -1, sh->grp.epoch - 1, s));  // the peers' last tail is done
        wsc_gather_kernel<<<peer_grid(sh->nloc * sh->width), 256, 0, s>>>(block, nullptr, sh->nloc, (int)sh->width, 1, (size_t)r.rank * sh->nloc, sh->world,
                                                                          sh->grp.peers(), a.tail_m, a.tail_d);
        MLB_KERNEL_CHECK();
        MLB_TRY(eq_table_launch(r.ctx, pts.data(), (size_t)v, at(r, a.tail_d), s));
    }
    return peer_signal(sh->grp, r, PX, -1, s);
}

// round k, phase A: the rank's td point sums (posted to every rank at G > 1)
int stage_points(ml_wsumcheck_shard* sh, PeerRank& r, int k, int td, const WTerms& terms, int* nb) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    const WLayout& a = sh->lay;
    const size_t hl = (sh->world == 1 ? sh->h : sh->nloc) >> k;
    if (k == 0 && sh->world > 1) MLB_TRY(peer_wait(sh->grp, r, PX, -1, s));
    MLB_TRY(wsumcheck_points_partials_launch(at(r, a.m), at(r, a.d), hl, sh->width, terms, td, at(r, a.part), nb, s));
    if (sh->world == 1) return ML_OK;
    wsc_post_kernel<<<1, 256, 0, s>>>(at(r, a.part), *nb, td, r.rank, sh->world, sh->grp.peers(), a.mail + (size_t)k * SLOT_BYTES,
                                      a.flags + (size_t)(PR0 + k) * PEER_MAXR * 8, sh->grp.epoch);
    MLB_KERNEL_CHECK();
    return ML_OK;
}
// round k, phase B: round polynomial and challenge from every rank's sums (identical on every rank), fold
int stage_finish(ml_wsumcheck_shard* sh, PeerRank& r, int k, int td, int nb) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    const WLayout& a = sh->lay;
    const size_t hl = (sh->world == 1 ? sh->h : sh->nloc) >> k;
    uint8_t* hdr = r.arena + a.hdr;
    const fe* partials = at(r, a.part);
    if (sh->world > 1) {
        MLB_TRY(peer_wait(sh->grp, r, PR0 + k, -1, s));
        partials = at(r, a.mail + (size_t)k * SLOT_BYTES);
        nb = sh->world;
    }
    MLB_TRY(wchain_finish_launch(partials, nb, td, (const fe*)(hdr + OFF_LAG), (fe*)(hdr + OFF_PREV), (DevTranscript*)(hdr + OFF_TR),
                                 (fe*)(hdr + OFF_CO) + (size_t)k * td, (fe*)(hdr + OFF_RS) + k, (fe*)(hdr + OFF_R), s));
    return wsumcheck_fold_dev_launch(at(r, a.m), at(r, a.d), hl, sh->width, (const fe*)(hdr + OFF_R), s);
}
// the local rows at global height T -> every rank's tail tables (G > 1)
int stage_gather(ml_wsumcheck_shard* sh, PeerRank& r) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    const WLayout& a = sh->lay;
    const size_t rows = T_ROWS / sh->world;
    wsc_gather_kernel<<<peer_grid(rows * (sh->width + 1)), 256, 0, s>>>(at(r, a.m), at(r, a.d), rows, (int)sh->width, (size_t)sh->world, (size_t)r.rank,
                                                                        sh->world, sh->grp.peers(), a.tail_m, a.tail_d);
    MLB_KERNEL_CHECK();
    return peer_signal(sh->grp, r, PG, -1, s);
}
// the remaining rounds in one CTA on T (or h) rows, identically on every rank
int stage_tail(ml_wsumcheck_shard* sh, PeerRank& r, int k, int td, const WTerms& terms) {
    MLB_CUDA(cudaSetDevice(r.device));
    cudaStream_t s = r.st.main;
    uint8_t* hdr = r.arena + sh->lay.hdr;
    const bool sharded = sharded_rounds(sh);
    if (sh->world > 1) MLB_TRY(peer_wait(sh->grp, r, sharded ? PG : PX, -1, s));
    MLB_TRY(wchain_tail_launch(tail_m(sh, r), tail_d(sh, r), sh->h >> k, (int)sh->width, terms, td, (const fe*)(hdr + OFF_LAG), (fe*)(hdr + OFF_PREV),
                               (DevTranscript*)(hdr + OFF_TR), (fe*)(hdr + OFF_CO) + (size_t)k * td, (fe*)(hdr + OFF_RS) + k, s));
    if (sh->world > 1 && !sharded) return peer_signal(sh->grp, r, PD, -1, s);
    return ML_OK;
}

}  // namespace

extern "C" {

int ml_wsumcheck_shard_create(int world, int n_local, const int* local_ranks, const int* local_devices, size_t width, size_t n_vars,
                              ml_wsumcheck_shard** out) {
    MLB_TRY(peer_check_world("ml_wsumcheck_shard_create", world, n_local));
    if (width == 0 || width > (size_t)W_MAX_WIDTH) { set_error("ml_wsumcheck_shard_create: trace width must be 1..%d", W_MAX_WIDTH); return ML_ERR_ARG; }
    const int L = (int)ilog2((size_t)world);
    if (n_vars < 1 || n_vars < (size_t)L || n_vars >= 40) {
        set_error("ml_wsumcheck_shard_create: n_vars = %zu, need max(1, log2(world)) = %d <= n_vars < 40", n_vars, L ? L : 1);
        return ML_ERR_SIZE;
    }
    DeviceGuard guard;
    ml_wsumcheck_shard* sh = new ml_wsumcheck_shard();
    sh->who = WHO;
    sh->L = L; sh->n_vars = n_vars; sh->h = (size_t)1 << n_vars; sh->nloc = sh->h / world; sh->width = width;
    sh->lay = make_layout(sh->h, width, world);
    int st = sh->init(world, n_local, local_ranks, local_devices, sh->lay.total, sh->lay.flags, sh->lay.status, sh->lay.hdr);
    if (st != ML_OK) { delete sh; return st; }
    *out = sh;
    return ML_OK;
}

void ml_wsumcheck_shard_free(ml_wsumcheck_shard* sh) { delete sh; }
int ml_wsumcheck_shard_export(ml_wsumcheck_shard* sh, uint8_t* records_out) { return sh->export_records(records_out); }
int ml_wsumcheck_shard_connect(ml_wsumcheck_shard* sh, const uint8_t* records, size_t n_records) { return sh->connect(records, n_records); }
void* ml_wsumcheck_shard_stream(const ml_wsumcheck_shard* sh, int local_index) { return sh->stream(local_index); }
size_t ml_wsumcheck_shard_arena_bytes(const ml_wsumcheck_shard* sh) { return sh->lay.total; }

int ml_wsumcheck_shard_set_composition(ml_wsumcheck_shard* sh, size_t n_terms, const uint8_t* coefs, const uint32_t* term_lens, const uint32_t* term_cols) {
    std::vector<uint32_t> off;
    size_t total = 0;
    MLB_TRY(wsumcheck_check_terms(sh->width, n_terms, term_lens, term_cols, off, &total));
    DeviceGuard guard;
    const WLayout& a = sh->lay;
    for (auto& r : sh->local) {
        MLB_CUDA(cudaSetDevice(r.device));
        cudaStream_t s = r.st.main;
        MLB_TRY(h2d(r.arena + a.coef, coefs, n_terms * 16, s));
        MLB_TRY(h2d(r.arena + a.len, term_lens, n_terms * 4, s));
        MLB_TRY(h2d(r.arena + a.off, off.data(), n_terms * 4, s));
        MLB_TRY(h2d(r.arena + a.cols, term_cols, total * 4, s));
        MLB_CUDA(cudaStreamSynchronize(s));  // off is a host temporary
    }
    sh->n_terms = n_terms; sh->n_cols = total;
    return ML_OK;
}

// SumcheckTables::compute_sumcheck_polynomials (sumcheck.rs:147-202) over the trace whose row block [rank*h/G, (rank+1)*h/G) local
// rank i holds at local_blocks_dev[i] (row-major [rows][width], only read).  Every process passes the same row point, sum and
// transcript and gets the whole result.
int ml_wsumcheck_shard_compute_polynomials_dev(ml_wsumcheck_shard* sh, const uint8_t* row_point, size_t n_vars, const void* const* local_blocks_dev,
                                               size_t composition_degree, ml_transcript* t, const uint8_t sum[16], uint8_t* coeffs_out,
                                               uint8_t* randoms_out) {
    if (composition_degree + 1 > (size_t)W_MAX_TD) {
        set_error("%s: composition_degree %zu, at most %d", WHO, composition_degree, W_MAX_TD - 1);
        return ML_ERR_ARG;
    }
    MLB_TRY(sh->check_ready());
    if (n_vars != sh->n_vars) { set_error("%s: the row point has %zu variables, the handle %zu", WHO, n_vars, sh->n_vars); return ML_ERR_SIZE; }
    DeviceGuard guard;
    const int td = (int)composition_degree + 1, v = (int)n_vars;
    sh->grp.epoch++;
    std::vector<hfe> pts(n_vars);
    for (size_t i = 0; i < n_vars; i++) pts[i] = hfe_load(row_point + 16 * i);
    std::vector<uint8_t> lag;
    MLB_TRY(wsumcheck_lagrange((size_t)td, lag));
    std::vector<uint8_t> hdr_init(OFF_LAG + 25 * 16, 0);  // transcript | r | prev = sum | Lagrange matrix
    memcpy(hdr_init.data() + OFF_TR, &t->sha, sizeof(DevTranscript));
    memcpy(hdr_init.data() + OFF_PREV, sum, 16);
    memcpy(hdr_init.data() + OFF_LAG, lag.data(), lag.size());
    const size_t nl = sh->local.size();
    std::vector<int> nb(nl, 0);
    for (size_t i = 0; i < nl; i++) MLB_TRY(stage_tables(sh, sh->local[i], (const fe*)local_blocks_dev[i], pts, hdr_init.data()));
    const int sr = sharded_rounds(sh) ? v - WTAIL_LOG : 0;
    for (int k = 0; k < sr; k++) {
        for (size_t i = 0; i < nl; i++) {
            PeerRank& r = sh->local[i];
            const WTerms terms{at(r, sh->lay.coef), (const uint32_t*)(r.arena + sh->lay.len), (const uint32_t*)(r.arena + sh->lay.off),
                               (const uint32_t*)(r.arena + sh->lay.cols), (int)sh->n_terms, (int)sh->n_cols};
            MLB_TRY(stage_points(sh, r, k, td, terms, &nb[i]));
        }
        for (size_t i = 0; i < nl; i++) MLB_TRY(stage_finish(sh, sh->local[i], k, td, nb[i]));
    }
    if (sr > 0 && sh->world > 1)
        for (size_t i = 0; i < nl; i++) MLB_TRY(stage_gather(sh, sh->local[i]));
    for (size_t i = 0; i < nl; i++) {
        PeerRank& r = sh->local[i];
        const WTerms terms{at(r, sh->lay.coef), (const uint32_t*)(r.arena + sh->lay.len), (const uint32_t*)(r.arena + sh->lay.off),
                           (const uint32_t*)(r.arena + sh->lay.cols), (int)sh->n_terms, (int)sh->n_cols};
        MLB_TRY(stage_tail(sh, r, sr, td, terms));
    }
    int st = ML_OK;
    for (auto& r : sh->local) {  // a timed-out wait on any local rank fails the call
        const int s1 = peer_read_status(sh->grp, r, WHO);
        if (s1 != ML_OK) st = s1;
    }
    MLB_TRY(st);
    PeerRank& r0 = sh->local[0];
    MLB_CUDA(cudaSetDevice(r0.device));
    std::vector<uint8_t> host(HDR_BYTES);
    MLB_TRY(d2h_sync(host.data(), r0.arena + sh->lay.hdr, HDR_BYTES, r0.st.main));
    memcpy(coeffs_out, host.data() + OFF_CO, n_vars * td * 16);
    memcpy(randoms_out, host.data() + OFF_RS, n_vars * 16);
    memcpy(&t->sha, host.data() + OFF_TR, sizeof(DevTranscript));
    return ML_OK;
}

// host rows (all h) and a handle that hosts every rank: the drop-in for build + set_composition + compute_sumcheck_polynomials
int ml_wsumcheck_shard_compute_polynomials(ml_wsumcheck_shard* sh, const uint8_t* row_point, size_t n_vars, const uint8_t* matrix, size_t width,
                                           size_t height, size_t composition_degree, ml_transcript* t, const uint8_t sum[16], uint8_t* coeffs_out,
                                           uint8_t* randoms_out) {
    if (width != sh->width) { set_error("ml_wsumcheck_shard_compute_polynomials: trace width %zu, the handle's %zu", width, sh->width); return ML_ERR_ARG; }
    if (n_vars != sh->n_vars || height != sh->h) { set_error("ml_wsumcheck_shard_compute_polynomials: need 2^n_vars == height == the handle's"); return ML_ERR_SIZE; }
    const size_t bytes = sh->nloc * width * 16;
    return sh->host_call("ml_wsumcheck_shard_compute_polynomials", 1, bytes, [&](int rank, size_t) { return matrix + (size_t)rank * bytes; },
                         [&](const void* const* dev) {
                             return ml_wsumcheck_shard_compute_polynomials_dev(sh, row_point, n_vars, dev, composition_degree, t, sum, coeffs_out, randoms_out);
                         });
}

}  // extern "C"
