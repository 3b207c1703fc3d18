// Host side of the rank-based 3-D ant colony search: handle, buffers in HBM, the per-iteration
// kernel sequence, and the C ABI (include/wr_gpu.h) that stands in for ACS_Rank
// (core/ACSRank_3D.hpp).  An iteration is a fixed sequence of launches whose sizes live on the
// device (IterState), so wr_acs_iterate(n) never synchronises with the host.
#include <stdarg.h>
#include <stddef.h>
#include <stdlib.h>

#include <algorithm>
#include <mutex>
#include <utility>
#include <vector>

#include "acs_kernels.cuh"
#include "walk2.cuh"
#include "walk26.cuh"
#include "walk3.cuh"
#include "rank_small.cuh"
#include "rankset.cuh"
#include "batch.cuh"
#include "batch26.cuh"
#include "wr_internal.cuh"

namespace wr {

constexpr uint32_t kPubBlocks = 262144;   // sharded colonies: row blocks a rank can publish per iteration (35.7 MB of its peer slab)

static thread_local std::string g_err;
void set_error(const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
}

cudaError_t pool_malloc(void** p, size_t bytes, cudaStream_t s)
{
    static bool configured[64] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64 && !configured[dev]) {
        cudaMemPool_t pool;
        e = cudaDeviceGetDefaultMemPool(&pool, dev);
        if (e != cudaSuccess) return e;
        unsigned long long keep = ~0ull;
        e = cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        if (e != cudaSuccess) return e;
        configured[dev] = true;
    }
    return cudaMallocAsync(p, bytes ? bytes : 1, s);
}
void pool_free(void* p, cudaStream_t s)
{
    if (p) cudaFreeAsync(p, s);
}

static int ceil_log2(unsigned long long v)
{
    int b = 0;
    while ((1ull << b) < v) b++;
    return b;
}

struct PhaseTimer {
    std::vector<cudaEvent_t> ev;
    size_t used = 0;
    float ms[5] = {0, 0, 0, 0, 0};
    bool enabled = false;
    cudaEvent_t next()
    {
        if (used == ev.size()) { cudaEvent_t e; cudaEventCreate(&e); ev.push_back(e); }
        return ev[used++];
    }
    void resolve()
    {   // groups of 5 events: [begin, after walk, after rank, after deposit build, end]
        for (size_t i = 0; i + 5 <= used; i += 5) {
            float t;
            for (int k = 0; k < 4; k++) { if (cudaEventElapsedTime(&t, ev[i + k], ev[i + k + 1]) == cudaSuccess) ms[k] += t; }
            if (cudaEventElapsedTime(&t, ev[i], ev[i + 4]) == cudaSuccess) ms[4] += t;
        }
        used = 0;
    }
    ~PhaseTimer() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }
};

}  // namespace wr

using namespace wr;

struct wr_acs {
    wr_grid* g = nullptr;
    wr_acs_params p;
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    size_t N = 0, n_slots = 0, n_slots_pad = 0;
    int K = 6;                        // directed slots per node: 6 (the reference) or 26 (walk26.cuh)
    float* d_ant_L = nullptr;         // K = 26: length of every ant of the last iteration (+inf: dead)
    unsigned ntiles = 0;
    int cap = 0, rank_bits = 0, slot_bits = 0;
    int table_log2 = 9, gtable_log2 = 0;
    int table_entries = 512;          // k_walk2: entries per ant (768 by default: two 16-ant CTAs per SM)
    int64_t start = -1, goal = -1;
    // many searches (wr_acs_search_pairs / wr_acs_search_batch): packed results of the last call, batch buffers
    std::vector<float> res_L; std::vector<int> res_n; std::vector<size_t> res_off; std::vector<uint32_t> res_ids; std::vector<uint8_t> res_dirs;
    struct wr_batch* batch = nullptr;
    uint32_t batch_last_entries = 0, batch_fallbacks = 0;
    bool field_clean = true;          // the pheromone field is in its initial / reset() state
    int gtable_log2_for_cap() const { int b = 0; while ((1ull << b) < (unsigned long long)cap + 3) b++; return b; }
    uint32_t search = 0, next_search = 0;   // Philox: index of the current computeSolution on this handle / of the next wr_acs_begin
    bool begun = false;
    int colony_max = 0, w_max = 0;
    // shard (multi-rank)
    int rank = 0, nranks = 1, chunk = 0;
    // Sharded colonies on NVLink: everything a peer reads lives in ONE cudaMalloc'd slab (IPC-exportable with a single
    // handle, same layout on every rank): the ant trails and the list of final slot values of the owner-computes
    // update, each double-buffered by iteration parity.   [ids0 | ids1 | dirs0 | dirs1 | fin0 | fin1]
    unsigned char* d_slab = nullptr;
    size_t slab_bytes = 0, off_ids[2] = {0, 0}, off_dirs[2] = {0, 0}, off_fin[2] = {0, 0}, off_steps[2] = {0, 0}, off_pub = 0, off_flags = 0;
    const void** d_tabs = nullptr;    // device: [kind 0 ids,1 dirs,2 fin,3 steps,4 publish area,5 barrier flags][parity][rank] -> pointer into rank's slab
    cudaStream_t side = nullptr;      // sharded rank-set iterations: the evaporation pass runs here, beside the exchange (barriers, ranking, merge)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    bool evap_forked = false;
    void* comm = nullptr;             // NCCL communicator (wr_acs_comm_init): wr_acs_begin exchanges the peer slabs through it
    uint32_t* d_epoch = nullptr;      // [0] unused [1] = d_peer_err
    uint32_t* d_peer_err = nullptr;   // set by a barrier that timed out (a peer died): reported by wr_acs_sync
    unsigned long long barrier_timeout_ns = 20000000000ull;
    std::vector<void*> ipc_opened;
    bool peers_set = false;
    bool in_process_peers = false;   // the peers are handles of THIS process (wr_acs_peer_set_pointers; tests): one plain stream per shard, see there
    int* d_nq = nullptr;              // records in this rank's slot slice
    unsigned parity = 0;              // flips at every wr_acs_walk of a sharded handle
    bool warm_by_pull = false;        // the last iteration ended with k_pull_finals (which doubles as the L2 warm-up)

    float* d_tau = nullptr;
    float* d_heur = nullptr;          // [N][6] heuristic factor for the current goal
    int64_t heur_goal = -1;           // goal it was computed for
    IterState* d_state = nullptr;
    uint32_t* d_onbest = nullptr;
    float* d_Ltab = nullptr;
    std::vector<float> h_Ltab;
    int* d_best_n = nullptr;
    uint32_t* d_best_ids = nullptr;
    uint8_t* d_best_dirs = nullptr;
    // per-colony buffers (sized at begin)
    int* d_ant_steps = nullptr;      // global colony order (ranking input)
    int* d_local_steps = nullptr;    // this rank's chunk (== d_ant_steps when nranks == 1)
    uint32_t* d_path_ids = nullptr;
    uint8_t* d_path_dirs = nullptr;
    uint32_t* d_overflow = nullptr;
    uint32_t* d_gkeys = nullptr;      // HBM visited tables for overflowed ants, one per local ant
    unsigned long long* d_gmasks = nullptr;
    int4* d_resume = nullptr;
    int walk2_blocks = 0;
    uint32_t* d_rec_off = nullptr;
    int* d_order = nullptr;
    uint32_t* d_tile_off = nullptr;
    uint32_t* d_dep_list = nullptr;   // tiles that receive deposits this iteration
    uint32_t* d_upd_q = nullptr;      // [0] deposit-tile queue [1] plain-chunk queue [2] deposit-tile count
    SortPlan sort_ants, sort_recs;
    bool ants_in_b = false, recs_in_b = false;
    size_t alloc_colony = 0;
    PhaseTimer timer;
    // WR_UPDATE_RANKSET (rankset.cuh)
    bool want_rankset = false, rankset = false;
    RankSet rs = {};
    size_t rs_entries = 0;
    int rs_groups = 1;                // apply launches per iteration: ceil(w_max / 1024)
    int rs_policy = 0;                // 0 adaptive, 1 rank sets always, 2 records always (WR_RANKSET_POLICY)
    // adaptive choice: device -> host feedback through mapped pinned memory, host kept <= kRsAhead iterations ahead
    uint32_t* h_feedback = nullptr;   // ring of kFeedbackRing x {generation << 16 | iteration, path of the previous iteration, deposit tiles, row blocks}
    uint32_t* d_feedback = nullptr;   // the same words as the device sees them
    uint32_t rs_generation = 0;       // bumped by wr_acs_begin: feedback of an earlier search on the same stream is ignored
    int rs_choice = 0;                // path of the iteration being enqueued
    uint8_t rs_history[16] = {};      // path of the last 16 iterations enqueued (index = iteration & 15)
    static constexpr int kRsAhead = 4;
    cudaEvent_t rs_ev[kRsAhead] = {};
    unsigned long long rs_enqueued = 0;
    unsigned rs_on = 2000, rs_off = 120000;   // switch thresholds: deposit tiles / distinct slots (WR_RANKSET_ON / WR_RANKSET_OFF)
    bool upd_q_zeroed = false;        // this iteration's k_iter_begin already cleared d_upd_q (wr_acs_iterate)
    // steady-state rank-set iteration (previous and current iteration on the rank-set path, folded k_iter_end, no timers) as ONE
    // CUDA graph launch: 9 kernels whose arguments do not change within a search; re-captured after wr_acs_begin
    cudaGraphExec_t rs_graph[2] = {nullptr, nullptr};   // sharded handles: one per trail-buffer parity
    bool rs_graph_failed = false;
    // device time of the streaming kernel alone (k_update_fused / k_evaporate_tiles), inside the loop: event pairs around it
    std::vector<cudaEvent_t> sk_ev;
    size_t sk_used = 0;
    float sk_ms = 0;
    int sk_launches = 0;
    cudaEvent_t sk_next()
    {
        if (sk_used == sk_ev.size()) { cudaEvent_t e; cudaEventCreate(&e); sk_ev.push_back(e); }
        return sk_ev[sk_used++];
    }
    void sk_resolve()
    {
        for (size_t i = 0; i + 2 <= sk_used; i += 2) {
            float t;
            if (cudaEventElapsedTime(&t, sk_ev[i], sk_ev[i + 1]) == cudaSuccess) { sk_ms += t; sk_launches++; }
        }
        sk_used = 0;
    }
    // clean-tile field (acs_kernels.cuh): per-tile dirty flags; lazy = in-bounds slots start as sentinels (FUSED / RANKSET handles)
    uint8_t* d_dirty = nullptr;
    bool lazy = false;
    bool oob_zero = true;             // out-of-bounds slots still hold their initial 0 (until the first reset())

    static constexpr int kTabKinds = 6;
    const void** tab(int kind, unsigned par) const { return d_tabs + ((size_t)kind * 2 + par) * nranks; }
    uint32_t* fin_buf(unsigned par) const { return reinterpret_cast<uint32_t*>(d_slab + off_fin[par]); }
    uint32_t* pub_buf() const { return reinterpret_cast<uint32_t*>(d_slab + off_pub); }
    const uint32_t* const* trail_ids_tab() const { return reinterpret_cast<const uint32_t* const*>(tab(0, parity)); }   // [rank] -> trail buffers of this iteration
    const uint8_t* const* trail_dirs_tab() const { return reinterpret_cast<const uint8_t* const*>(tab(1, parity)); }
    uint32_t* flags_buf() const { return reinterpret_cast<uint32_t*>(d_slab + off_flags); }
    const int* dptr_colony() const { return reinterpret_cast<const int*>(reinterpret_cast<const char*>(d_state) + offsetof(IterState, colony)); }
    const int* dptr_nrec() const { return reinterpret_cast<const int*>(reinterpret_cast<const char*>(d_state) + offsetof(IterState, n_records)); }
    // record count the record path's kernels see: 0 on iterations an adaptive handle runs through rank sets
    const int* dptr_nrec_upd() const
    {
        return reinterpret_cast<const int*>(reinterpret_cast<const char*>(d_state) + (rankset ? offsetof(IterState, n_records_sort) : offsetof(IterState, n_records)));
    }
};

static void drop_steady_graph(wr_acs* a)
{
    for (cudaGraphExec_t& g : a->rs_graph) if (g) { cudaGraphExecDestroy(g); g = nullptr; }
    a->rs_graph_failed = false;
}

// A rank-set table is all zeros whenever no iteration is in flight (k_rankset_apply clears what k_rankset_gen set), so a
// destroyed handle's table can be handed to the next handle of the same shape without the 1-2 GB memset: one parked
// table per process (searches created in a loop, one per request, are the e2e pattern).
struct RankSetCache {
    int device = -1;
    size_t entries = 0;
    uint32_t limit = 0;
    int w_max = 0;
    RankSet rs = {};   // all six buffers travel together, so a handle that adopts them adds no traffic to the memory pool
};
static RankSetCache g_rs_cache;
static std::mutex g_rs_cache_mu;   // handles may be created and destroyed on different host threads

// Feedback words (device -> host, mapped pinned memory): pinned allocations cost milliseconds, handles are created per
// request, so one block is pinned per process and handles borrow a 128-byte slot of it (a ring of kFeedbackRing records:
// the host reads the record of one specific, already finished iteration, so that its choice of the deposit path is a
// pure function of the search — the same on every rank of a sharded colony, the same in every run).
constexpr int kFeedbackRing = 8;
constexpr int kFeedbackWords = 4 * kFeedbackRing;
struct FeedbackPage {
    uint32_t* host = nullptr;
    uint32_t* dev = nullptr;
    bool used[256] = {};
};
static FeedbackPage g_feedback;

static int feedback_acquire(uint32_t** h, uint32_t** d)
{
    std::lock_guard<std::mutex> lock(g_rs_cache_mu);
    if (!g_feedback.host) {
        WR_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&g_feedback.host), 256 * kFeedbackWords * sizeof(uint32_t), cudaHostAllocMapped | cudaHostAllocPortable));
        WR_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&g_feedback.dev), g_feedback.host, 0));
    }
    for (int i = 0; i < 256; i++)
        if (!g_feedback.used[i]) {
            g_feedback.used[i] = true;
            *h = g_feedback.host + kFeedbackWords * i; *d = g_feedback.dev + kFeedbackWords * i;
            for (int k = 0; k < kFeedbackWords; k++) (*h)[k] = 0xFFFFFFFFu;
            return WR_OK;
        }
    *h = nullptr; *d = nullptr;   // all slots taken: the handle runs without feedback (records path only)
    return WR_OK;
}
static void feedback_release(uint32_t* h)
{
    if (!h) return;
    std::lock_guard<std::mutex> lock(g_rs_cache_mu);
    g_feedback.used[(h - g_feedback.host) / kFeedbackWords] = false;
}

// The rank-set buffers outlive handles (they are parked between searches), so they come from cudaMalloc, not from the
// stream-ordered pool whose blocks are tied to the allocating handle's stream.
static void rankset_release_buffers(RankSet& rs, cudaStream_t)
{
    cudaFree(rs.key); cudaFree(rs.rows); cudaFree(rs.list); cudaFree(rs.touched); cudaFree(rs.count); cudaFree(rs.vtab);
    rs = RankSet{};
}

static void free_rankset(wr_acs* a)
{
    cudaStream_t s = a->stream;
    if (a->rs.key) {
        cudaStreamSynchronize(s);   // the table is clean once the stream has drained
        std::lock_guard<std::mutex> lock(g_rs_cache_mu);
        if (g_rs_cache.rs.key) rankset_release_buffers(g_rs_cache.rs, s);
        g_rs_cache.device = a->device; g_rs_cache.entries = a->rs_entries; g_rs_cache.limit = a->rs.limit; g_rs_cache.w_max = a->w_max;
        g_rs_cache.rs = a->rs;
    }
    a->rs = RankSet{};
    a->rankset = false; a->rs_entries = 0;
}

// Sharded searches created in a loop (one per request): the peer slab and the IPC mappings of the peers' slabs are kept
// across handles.  cudaMalloc/cudaFree of a ~0.5 GB slab and cudaIpcOpenMemHandle/Close of every peer's cost tens of
// milliseconds per search; a parked slab keeps its address, hence its IPC handle, hence the peers' mappings stay valid.
struct SlabCache {
    int device = -1;
    size_t bytes = 0;
    unsigned char* ptr = nullptr;
};
static SlabCache g_slab_cache;
struct IpcMapping {
    cudaIpcMemHandle_t handle;
    void* ptr = nullptr;
};
static std::vector<IpcMapping> g_ipc_maps;   // one per peer rank (a process drives one GPU)
struct SideStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
    int device = -1;
    bool in_use = false;
};
static std::vector<SideStream> g_side_streams;   // side streams of sharded handles, parked between handles

static void free_colony_buffers(wr_acs* a)
{
    cudaStream_t s = a->stream;
    drop_steady_graph(a);
    free_rankset(a);
    pool_free(a->d_ant_steps, s); pool_free(a->d_overflow, s); pool_free(a->d_ant_L, s); a->d_ant_L = nullptr;
    if (!a->d_slab) { pool_free(a->d_path_ids, s); pool_free(a->d_path_dirs, s); }
    pool_free(a->d_gkeys, s); pool_free(a->d_gmasks, s); pool_free(a->d_resume, s); a->d_resume = nullptr; pool_free(a->d_rec_off, s); pool_free(a->d_order, s);
    a->d_local_steps = nullptr;   // aliases d_ant_steps (one GPU) or lives in the slab (sharded)
    pool_free(a->d_epoch, s); a->d_epoch = nullptr; a->d_peer_err = nullptr;
    a->d_ant_steps = nullptr; a->d_path_ids = nullptr; a->d_path_dirs = nullptr; a->d_overflow = nullptr;
    a->d_gkeys = nullptr; a->d_gmasks = nullptr; a->d_rec_off = nullptr; a->d_order = nullptr;
    sort_plan_destroy(&a->sort_ants, s); sort_plan_destroy(&a->sort_recs, s);
    a->ipc_opened.clear();   // the mappings live in g_ipc_maps
    if (a->d_slab) {
        cudaStreamSynchronize(s);
        {
            std::lock_guard<std::mutex> lock(g_rs_cache_mu);
            if (g_slab_cache.ptr) cudaFree(g_slab_cache.ptr);   // peers that still map it re-open on the next handle exchange
            g_slab_cache.device = a->device; g_slab_cache.bytes = a->slab_bytes; g_slab_cache.ptr = a->d_slab;
        }
        a->d_slab = nullptr;
        a->d_path_ids = nullptr; a->d_path_dirs = nullptr;   // they pointed into the slab
    }
    pool_free(a->d_tabs, s); a->d_tabs = nullptr;
    pool_free(a->d_nq, s); a->d_nq = nullptr;
    a->peers_set = false; a->slab_bytes = 0;
    a->alloc_colony = 0;
}

static int alloc_colony_buffers(wr_acs* a, int colony_max)
{
    if ((size_t)colony_max <= a->alloc_colony && a->alloc_colony) return WR_OK;
    free_colony_buffers(a);
    const size_t cm = std::max(colony_max, 1);
    const size_t cap = a->cap;
    a->chunk = (int)((cm + a->nranks - 1) / a->nranks);
    const size_t chunk = a->chunk;
    a->w_max = (int)(0.2 * (double)cm) + 1;
    const size_t rec_max = (size_t)a->w_max * cap;
    if (rec_max >= 0x7fffffffull) { set_error("colony %zu x step cap %zu needs too many deposit records; set step_cap", cm, cap); return WR_ERR_NOMEM; }
    WR_CUDA(dmalloc(&a->d_ant_steps, (chunk * a->nranks) * sizeof(int), a->stream));   // global colony: ranking reads all ranks' steps
    if (a->nranks > 1) {
        auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
        size_t o = 0;
        a->off_flags = o; o += up(4096);                                             // barrier flags: one epoch word per source rank
        for (int b = 0; b < 2; b++) { a->off_steps[b] = o; o += up(chunk * sizeof(int)); }
        for (int b = 0; b < 2; b++) { a->off_ids[b] = o; o += up(chunk * cap * sizeof(uint32_t)); }
        for (int b = 0; b < 2; b++) { a->off_dirs[b] = o; o += up(chunk * cap); }
        for (int b = 0; b < 2; b++) { a->off_fin[b] = o; o += up((4 + 2 * rec_max) * sizeof(uint32_t)); }
        a->off_pub = o; o += up(((size_t)4 + (size_t)kPubBlocks * kRsPubWords) * sizeof(uint32_t));
        a->slab_bytes = o;
        {
            std::lock_guard<std::mutex> lock(g_rs_cache_mu);
            if (g_slab_cache.ptr && g_slab_cache.device == a->device && g_slab_cache.bytes == a->slab_bytes) {
                a->d_slab = g_slab_cache.ptr;
                g_slab_cache = SlabCache();
            }
        }
        if (!a->d_slab) WR_CUDA(cudaMalloc(&a->d_slab, a->slab_bytes));
        for (int b = 0; b < 2; b++) WR_CUDA(cudaMemsetAsync(a->d_slab + a->off_fin[b], 0, 4 * sizeof(uint32_t), a->stream));
        WR_CUDA(cudaMemsetAsync(a->d_slab + a->off_pub, 0, 4 * sizeof(uint32_t), a->stream));
        WR_CUDA(dmalloc(&a->d_tabs, (size_t)wr_acs::kTabKinds * 2 * a->nranks * sizeof(void*), a->stream));
        WR_CUDA(dmalloc(&a->d_nq, sizeof(int), a->stream));
        WR_CUDA(dmalloc(&a->d_epoch, 2 * sizeof(uint32_t), a->stream));
        a->d_peer_err = a->d_epoch + 1;
        a->parity = 0;
        a->d_path_ids = reinterpret_cast<uint32_t*>(a->d_slab + a->off_ids[0]);
        a->d_path_dirs = a->d_slab + a->off_dirs[0];
        a->d_local_steps = reinterpret_cast<int*>(a->d_slab + a->off_steps[0]);
    } else a->d_local_steps = a->d_ant_steps;
    if (a->nranks == 1) {
        WR_CUDA(dmalloc(&a->d_path_ids, chunk * cap * sizeof(uint32_t), a->stream));
        WR_CUDA(dmalloc(&a->d_path_dirs, chunk * cap, a->stream));
        WR_CUDA(dmalloc(&a->d_tabs, (size_t)wr_acs::kTabKinds * 2 * sizeof(void*), a->stream));   // a one-rank table for the kernels that take one
        const void* tab[wr_acs::kTabKinds * 2] = {};
        tab[0] = tab[1] = a->d_path_ids; tab[2] = tab[3] = a->d_path_dirs;
        WR_CUDA(cudaMemcpyAsync(a->d_tabs, tab, sizeof tab, cudaMemcpyHostToDevice, a->stream));
        WR_CUDA(cudaStreamSynchronize(a->stream));   // `tab` is on the stack
    }
    WR_CUDA(dmalloc(&a->d_overflow, chunk * sizeof(uint32_t), a->stream));
    if (a->K == kK26) WR_CUDA(dmalloc(&a->d_ant_L, chunk * sizeof(float), a->stream));
    WR_CUDA(dmalloc(&a->d_rec_off, cm * sizeof(uint32_t), a->stream));
    WR_CUDA(dmalloc(&a->d_order, cm * sizeof(int), a->stream));
    WR_CUDA(cudaMemsetAsync(a->d_order, 0, cm * sizeof(int), a->stream));
    // HBM visited tables for ants whose shared-memory table fills up: every tile an ant can touch fits
    // (tiles <= steps+1 <= cap+1), one table per local ant so that any number of them can overflow
    a->gtable_log2 = ceil_log2((unsigned long long)cap + 3);
    a->walk2_blocks = (int)std::min<size_t>((chunk + kAntsPerCta - 1) / kAntsPerCta, (size_t)kNumSMs * 4);
    const size_t gslots = chunk << a->gtable_log2;
    if (gslots * 12 > ((size_t)48 << 30)) { set_error("colony %zu x step cap %zu needs %zu GB of overflow tables; set a smaller step_cap", cm, cap, (gslots * 12) >> 30); return WR_ERR_NOMEM; }
    WR_CUDA(dmalloc(&a->d_gkeys, gslots * sizeof(uint32_t), a->stream));
    WR_CUDA(dmalloc(&a->d_gmasks, gslots * sizeof(unsigned long long), a->stream));
    WR_CUDA(dmalloc(&a->d_resume, chunk * sizeof(int4), a->stream));
    int st = sort_plan_create(&a->sort_ants, cm, a->stream);
    if (st != WR_OK) return st;
    // WR_UPDATE_RANKSET: open-addressed table of (slot, rank group) row blocks with a FIXED capacity (rankset.cuh): the path is
    // only chosen while the colony's deposits are concentrated, an overflow falls back to an exact serial pass
    a->rankset = false;
    if (a->want_rankset) {
        int log2R = 20;   // 2^20 blocks: 8 MB of keys + 134 MB of rows
        if (const char* e = getenv("WR_RANKSET_LOG2")) log2R = std::max(6, std::min(26, atoi(e)));
        const size_t R = (size_t)1 << log2R;
        uint32_t limit = (uint32_t)(R / 2);
        if (a->nranks > 1) limit = std::min<uint32_t>(limit, kPubBlocks);   // what fits in the publish area of the peer slab
        cudaStream_t s = a->stream;
        {
            std::lock_guard<std::mutex> lock(g_rs_cache_mu);
            if (g_rs_cache.rs.key && g_rs_cache.device == a->device && g_rs_cache.entries == R && g_rs_cache.limit == limit && g_rs_cache.w_max == a->w_max) {
                a->rs = g_rs_cache.rs;
                g_rs_cache = RankSetCache();
            }
        }
        if (!a->rs.key) {
            WR_CUDA(cudaMalloc(&a->rs.key, R * sizeof(unsigned long long)));
            WR_CUDA(cudaMalloc(&a->rs.rows, R * kRsRowWords * sizeof(uint32_t)));
            WR_CUDA(cudaMemsetAsync(a->rs.key, 0, R * sizeof(unsigned long long), s));
            WR_CUDA(cudaMemsetAsync(a->rs.rows, 0, R * kRsRowWords * sizeof(uint32_t), s));
            WR_CUDA(cudaMalloc(&a->rs.list, ((size_t)limit + 1) * sizeof(uint32_t)));
            WR_CUDA(cudaMalloc(&a->rs.touched, ((size_t)limit + 1) * sizeof(uint32_t)));
            WR_CUDA(cudaMalloc(&a->rs.count, 8 * sizeof(uint32_t)));
            WR_CUDA(cudaMalloc(&a->rs.vtab, (size_t)2 * (a->w_max + 1) * sizeof(float)));
        }
        WR_CUDA(cudaMemsetAsync(a->rs.count, 0, 8 * sizeof(uint32_t), s));
        a->rs_entries = R;
        a->rs.rmask = (uint32_t)(R - 1); a->rs.shift = 32 - log2R; a->rs.limit = limit;
        a->rs_groups = (a->w_max + kRsGroupRanks - 1) / kRsGroupRanks;
        if (!a->rs_ev[0]) {
            int rc = feedback_acquire(&a->h_feedback, &a->d_feedback);
            if (rc != WR_OK) return rc;
            for (cudaEvent_t& e : a->rs_ev) WR_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        a->rankset = a->h_feedback != nullptr || a->rs_policy == 1;
    }
    st = sort_plan_create(&a->sort_recs, rec_max, a->stream);   // the record list and its slot sort
    if (st != WR_OK) return st;
    a->alloc_colony = cm;
    return WR_OK;
}

static bool evap_overlap()
{
    static const bool on = [] { const char* e = getenv("WR_EVAP_OVERLAP"); return !e || atoi(e) != 0; }();
    return on;
}
static int preload_iteration_kernels();
static bool batch_enabled()
{
    static const bool on = [] { const char* e = getenv("WR_BATCH"); return !e || atoi(e) != 0; }();
    return on;
}
static int walk_prefetch()
{
    static const int env = [] { const char* e = getenv("WR_WALK_PREFETCH"); return e ? atoi(e) : -1; }();   // -1: chosen per iteration (launch_walk)
    return env;
}
static int stream_cs()
{
    static const int env = [] { const char* e = getenv("WR_STREAM_CS"); return e ? atoi(e) : 1; }();   // evict-first streaming of the tiles without deposits (default on)
    return env;
}
static int walk_warm()
{
    // The L2 warm-up of the rows under the last deposits (k_path_warm / k_rankset_warm) paid in round 1, when every step's gather
    // was a demand load; with the gathers predicted a trip ahead (converged colony) or prefetched a step ahead (wandering colony)
    // it no longer does: off, value 7.42 -> 7.46e9, converged iteration 0.3185 -> 0.3154 ms, e2e 3.27 -> 3.31e9.  WR_WALK_WARM=1 restores it.
    static const int env = [] { const char* e = getenv("WR_WALK_WARM"); return e ? atoi(e) : 0; }();
    return env;
}
static size_t walk_smem(const wr_acs* a)
{
    if (a->K == kK26) return ((size_t)kWalk26Ants << a->table_log2) * 12 + kWalk26pExtra;   // + k_walk26p's move table and exchange rows
    return kWalk2Lut + 128 + (size_t)kAntsPerCta * a->table_entries * sizeof(unsigned long long);
}

static void free_batch(wr_acs* a);
extern "C" const char* wr_last_error(void) { return g_err.c_str(); }
extern "C" int wr_version(void) { return 100; }
extern "C" int wr_device_count(int* count)
{
    WR_REQUIRE(count, WR_ERR_INVALID, "wr_device_count: null");
    *count = 0;
    WR_CUDA(cudaGetDeviceCount(count));
    return WR_OK;
}
extern "C" int wr_set_device(int device)
{
    WR_CUDA(cudaSetDevice(device));
    return WR_OK;
}

extern "C" int wr_release_caches(void)
{   // buffers parked between handles (rank-set table, peer slab, IPC mappings of the peers' slabs); call with no search in flight
    std::lock_guard<std::mutex> lock(g_rs_cache_mu);
    if (g_rs_cache.rs.key) { rankset_release_buffers(g_rs_cache.rs, nullptr); g_rs_cache = RankSetCache(); }
    if (g_slab_cache.ptr) { cudaFree(g_slab_cache.ptr); g_slab_cache = SlabCache(); }
    for (IpcMapping& m : g_ipc_maps) if (m.ptr) { cudaIpcCloseMemHandle(m.ptr); m.ptr = nullptr; }
    comm_release();
    return WR_OK;
}

extern "C" int wr_acs_default_params(wr_acs_params* p)
{
    WR_REQUIRE(p, WR_ERR_INVALID, "wr_acs_default_params: null");
    p->alpha = 1; p->beta = 0.6; p->rho = 0.8; p->tau0 = 1;   // ACSRank_3D.hpp:319-324
    p->fixed_colony = 0; p->step_cap = 0; p->K = 6; p->seed = 0;
    p->update_mode = WR_UPDATE_RANKSET; p->walk_table_log2 = 0;   // adaptive deposit path; runs as WR_UPDATE_FUSED where rank sets do not apply
    return WR_OK;
}

extern "C" int wr_acs_destroy(wr_acs* a)
{
    if (!a) return WR_OK;
    if (a->stream) cudaStreamSynchronize(a->stream);
    free_batch(a);
    free_colony_buffers(a);
    cudaStream_t s = a->stream;
    pool_free(a->d_tau, s); pool_free(a->d_heur, s); pool_free(a->d_state, s); pool_free(a->d_onbest, s); pool_free(a->d_Ltab, s);
    pool_free(a->d_best_n, s); pool_free(a->d_best_ids, s); pool_free(a->d_best_dirs, s); pool_free(a->d_tile_off, s); pool_free(a->d_dep_list, s);
    pool_free(a->d_upd_q, s); pool_free(a->d_dirty, s);
    if (a->stream) cudaStreamSynchronize(a->stream);
    feedback_release(a->h_feedback);
    for (cudaEvent_t e : a->sk_ev) cudaEventDestroy(e);
    for (cudaEvent_t e : a->rs_ev) if (e) cudaEventDestroy(e);
    if (a->side) {
        cudaStreamSynchronize(a->side);
        std::lock_guard<std::mutex> lock(g_rs_cache_mu);
        for (SideStream& ss : g_side_streams) if (ss.stream == a->side) ss.in_use = false;
    }
    if (a->own_stream && a->stream) cudaStreamDestroy(a->stream);
    delete a;
    return WR_OK;
}

// initFromGridMap, ACSRank_3D.hpp:317-410: the 6-slot adjacency in order [-z,-y,-x,+x,+y,+z],
// every in-bounds slot at tau0, out-of-bounds slots at 0.  The node cuboid itself is never
// materialised: coordinates and neighbours are recomputed from indices.
extern "C" int wr_acs_create(wr_grid* g, const wr_acs_params* p, wr_acs** out)
{
    WR_REQUIRE(g && p && out, WR_ERR_INVALID, "wr_acs_create: null");
    *out = nullptr;
    WR_REQUIRE(p->K == 6 || p->K == kK26, WR_ERR_INVALID, "wr_acs_create: K must be 6 (the reference's neighbourhood) or 26 (its disabled extension)");
    WR_REQUIRE(p->alpha >= 0 && p->alpha < 64, WR_ERR_INVALID, "wr_acs_create: alpha out of range");
    WR_REQUIRE(p->update_mode >= WR_UPDATE_FUSED && p->update_mode <= WR_UPDATE_RANKSET && p->update_mode != 3, WR_ERR_INVALID, "wr_acs_create: bad update_mode");
    WR_REQUIRE(p->K != 6 || (g->rx <= 1024 && g->ry <= 1024 && g->rz <= 1024), WR_ERR_INVALID,
               "wr_acs_create: a grid axis exceeds 1024 nodes (k_walk2 packs node coordinates into 10 bits per axis)");
    WR_REQUIRE((unsigned long long)g->N * p->K < 0xFFFFFFFFull - kUpdTile, WR_ERR_INVALID, "wr_acs_create: grid too large for 32-bit slot ids");
    WR_REQUIRE(g->N >= 2, WR_ERR_INVALID, "wr_acs_create: grid too small");
    // every kernel an iteration can launch is loaded now, once per device: CUDA loads kernels lazily at their first launch, which
    // would otherwise land in the middle of a search (the rank-set kernels and the graph first run when the colony has converged)
    { WR_CUDA(cudaSetDevice(g->device)); int rc = preload_iteration_kernels(); if (rc != WR_OK) return rc; }
    wr_acs* a = new wr_acs();
    a->g = g; a->p = *p; a->N = g->N;
    if (p->update_mode == WR_UPDATE_RANKSET) {   // the record path it alternates with (and falls back to) is FUSED
        a->want_rankset = true; a->p.update_mode = WR_UPDATE_FUSED;
        if (const char* e = getenv("WR_RANKSET_POLICY")) a->rs_policy = atoi(e);
        if (const char* e = getenv("WR_RANKSET_ON")) a->rs_on = (unsigned)atoi(e);
        if (const char* e = getenv("WR_RANKSET_OFF")) a->rs_off = (unsigned)atoi(e);
    }
    if (const char* e = getenv("WR_PEER_TIMEOUT_MS")) a->barrier_timeout_ns = (unsigned long long)std::max(1, atoi(e)) * 1000000ull;
    a->K = p->K;
    a->n_slots = g->N * (size_t)p->K;
    a->n_slots_pad = (a->n_slots + kUpdTile - 1) / kUpdTile * kUpdTile;
    a->ntiles = (unsigned)(a->n_slots_pad / kUpdTile);
    a->slot_bits = ceil_log2(a->n_slots);
    a->cap = p->step_cap > 0 ? p->step_cap : (int)std::min<size_t>(g->N - 1, 65532);
    a->rank_bits = a->K == kK26 ? 31 : ceil_log2((unsigned long long)a->cap + 2);   // K = 26 ranks by the bits of L (<= +inf = 0x7F800000)
    a->table_log2 = p->walk_table_log2 > 0 ? p->walk_table_log2 : 9;
    a->table_entries = p->walk_table_log2 > 0 ? (1 << p->walk_table_log2) : 768;
    if (a->table_log2 < 4 || a->table_log2 > 10) { delete a; set_error("wr_acs_create: walk_table_log2 must be in [4,10]"); return WR_ERR_INVALID; }
#define WR_CUDA_A(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { set_error("%s failed: %s", #expr, cudaGetErrorString(_e)); wr_acs_destroy(a); return WR_ERR_CUDA; } } while (0)
    WR_CUDA_A(cudaGetDevice(&a->device));
    WR_CUDA_A(cudaStreamCreateWithFlags(&a->stream, cudaStreamNonBlocking));
    a->own_stream = true;
    WR_CUDA_A(dmalloc(&a->d_tau, a->n_slots_pad * sizeof(float), a->stream));
    if (a->n_slots_pad > a->n_slots)   // the slots themselves are written by k_tau_init below; only the padding of the last tile needs zeros
        WR_CUDA_A(cudaMemsetAsync(a->d_tau + a->n_slots, 0, (a->n_slots_pad - a->n_slots) * sizeof(float), a->stream));
    // clean-tile field for the modes whose kernels know the sentinel (FUSED and the adaptive RANKSET); WR_LAZY_TAU=0 materialises it
    {
        const char* e = getenv("WR_LAZY_TAU");
        a->lazy = a->p.update_mode == WR_UPDATE_FUSED && !(e && atoi(e) == 0);
    }
    WR_CUDA_A(dmalloc(&a->d_dirty, (size_t)a->ntiles + 1, a->stream));
    WR_CUDA_A(cudaMemsetAsync(a->d_dirty, a->lazy ? 0 : 1, (size_t)a->ntiles + 1, a->stream));
    {
        const float init_val = a->lazy ? -0.0f : p->tau0;   // -0.0f: the sentinel (kSentinelBits)
        if (a->K == kK26) k_tau_init26<<<(unsigned)((a->n_slots + 255) / 256), 256, 0, a->stream>>>(a->d_tau, g->rx, g->ry, g->rz, a->N, init_val);
        else k_tau_init<<<(unsigned)((a->N + 255) / 256), 256, 0, a->stream>>>(a->d_tau, g->rx, g->ry, g->rz, a->N, init_val);
    }
    WR_CUDA_A(cudaGetLastError());
    WR_CUDA_A(dmalloc(&a->d_state, sizeof(IterState), a->stream));
    WR_CUDA_A(cudaMemsetAsync(a->d_state, 0, sizeof(IterState), a->stream));
    k_begin<<<1, 1, 0, a->stream>>>(a->d_state, 0.0f);
    k_set_base<<<1, 1, 0, a->stream>>>(a->d_state, p->tau0);
    WR_CUDA_A(dmalloc(&a->d_onbest, (a->N / 32 + 2) * sizeof(uint32_t), a->stream));
    WR_CUDA_A(cudaMemsetAsync(a->d_onbest, 0, (a->N / 32 + 2) * sizeof(uint32_t), a->stream));
    // L after s steps: precision added s times in float (Agent::addNextNode :78)
    a->h_Ltab.resize((size_t)a->cap + 2);
    { float L = 0; a->h_Ltab[0] = 0; for (int s = 1; s <= a->cap + 1; s++) { L += g->precision; a->h_Ltab[s] = L; } }
    a->h_Ltab.push_back(kClosedSlot);   // + the marker k_walk2's idle lanes read (not part of the table)
    WR_CUDA_A(dmalloc(&a->d_Ltab, a->h_Ltab.size() * sizeof(float), a->stream));
    WR_CUDA_A(cudaMemcpyAsync(a->d_Ltab, a->h_Ltab.data(), a->h_Ltab.size() * sizeof(float), cudaMemcpyHostToDevice, a->stream));
    a->h_Ltab.pop_back();
    WR_CUDA_A(dmalloc(&a->d_best_n, sizeof(int), a->stream));
    WR_CUDA_A(cudaMemsetAsync(a->d_best_n, 0, sizeof(int), a->stream));
    WR_CUDA_A(dmalloc(&a->d_best_ids, ((size_t)a->cap + 16) * sizeof(uint32_t), a->stream));   // k_walk3 reads ids up to 7 positions past the walk: every entry must be a node id
    WR_CUDA_A(cudaMemsetAsync(a->d_best_ids, 0, ((size_t)a->cap + 16) * sizeof(uint32_t), a->stream));
    WR_CUDA_A(dmalloc(&a->d_best_dirs, (size_t)a->cap + 2, a->stream));
    WR_CUDA_A(dmalloc(&a->d_tile_off, ((size_t)a->ntiles + 2) * sizeof(uint32_t), a->stream));
    WR_CUDA_A(dmalloc(&a->d_dep_list, ((size_t)a->ntiles + 2) * sizeof(uint32_t), a->stream));
    WR_CUDA_A(dmalloc(&a->d_upd_q, 4 * sizeof(uint32_t), a->stream));
    {
        WR_CUDA_A(cudaFuncSetAttribute(k_rank_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRankSmallSmem));
        WR_CUDA_A(cudaFuncSetAttribute(k_rank_chunks, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRankChunkSmem));
        WR_CUDA_A(cudaFuncSetAttribute(k_rank_merge, cudaFuncAttributeMaxDynamicSharedMemorySize, 24 * kRankChunk * (int)sizeof(uint16_t)));
        const size_t ws = walk_smem(a);
        if (ws > 227 * 1024) { set_error("wr_acs_create: walk shared memory %zu B exceeds 227 KB", ws); wr_acs_destroy(a); return WR_ERR_INVALID; }
        if (a->K == kK26) {
            WR_CUDA_A(cudaFuncSetAttribute(k_walk26<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ws));
            WR_CUDA_A(cudaFuncSetAttribute(k_walk26p, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ws));
        }
        else {
        WR_CUDA_A(cudaFuncSetAttribute(k_walk3<true, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ws));
        WR_CUDA_A(cudaFuncSetAttribute(k_walk3<true, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ws));
        WR_CUDA_A(cudaFuncSetAttribute(k_walk3<false, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ws));
        WR_CUDA_A(cudaFuncSetAttribute(k_walk3<false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ws));
        }
    }
    WR_CUDA_A(cudaStreamSynchronize(a->stream));
#undef WR_CUDA_A
    *out = a;
    return WR_OK;
}

extern "C" int wr_acs_set_stream(wr_acs* a, void* cuda_stream)
{
    WR_REQUIRE(a, WR_ERR_INVALID, "wr_acs_set_stream: null");
    WR_CUDA(cudaStreamSynchronize(a->stream));
    drop_steady_graph(a);
    if (a->own_stream) cudaStreamDestroy(a->stream);
    a->stream = (cudaStream_t)cuda_stream;
    a->own_stream = false;
    return WR_OK;
}

// setPoints, ACSRank_3D.hpp:537-565.  The reference scans every node; the per-axis test is
// separable, so the match set is a product of (tiny) per-axis index lists and "last match in
// z,y,x order" is the largest free id in it.
static int64_t snap_point(const wr_grid* g, const float p[3])
{
    const float t = 1.2 * g->precision;   // double product rounded to float, as `float t = 1.2*precision`
    std::vector<int> cx, cy, cz;
    auto wabs = [](float v) { return v > 0 ? v : -v; };
    for (int x = 0; x < g->rx; x++) if (wabs(p[0] - g->h_xs[x]) < t) cx.push_back(x);
    for (int y = 0; y < g->ry; y++) if (wabs(p[1] - g->h_ys[y]) < t) cy.push_back(y);
    for (int z = 0; z < g->rz; z++) if (wabs(p[2] - g->h_zs[z]) < t) cz.push_back(z);
    int64_t last = -1;
    for (int z : cz) for (int y : cy) for (int x : cx) {
        int64_t id = ((int64_t)z * g->ry + y) * g->rx + x;
        if (grid_is_free_host(g, (size_t)id) && id > last) last = id;
    }
    return last;
}

extern "C" int wr_acs_set_points(wr_acs* a, const float s[3], const float e[3], int64_t ids[2])
{
    WR_REQUIRE(a && s && e && ids, WR_ERR_INVALID, "wr_acs_set_points: null");
    int st = grid_ensure_host_bits(a->g);
    if (st != WR_OK) return st;
    ids[0] = snap_point(a->g, s);
    ids[1] = snap_point(a->g, e);
    a->start = ids[0]; a->goal = ids[1];
    if (ids[0] < 0 || ids[1] < 0) { set_error("route point does not snap to a free node"); return WR_ERR_NOTFOUND; }
    return WR_OK;
}

// setPoints' scan as a kernel: no host mirror of the occupancy bits, any number of points per call
extern "C" int wr_acs_snap_points(wr_acs* a, const float* pts_xyz, int npoints, int64_t* ids)
{
    WR_REQUIRE(a && pts_xyz && ids && npoints >= 0, WR_ERR_INVALID, "wr_acs_snap_points: bad argument");
    if (npoints == 0) return WR_OK;
    WR_CUDA(cudaSetDevice(a->device));
    cudaStream_t s = a->stream;
    float* d_pts = nullptr;
    long long* d_ids = nullptr;
    WR_CUDA(dmalloc(&d_pts, (size_t)npoints * 3 * sizeof(float), s));
    WR_CUDA(dmalloc(&d_ids, (size_t)npoints * sizeof(long long), s));
    WR_CUDA(cudaMemcpyAsync(d_pts, pts_xyz, (size_t)npoints * 3 * sizeof(float), cudaMemcpyHostToDevice, s));
    const float t = 1.2 * a->g->precision;   // double product rounded to float, as `float t = 1.2*precision`
    k_snap_points<<<npoints, 128, 0, s>>>(d_pts, npoints, a->g->d_coords, a->g->rx, a->g->ry, a->g->rz, t, a->g->d_bits, d_ids);
    std::vector<long long> h(npoints);
    WR_CUDA(cudaMemcpyAsync(h.data(), d_ids, (size_t)npoints * sizeof(long long), cudaMemcpyDeviceToHost, s));
    WR_CUDA(cudaStreamSynchronize(s));
    pool_free(d_pts, s); pool_free(d_ids, s);
    for (int i = 0; i < npoints; i++) ids[i] = h[i];
    return WR_OK;
}

extern "C" int wr_acs_set_endpoints(wr_acs* a, int64_t s, int64_t e)
{
    WR_REQUIRE(a, WR_ERR_INVALID, "wr_acs_set_endpoints: null");
    WR_REQUIRE(s >= 0 && e >= 0 && (size_t)s < a->N && (size_t)e < a->N, WR_ERR_INVALID, "wr_acs_set_endpoints: id out of range");
    a->start = s; a->goal = e;
    return WR_OK;
}

extern "C" int wr_acs_peer_export(wr_acs* a, void* ipc_handle, void** raw_pointer);
extern "C" int wr_acs_peer_import(wr_acs* a, const void* all_ipc_handles);
extern "C" int wr_acs_set_shard(wr_acs* a, int rank, int nranks);

// wr_acs_begin of a handle that owns a communicator: all_gather of the slabs' CUDA IPC handles over NCCL
static int exchange_slabs(wr_acs* a)
{
    unsigned char mine[64];
    int rc = wr_acs_peer_export(a, mine, nullptr);
    if (rc != WR_OK) return rc;
    cudaStream_t s = a->stream;
    unsigned char* d_buf = nullptr;
    WR_CUDA(dmalloc(&d_buf, (size_t)64 * (a->nranks + 1), s));
    WR_CUDA(cudaMemcpyAsync(d_buf, mine, 64, cudaMemcpyHostToDevice, s));
    rc = comm_all_gather(a->comm, d_buf, d_buf + 64, 64, s);
    std::vector<unsigned char> all((size_t)64 * a->nranks);
    if (rc == WR_OK) {
        WR_CUDA(cudaMemcpyAsync(all.data(), d_buf + 64, all.size(), cudaMemcpyDeviceToHost, s));
        WR_CUDA(cudaStreamSynchronize(s));
    }
    pool_free(d_buf, s);
    if (rc != WR_OK) return rc;
    return wr_acs_peer_import(a, all.data());
}

extern "C" int wr_acs_comm_init(wr_acs* a, const void* nccl_unique_id, int rank, int nranks)
{
    WR_REQUIRE(a && nccl_unique_id, WR_ERR_INVALID, "wr_acs_comm_init: null");
    int rc = wr_acs_set_shard(a, rank, nranks);
    if (rc != WR_OK) return rc;
    a->comm = nullptr;
    if (nranks == 1) return WR_OK;
    WR_CUDA(cudaSetDevice(a->device));
    return comm_get(nccl_unique_id, rank, nranks, &a->comm);
}

extern "C" int wr_acs_set_next_search(wr_acs* a, uint32_t index)
{
    WR_REQUIRE(a, WR_ERR_INVALID, "wr_acs_set_next_search: null");
    a->next_search = index;
    return WR_OK;
}

extern "C" int wr_acs_begin(wr_acs* a, float predict)
{
    WR_REQUIRE(a, WR_ERR_INVALID, "wr_acs_begin: null");
    WR_REQUIRE(a->start >= 0 && a->goal >= 0, WR_ERR_STATE, "wr_acs_begin: endpoints not set");
    int cm = a->p.fixed_colony > 0 ? a->p.fixed_colony : (int)(0.35 * (double)predict / (double)a->g->precision);   // :247 with best = inf
    WR_REQUIRE(cm >= 0 && cm < (1 << 24), WR_ERR_INVALID, "wr_acs_begin: colony size out of range");
    WR_CUDA(cudaSetDevice(a->device));
    int st = alloc_colony_buffers(a, cm);
    if (st != WR_OK) return st;
    a->colony_max = cm;
    a->search = a->next_search++;
    if (!a->d_heur) WR_CUDA(dmalloc(&a->d_heur, a->n_slots_pad * sizeof(float), a->stream));
    if (a->heur_goal != a->goal && a->K == kK26) {
        k_heuristic26<<<(unsigned)((a->n_slots + 255) / 256), 256, 0, a->stream>>>(a->d_heur, a->g->d_coords, a->g->d_bits, a->g->rx, a->g->ry, a->g->rz, a->N,
                                                                                  (int)a->goal, a->p.beta);
        a->heur_goal = a->goal;
    } else if (a->heur_goal != a->goal) {   // selectNext's geometric factor, tabulated once per goal
        k_heuristic<<<(unsigned)((a->N + 255) / 256), 256, 0, a->stream>>>(a->d_heur, a->g->d_coords, a->g->d_bits, a->g->rx, a->g->ry, a->g->rz, a->N, (int)a->goal,
                                                                            a->p.beta);
        a->heur_goal = a->goal;
    }
    k_begin<<<1, 1, 0, a->stream>>>(a->d_state, predict);
    WR_CUDA(cudaGetLastError());
    a->rs_generation = (a->rs_generation + 1) & 0xFFFFu; a->rs_choice = 0; a->rs_enqueued = 0;
    drop_steady_graph(a);   // endpoints, heuristic table and generation are baked into the captured launches
    a->sk_used = 0; a->sk_ms = 0; a->sk_launches = 0;
    a->peers_set = false;   // sharded: the barrier epochs restart with the iteration counter, so the slabs are exchanged (and their flag words zeroed) per search
    a->begun = true;
    a->timer.used = 0;
    for (float& m : a->timer.ms) m = 0;
    if (a->nranks > 1 && a->comm) return exchange_slabs(a);   // without a communicator the caller exchanges them (wr_acs_peer_export / _import)
    return WR_OK;
}

// before k_iter_begin: pull the rows under last iteration's deposits into L2 (see k_path_warm)
static void launch_warm(wr_acs* a, bool prev_rankset)
{
    if (!walk_warm() || a->p.update_mode == WR_UPDATE_ATOMIC || a->K != 6) return;
    if (a->rankset && a->rs_enqueued > 0 && prev_rankset) {   // the previous iteration's deposits went through rank sets
        k_rankset_warm<<<kNumSMs, 256, 0, a->stream>>>(a->rs.touched, a->rs.count, a->d_tau, a->d_heur, a->d_state);
        return;
    }
    if (a->warm_by_pull) return;   // owner-computes update: k_pull_finals has just touched the rows under the deposits
    const uint32_t* ck = a->recs_in_b ? a->sort_recs.keys_b : a->sort_recs.keys_a;
    k_path_warm<<<kNumSMs, 256, 0, a->stream>>>(a->d_state, ck, a->d_tau, a->d_heur);
}

static int launch_walk(wr_acs* a)
{
    const wr_grid* g = a->g;
    WalkArgs w;
    w.st = a->d_state; w.tau = a->d_tau; w.heur = a->d_heur; w.coords = g->d_coords;
    w.closed_marker = a->d_Ltab + a->h_Ltab.size();   // one float behind the length table
    w.rx = g->rx; w.ry = g->ry; w.rz = g->rz;
    w.start = (int)a->start; w.goal = (int)a->goal;
    w.seed_lo = (uint32_t)a->p.seed; w.seed_hi = (uint32_t)(a->p.seed >> 32);
    w.stream_word = kStreamAcs3D + (a->search & 0xFFFFu); w.block_hi = (a->search >> 16) << 16;
    w.alpha = a->p.alpha; w.beta = a->p.beta; w.cap = a->cap;
    w.shard_first = a->rank * a->chunk; w.shard_chunk = a->chunk;
    w.ant_steps = a->d_local_steps;
    w.path_ids = a->d_path_ids; w.path_dirs = a->d_path_dirs;
    w.table_log2 = a->table_log2; w.table_entries = a->table_entries; w.overflow_list = a->d_overflow;
    w.gkeys = a->d_gkeys; w.gmasks = a->d_gmasks; w.gtab = a->d_gmasks; w.gtable_log2 = a->gtable_log2; w.resume = a->d_resume;
    w.precision = g->precision; w.ant_L = a->d_ant_L; w.best_ids = a->d_best_ids;
    if (a->K == kK26) {
        const size_t smem = walk_smem(a);
        const int per_sm = std::max(1, std::min((int)((227 * 1024) / (smem + 1024)), 16));
        const int blocks = std::max(1, std::min((a->chunk + kWalk26Ants - 1) / kWalk26Ants, kNumSMs * per_sm));
        if (g->rx <= 1024 && g->ry <= 1024 && g->rz <= 1024) k_walk26p<<<blocks, kWalk26Threads, smem, a->stream>>>(w);
        else k_walk26<false><<<blocks, kWalk26Threads, smem, a->stream>>>(w);
        w.table_log2 = a->gtable_log2;
        k_walk26<true><<<std::max(1, std::min((a->chunk + kWalk26Ants - 1) / kWalk26Ants, kNumSMs * 4)), kWalk26Threads, 0, a->stream>>>(w);
        WR_CUDA(cudaGetLastError());
        return WR_OK;
    }
    const size_t smem1 = walk_smem(a);
    const int per_sm = std::max(1, (int)((227 * 1024) / (smem1 + 1024)));
    const int blocks1 = std::max(1, std::min((a->chunk + kAntsPerCta - 1) / kAntsPerCta, kNumSMs * std::min(per_sm, 16)));
    const bool alpha1 = a->p.alpha == 1;
    // L1 prefetch of the six neighbour rows pays while the colony wanders (rows come from L2/HBM); once its deposits are
    // concentrated — the same device feedback that selects the rank-set path — the rows are hot and the twelve prefetch
    // instructions per step are pure issue cost (converged walk 0.346 -> 0.317 ms without them)
    int pf = walk_prefetch();
    if (pf < 0) pf = (a->rankset && a->rs_choice) ? 0 : 2;
    if (!alpha1 && pf) k_walk3<false, 1><<<blocks1, kWalkThreads, smem1, a->stream>>>(w);
    else if (!alpha1) k_walk3<false, 0><<<blocks1, kWalkThreads, smem1, a->stream>>>(w);
    else if (pf) k_walk3<true, 1><<<blocks1, kWalkThreads, smem1, a->stream>>>(w);
    else k_walk3<true, 0><<<blocks1, kWalkThreads, smem1, a->stream>>>(w);
    // pass 2: resume the ants that parked on a full shared-memory table (usually none: the kernel exits at once)
    w.table_log2 = a->gtable_log2;
    if (alpha1) k_walk2<true><<<a->walk2_blocks, kWalkThreads, kWalk2Lut, a->stream>>>(w);
    else k_walk2<false><<<a->walk2_blocks, kWalkThreads, kWalk2Lut, a->stream>>>(w);
    WR_CUDA(cudaGetLastError());
    return WR_OK;
}

static const uint32_t* rank_keys(const wr_acs* a) { return a->ants_in_b ? a->sort_ants.keys_b : a->sort_ants.keys_a; }
static const uint32_t* rank_vals(const wr_acs* a) { return a->ants_in_b ? a->sort_ants.vals_b : a->sort_ants.vals_a; }

// colony ranking (:273-274), best decision (:263-264), deposit eligibility and offsets (:200): rank_small.cuh
static int launch_rank(wr_acs* a, const int* d_all_steps)
{
    const int cm = std::max(a->colony_max, 1);
    cudaStream_t s = a->stream;
    const float* d_L = a->K == kK26 ? a->d_ant_L : nullptr;
    a->ants_in_b = false;
    if (cm <= 2 * kRankChunk) {   // the whole ranking in one single-CTA kernel
        k_rank_small<<<1, kRankSmallThreads, kRankSmallSmem, s>>>(a->d_state, d_all_steps, d_L, a->cap, a->rank_bits, a->d_Ltab, a->sort_ants.keys_a, a->sort_ants.vals_a,
                                                                   a->d_rec_off, a->d_order, a->d_best_n, a->d_best_ids, a->d_onbest);
    } else {                     // chunks of 4096 ants sorted in parallel, merged by rank counting, prefix-only finish
        const int nchunks = (cm + kRankChunk - 1) / kRankChunk;
        k_rank_chunks<<<nchunks, kRankSmallThreads, kRankChunkSmem, s>>>(a->d_state, d_all_steps, d_L, a->cap, a->rank_bits, a->sort_ants.keys_b, a->sort_ants.vals_b);
        const int stage = std::min(nchunks, 24);
        // 16-bit staged keys hold K = 6 step counts up to cap + 1 (a dead ant) while that fits: the automatic cap (<= 65532)
        // always does, an explicit step_cap of 65535 or more does not.  Those, and K = 26 (bits of L), compare in global memory.
        const int keys16 = a->K == 6 && (long long)a->cap + 1 <= 0xFFFF;
        k_rank_merge<<<(cm + kRankMergeThreads - 1) / kRankMergeThreads, kRankMergeThreads, (size_t)stage * kRankChunk * sizeof(uint16_t), s>>>(
            a->d_state, a->sort_ants.keys_b, a->sort_ants.vals_b, a->sort_ants.keys_a, a->sort_ants.vals_a, a->d_order, keys16);
        k_rank_finish_prefix<<<1, 1024, 0, s>>>(a->d_state, a->sort_ants.keys_a, a->sort_ants.vals_a, a->cap, a->d_Ltab, a->d_rec_off, a->w_max,
                                                a->K == kK26 ? d_all_steps : nullptr, a->d_best_n, a->d_best_ids, a->d_onbest);
    }
    WR_CUDA(cudaGetLastError());
    return WR_OK;
}

// deposit records of this rank's ants (:198-215), at their global (rank, step) positions
static int launch_deposit_gen(wr_acs* a)
{
    cudaStream_t s = a->stream;
    const int first = a->rank * a->chunk;
    if (a->p.update_mode == WR_UPDATE_ATOMIC) {
        k_evaporate<<<kNumSMs * 8, 256, 0, s>>>(reinterpret_cast<float4*>(a->d_tau), a->n_slots_pad / 4, a->p.rho);
        k_deposit_gen<true><<<a->w_max, 128, 0, s>>>(a->d_state, rank_keys(a), rank_vals(a), a->d_rec_off, a->d_path_ids, a->d_path_dirs, a->cap,
                                                     first, a->chunk, (int)a->goal, a->d_Ltab, a->d_onbest, nullptr, nullptr, a->d_tau, nullptr, nullptr, a->K,
                                                     a->K == kK26 ? a->d_ant_steps : nullptr);
    } else {
        k_deposit_gen<false><<<a->w_max, 128, 0, s>>>(a->d_state, rank_keys(a), rank_vals(a), a->d_rec_off, a->d_path_ids, a->d_path_dirs, a->cap,
                                                      first, a->chunk, (int)a->goal, a->d_Ltab, a->d_onbest, a->sort_recs.keys_a,
                                                      a->sort_recs.vals_a, nullptr, nullptr, nullptr, a->K, a->K == kK26 ? a->d_ant_steps : nullptr);
    }
    WR_CUDA(cudaGetLastError());
    return WR_OK;
}

// K3, shipped variant: tile offsets + list of deposit tiles, then the fused single-pass update
static int launch_fused(wr_acs* a, const uint32_t* ck, const uint32_t* cv, const int* d_n = nullptr, uint32_t* fin = nullptr)
{
    cudaStream_t s = a->stream;
    if (!a->upd_q_zeroed) WR_CUDA(cudaMemsetAsync(a->d_upd_q, 0, 4 * sizeof(uint32_t), s));
    a->upd_q_zeroed = false;
    k_tile_offsets<<<(a->ntiles + 1 + 255) / 256, 256, 0, s>>>(d_n ? d_n : a->dptr_nrec(), ck, a->d_tile_off, a->ntiles, a->d_dep_list, a->d_upd_q + 2);
    if (a->timer.enabled) cudaEventRecord(a->sk_next(), s);
    if (fin) k_update_fused<true><<<kNumSMs * kFusedCtasPerSm, kUpdThreads, 0, s>>>(a->d_tau, a->ntiles, a->p.rho, ck, cv, a->d_tile_off, a->d_dep_list, a->d_upd_q, fin, stream_cs(),
                                                                                      a->d_state, a->d_dirty);
    else k_update_fused<false><<<kNumSMs * kFusedCtasPerSm, kUpdThreads, 0, s>>>(a->d_tau, a->ntiles, a->p.rho, ck, cv, a->d_tile_off, a->d_dep_list, a->d_upd_q, nullptr, stream_cs(),
                                                                                 a->d_state, a->d_dirty);
    if (a->timer.enabled) cudaEventRecord(a->sk_next(), s);
    WR_CUDA(cudaGetLastError());
    return WR_OK;
}

// slot sort (stable: rank order survives inside a slot) + evaporation + deposits (:268-280)
static int launch_update(wr_acs* a)
{
    cudaStream_t s = a->stream;
    if (a->p.update_mode == WR_UPDATE_ATOMIC) {
        if (a->timer.enabled) cudaEventRecord(a->timer.next(), s);
        return WR_OK;   // evaporation + atomic deposits already issued by launch_deposit_gen
    }
    int st = sort_pairs(&a->sort_recs, a->dptr_nrec_upd(), a->slot_bits, s, &a->recs_in_b);
    if (st != WR_OK) return st;
    const uint32_t* ck = a->recs_in_b ? a->sort_recs.keys_b : a->sort_recs.keys_a;
    const uint32_t* cv = a->recs_in_b ? a->sort_recs.vals_b : a->sort_recs.vals_a;
    if (a->timer.enabled) cudaEventRecord(a->timer.next(), s);
    if (a->p.update_mode == WR_UPDATE_FUSED) {
        int rc = launch_fused(a, ck, cv, a->dptr_nrec_upd());
        if (rc != WR_OK) return rc;
    } else {
        k_evaporate<<<kNumSMs * 8, 256, 0, s>>>(reinterpret_cast<float4*>(a->d_tau), a->n_slots_pad / 4, a->p.rho);
        k_deposit_apply<<<kNumSMs * 4, 256, 0, s>>>(a->d_state, ck, cv, a->d_tau);
    }
    WR_CUDA(cudaGetLastError());
    return WR_OK;
}

// ---- peer barrier of a sharded colony (acs_kernels.cuh: peer_barrier, executed inside the kernel that reads peer data) ----
// Grid of a kernel that contains a peer barrier.  Its CTAs spin until every rank has signalled, and a rank signals from the first
// CTAs of the same kernel.  With one process per GPU the spinning CTAs own their GPU.  Shards of ONE process share a GPU: a grid
// that fills the SMs' thread or register slots while it spins keeps the other shards' kernels — the ones it waits for — from
// being scheduled at all (seen as barrier timeouts in 1-3 % of the one-GPU test cases, e.g. two spinning k_rankset_merge CTAs per
// SM leave no room for another shard's 1024-thread k_rank_small).  Such handles spin with a handful of CTAs.
static int barrier_grid(const wr_acs* a, int blocks) { return a->in_process_peers ? std::min(blocks, 16) : blocks; }

static PeerBarrier barrier_args(const wr_acs* a)
{
    PeerBarrier b;
    b.flags_tab = reinterpret_cast<uint32_t* const*>(const_cast<void**>(a->tab(5, 0)));
    b.me = a->rank; b.nranks = a->nranks; b.err = a->d_peer_err; b.timeout_ns = a->barrier_timeout_ns;
    return b;
}

// ---- the rank-set deposit path (rankset.cuh): build [+ publish | barrier | merge], evaporate, one apply launch per rank group ----
static int launch_rankset_update(wr_acs* a)
{
    cudaStream_t s = a->stream;
    const int first = a->rank * a->chunk;
    k_rankset_gen<<<a->w_max, 128, 0, s>>>(a->d_state, rank_keys(a), rank_vals(a), a->d_path_ids, a->d_path_dirs, a->cap, (int)a->goal, a->d_Ltab, a->d_onbest,
                                           a->rs, a->K, a->K == kK26 ? a->d_ant_steps : nullptr, first, a->chunk);
    if (a->nranks > 1) {
        k_rankset_publish<<<kNumSMs, 256, 0, s>>>(a->d_state, a->rs, a->pub_buf());
        k_rankset_merge<<<barrier_grid(a, kNumSMs * 2), 256, 0, s>>>(barrier_args(a), a->d_state, a->rs, reinterpret_cast<const uint32_t* const*>(a->tab(4, 0)), a->nranks, a->rank);
    }
    if (a->timer.enabled) cudaEventRecord(a->timer.next(), s);
    if (a->evap_forked) {
        WR_CUDA(cudaStreamWaitEvent(s, a->ev_join, 0));
        a->evap_forked = false;
    } else {
        if (a->timer.enabled) cudaEventRecord(a->sk_next(), s);
        k_evaporate_tiles<<<kNumSMs * 8, 256, 0, s>>>(reinterpret_cast<float4*>(a->d_tau), a->ntiles, a->p.rho, a->d_dirty, stream_cs());
        if (a->timer.enabled) cudaEventRecord(a->sk_next(), s);
    }
    // ordered chains (all rank groups in one launch), wipe; on overflow of the fixed-capacity table (flag raised by gen / merge)
    // the chains are skipped, the whole table is swept and k_deposit_serial applies the deposits in the reference's own loop order
    k_rankset_apply<<<kNumSMs * 4, 256, 0, s>>>(a->d_state, a->d_tau, a->rs, a->p.rho, a->d_dirty, a->rs_groups);
    if (a->rs_groups > 1) k_rankset_clear<<<kNumSMs * 2, 256, 0, s>>>(a->d_state, a->rs);
    k_deposit_serial<<<1, 1024, 0, s>>>(a->d_state, rank_keys(a), rank_vals(a), a->trail_ids_tab(), a->trail_dirs_tab(), a->cap, a->chunk, (int)a->goal, a->d_Ltab,
                                        a->d_onbest, a->rs.count + 3, a->d_tau, a->p.rho, a->d_dirty, a->K, a->K == kK26 ? a->d_ant_steps : nullptr);
    WR_CUDA(cudaGetLastError());
    return WR_OK;
}

// ---- the sorted-record deposit path of a sharded colony: every rank generates the records of ALL eligible ants from their
//      owners' trails (peer loads), keeps, sorts and applies its slot slice, lists the final values; barrier; pull ----
static int launch_record_update_sharded(wr_acs* a)
{
    cudaStream_t s = a->stream;
    k_deposit_gen<false, true><<<a->w_max, 128, 0, s>>>(a->d_state, rank_keys(a), rank_vals(a), a->d_rec_off, nullptr, nullptr, a->cap, 0, a->chunk,
                                                         (int)a->goal, a->d_Ltab, a->d_onbest, a->sort_recs.keys_a, a->sort_recs.vals_a, nullptr,
                                                         a->trail_ids_tab(), a->trail_dirs_tab());
    WR_CUDA(cudaGetLastError());
    const unsigned t_lo = (unsigned)(((unsigned long long)a->ntiles * a->rank) / a->nranks);
    const unsigned t_hi = (unsigned)(((unsigned long long)a->ntiles * (a->rank + 1)) / a->nranks);
    int st = sort_partition(&a->sort_recs, a->dptr_nrec_upd(), t_lo * (uint32_t)kUpdTile, (t_hi - t_lo) * (uint32_t)kUpdTile, s, a->d_nq);
    if (st != WR_OK) return st;
    st = sort_pairs(&a->sort_recs, a->d_nq, a->slot_bits, s, &a->recs_in_b, true);
    if (st != WR_OK) return st;
    const uint32_t* ck = a->recs_in_b ? a->sort_recs.keys_b : a->sort_recs.keys_a;
    const uint32_t* cv = a->recs_in_b ? a->sort_recs.vals_b : a->sort_recs.vals_a;
    if (a->timer.enabled) cudaEventRecord(a->timer.next(), s);
    uint32_t* fin = a->fin_buf(a->parity);
    WR_CUDA(cudaMemsetAsync(fin, 0, 4 * sizeof(uint32_t), s));
    st = launch_fused(a, ck, cv, a->d_nq, fin);
    if (st != WR_OK) return st;
    k_pull_finals<<<barrier_grid(a, kNumSMs * 2), 256, 0, s>>>(barrier_args(a), a->d_state, a->d_tau, walk_warm() ? a->d_heur : nullptr,
                                              reinterpret_cast<const uint32_t* const*>(a->tab(2, a->parity)), a->nranks, a->rank, a->d_dirty, a->d_upd_q);
    WR_CUDA(cudaGetLastError());
    return WR_OK;
}

static bool graph_enabled()
{
    static const bool on = [] { const char* e = getenv("WR_GRAPH"); return !e || atoi(e) != 0; }();
    return on;
}

// Everything of one iteration between the iteration parameters and the deposits: construction, [exchange of the step counts],
// ranking, best path.
static int launch_construct_and_rank(wr_acs* a, bool rankset_iteration)
{
    cudaStream_t s = a->stream;
    if (a->nranks > 1) WR_CUDA(cudaMemsetAsync(a->d_local_steps, 0xFF, (size_t)a->chunk * sizeof(int), s));   // -1: beyond the colony
    int st = launch_walk(a);
    if (st != WR_OK) return st;
    if (a->timer.enabled) cudaEventRecord(a->timer.next(), s);
    a->evap_forked = false;
    if (a->nranks > 1 && rankset_iteration && evap_overlap() && !a->in_process_peers) {
        // The walk was the last reader of the field: its evaporation (:268-272) can start now, on a side stream, while this
        // stream waits for the peers, ranks the colony and merges the rank sets; the ordered chains join it again.  (On one GPU
        // the same overlap was measured and rejected: the chain of small kernels slows down under a saturated memory system and
        // there is no barrier wait to hide behind.)
        if (!a->side) {   // parked between handles (searches created per request): creating a stream costs more than an iteration
            std::lock_guard<std::mutex> lock(g_rs_cache_mu);
            for (SideStream& ss : g_side_streams)
                if (ss.stream && !ss.in_use && ss.device == a->device) { ss.in_use = true; a->side = ss.stream; a->ev_fork = ss.fork; a->ev_join = ss.join; break; }
            if (!a->side) {
                SideStream ss;
                WR_CUDA(cudaStreamCreateWithFlags(&ss.stream, cudaStreamNonBlocking));
                WR_CUDA(cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming));
                WR_CUDA(cudaEventCreateWithFlags(&ss.join, cudaEventDisableTiming));
                ss.device = a->device; ss.in_use = true;
                g_side_streams.push_back(ss);
                a->side = ss.stream; a->ev_fork = ss.fork; a->ev_join = ss.join;
            }
        }
        WR_CUDA(cudaEventRecord(a->ev_fork, s));
        WR_CUDA(cudaStreamWaitEvent(a->side, a->ev_fork, 0));
        if (a->timer.enabled) cudaEventRecord(a->sk_next(), a->side);
        k_evaporate_tiles<<<kNumSMs * 8, 256, 0, a->side>>>(reinterpret_cast<float4*>(a->d_tau), a->ntiles, a->p.rho, a->d_dirty, stream_cs());
        if (a->timer.enabled) cudaEventRecord(a->sk_next(), a->side);
        WR_CUDA(cudaEventRecord(a->ev_join, a->side));
        a->evap_forked = true;
    }
    if (a->nranks > 1) {   // barrier (trails and step counts of every rank complete and visible), then the global colony
        const int total = a->chunk * a->nranks;
        k_gather_steps<<<barrier_grid(a, std::max(1, std::min((total + 255) / 256, kNumSMs))), 256, 0, s>>>(barrier_args(a), a->d_state, reinterpret_cast<const int* const*>(a->tab(3, a->parity)),
                                                                                             a->nranks, a->chunk, a->d_ant_steps);
    }
    st = launch_rank(a, a->d_ant_steps);
    if (st != WR_OK) return st;
    if (a->nranks > 1)
        k_best_copy_peer<<<8, 256, 0, s>>>(a->d_state, a->d_best_n, a->d_best_ids, a->d_best_dirs, a->d_onbest, a->trail_ids_tab(), a->trail_dirs_tab(), a->cap, a->chunk,
                                           (int)a->goal);
    else
        k_best_copy<<<8, 256, 0, s>>>(a->d_state, a->d_best_n, a->d_best_ids, a->d_best_dirs, a->d_onbest, a->d_path_ids, a->d_path_dirs, a->cap, 0, (int)a->goal);
    if (a->timer.enabled) cudaEventRecord(a->timer.next(), s);
    WR_CUDA(cudaGetLastError());
    return WR_OK;
}

// One rank-set iteration whose predecessor was a rank-set iteration too, captured from the very launch sequence of
// wr_acs_iterate (k_iter_end of the predecessor folded into k_iter_begin): L2 warm-up, iteration parameters, walk pass 1 + 2,
// ranking, best copy, rank-set build, evaporation of the dirty tiles, ordered chains.  Every argument is fixed for the search
// (sharded handles alternate between two trail buffers, hence one graph per parity).
static int capture_steady_iteration(wr_acs* a, cudaGraphExec_t* out)
{
    cudaStream_t s = a->stream;
    if (s == nullptr || s == cudaStreamLegacy || s == cudaStreamPerThread) return WR_ERR_STATE;   // the default streams cannot be captured
    WR_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    launch_warm(a, true);
    k_iter_begin<<<1, 1, 0, s>>>(a->d_state, a->p.fixed_colony, a->colony_max, a->g->precision, a->p.tau0, 1, a->d_upd_q, a->rs.count, 1, a->d_feedback,
                                 a->rs_generation, a->p.rho);
    int st = launch_construct_and_rank(a, true);
    if (st == WR_OK) st = launch_rankset_update(a);
    cudaGraph_t graph = nullptr;
    cudaError_t e = cudaStreamEndCapture(s, &graph);
    if (e != cudaSuccess || st != WR_OK || !graph) {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        return WR_ERR_CUDA;
    }
    e = cudaGraphInstantiate(out, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) { *out = nullptr; cudaGetLastError(); return WR_ERR_CUDA; }
    return WR_OK;
}

// Which deposit path iteration number `n` of this search takes.  Adaptive handles: the record the device published when
// iteration n - kRsAhead started (statistics of iteration n - kRsAhead - 1; that iteration has finished, its event was
// waited for) — a pure function of the search, so every rank of a sharded colony takes the same decision.
static int choose_deposit_path(wr_acs* a)
{
    const unsigned long long n = a->rs_enqueued;
    if (n >= (unsigned long long)wr_acs::kRsAhead) WR_CUDA(cudaEventSynchronize(a->rs_ev[n % wr_acs::kRsAhead]));
    if (a->rs_policy == 1 || a->rs_policy == 2) a->rs_choice = a->rs_policy == 1;
    else if (a->h_feedback && n > (unsigned long long)wr_acs::kRsAhead) {
        const unsigned long long m = n - wr_acs::kRsAhead;
        const volatile uint32_t* f = a->h_feedback + 4 * (m & 7u);
        const uint32_t tag = f[0], prev = f[1], tiles = f[2], blocks = f[3];
        if (tag == ((a->rs_generation << 16) | (uint32_t)(m & 0xFFFFu))) {
            if (!a->rs_choice && prev == 0 && tiles <= a->rs_on) a->rs_choice = 1;
            else if (a->rs_choice && prev == 1 && blocks > a->rs_off) a->rs_choice = 0;
        }
    }
    return WR_OK;
}

extern "C" int wr_acs_iterate(wr_acs* a, int n)
{
    WR_REQUIRE(a && n >= 0, WR_ERR_INVALID, "wr_acs_iterate: bad argument");
    WR_REQUIRE(a->begun, WR_ERR_STATE, "wr_acs_iterate: call wr_acs_begin first");
    WR_REQUIRE(a->nranks == 1 || a->peers_set, WR_ERR_STATE, "wr_acs_iterate: sharded handle: exchange the peer slabs first (wr_acs_comm_init, or wr_acs_peer_export / _import)");
    WR_CUDA(cudaSetDevice(a->device));
    cudaStream_t s = a->stream;
    const bool sharded = a->nranks > 1;
    if (n > 0) a->field_clean = false;
    for (int it = 0; it < n; it++) {
        if (a->timer.enabled) cudaEventRecord(a->timer.next(), s);
        const bool rs_prev = a->rankset && a->rs_choice;   // path of the previous iteration (what the L2 warm-up reads)
        if (a->rankset) { int rc = choose_deposit_path(a); if (rc != WR_OK) return rc; }
        const bool rs_now = a->rankset && a->rs_choice;
        if (sharded) {   // trails and step counts are double-buffered: a peer may still be reading the previous iteration's
            a->parity ^= 1u;
            a->d_path_ids = reinterpret_cast<uint32_t*>(a->d_slab + a->off_ids[a->parity]);
            a->d_path_dirs = a->d_slab + a->off_dirs[a->parity];
            a->d_local_steps = reinterpret_cast<int*>(a->d_slab + a->off_steps[a->parity]);
        }
        // steady state of a converged search: the whole iteration is one graph launch
        if (rs_now && rs_prev && it > 0 && a->rs_enqueued > 0 && !a->timer.enabled && !a->rs_graph_failed && !a->in_process_peers && graph_enabled()) {
            cudaGraphExec_t& gx = a->rs_graph[sharded ? a->parity : 0];
            if (!gx && capture_steady_iteration(a, &gx) != WR_OK) a->rs_graph_failed = true;
            if (gx) {
                WR_CUDA(cudaGraphLaunch(gx, s));
                WR_CUDA(cudaEventRecord(a->rs_ev[a->rs_enqueued % wr_acs::kRsAhead], s)); a->rs_enqueued++;
                if (it == n - 1) k_iter_end<<<1, 1, 0, s>>>(a->d_state, a->p.rho);
                continue;
            }
        }
        launch_warm(a, rs_prev);
        k_iter_begin<<<1, 1, 0, s>>>(a->d_state, a->p.fixed_colony, a->colony_max, a->g->precision, a->p.tau0, it > 0 ? 1 : 0, a->d_upd_q,
                                     a->rankset ? a->rs.count : nullptr, rs_now ? 1 : 0, a->d_feedback, a->rs_generation, a->p.rho);
        a->upd_q_zeroed = true;
        int st = launch_construct_and_rank(a, rs_now);
        if (st != WR_OK) return st;
        if (rs_now) st = launch_rankset_update(a);   // rank sets instead of sorted records (rankset.cuh)
        else if (sharded) { st = launch_record_update_sharded(a); a->warm_by_pull = true; }
        else {
            st = launch_deposit_gen(a);
            if (st == WR_OK) st = launch_update(a);
        }
        if (st != WR_OK) return st;
        if (rs_now) a->warm_by_pull = false;
        if (a->rankset) { WR_CUDA(cudaEventRecord(a->rs_ev[a->rs_enqueued % wr_acs::kRsAhead], s)); a->rs_enqueued++; }
        a->upd_q_zeroed = false;
        if (it == n - 1) k_iter_end<<<1, 1, 0, s>>>(a->d_state, a->p.rho);   // otherwise folded into the next k_iter_begin
        if (a->timer.enabled) cudaEventRecord(a->timer.next(), s);
    }
    WR_CUDA(cudaGetLastError());
    return WR_OK;
}

// ---- many searches on one grid: the all-pairs loop of searchBestPathOfPoints (:472-499) / independent queries ------------
// Results of the last wr_acs_search_pairs / wr_acs_search_batch stay in the handle (host memory, packed): paths are read back
// by their true length (one count read-back, one packed copy) instead of as rows of step_cap + 1 entries.
__global__ void k_pack_paths(const uint32_t* __restrict__ rows_ids, const uint8_t* __restrict__ rows_dirs, size_t row_stride, const int* __restrict__ counts,
                             const unsigned long long* __restrict__ offs, uint32_t* __restrict__ out_ids, uint8_t* __restrict__ out_dirs)
{
    const int q = blockIdx.x;
    const int n = counts[q];
    const unsigned long long o = offs[q];
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        out_ids[o + i] = rows_ids[(size_t)q * row_stride + i];
        if (i + 1 < n) out_dirs[o + i] = rows_dirs[(size_t)q * row_stride + i];
    }
}

// device rows [count][row_stride] + d_L/d_n[count] -> appended to the handle's result cache (synchronises the stream)
static int collect_results(wr_acs* a, int count, const uint32_t* d_rows_ids, const uint8_t* d_rows_dirs, size_t row_stride, const float* d_L, const int* d_n)
{
    cudaStream_t s = a->stream;
    std::vector<float> hL(count);
    std::vector<int> hn(count);
    WR_CUDA(cudaMemcpyAsync(hL.data(), d_L, (size_t)count * sizeof(float), cudaMemcpyDeviceToHost, s));
    WR_CUDA(cudaMemcpyAsync(hn.data(), d_n, (size_t)count * sizeof(int), cudaMemcpyDeviceToHost, s));
    WR_CUDA(cudaStreamSynchronize(s));
    std::vector<unsigned long long> off(count);
    unsigned long long total = 0;
    for (int q = 0; q < count; q++) { off[q] = total; total += (unsigned long long)hn[q]; }
    const size_t base = a->res_ids.size();
    a->res_ids.resize(base + total); a->res_dirs.resize(base + total);
    if (total > 0) {
        unsigned long long* d_off = nullptr; uint32_t* d_pi = nullptr; uint8_t* d_pd = nullptr;
        WR_CUDA(dmalloc(&d_off, (size_t)count * sizeof(unsigned long long), s));
        WR_CUDA(dmalloc(&d_pi, total * sizeof(uint32_t), s));
        WR_CUDA(dmalloc(&d_pd, total, s));
        WR_CUDA(cudaMemcpyAsync(d_off, off.data(), (size_t)count * sizeof(unsigned long long), cudaMemcpyHostToDevice, s));
        k_pack_paths<<<count, 256, 0, s>>>(d_rows_ids, d_rows_dirs, row_stride, d_n, d_off, d_pi, d_pd);
        WR_CUDA(cudaMemcpyAsync(a->res_ids.data() + base, d_pi, total * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        WR_CUDA(cudaMemcpyAsync(a->res_dirs.data() + base, d_pd, total, cudaMemcpyDeviceToHost, s));
        WR_CUDA(cudaStreamSynchronize(s));
        pool_free(d_off, s); pool_free(d_pi, s); pool_free(d_pd, s);
    }
    for (int q = 0; q < count; q++) { a->res_L.push_back(hL[q]); a->res_n.push_back(hn[q]); a->res_off.push_back(base + off[q]); }
    return WR_OK;
}

// the searches [first, first + count) one after the other (begin + n iterations + reset(), enqueued back to back with no host
// synchronisation), results appended to the cache
static int run_pairs_sequential(wr_acs* a, const int64_t* start_ids, const int64_t* goal_ids, int first, int count, float predict, int n_iterations)
{
    cudaStream_t s = a->stream;
    const size_t stride = (size_t)a->cap + 1;
    float* d_L = nullptr; int* d_n = nullptr; uint32_t* d_ids = nullptr; uint8_t* d_dirs = nullptr;
    WR_CUDA(dmalloc(&d_L, (size_t)count * sizeof(float), s));
    WR_CUDA(dmalloc(&d_n, (size_t)count * sizeof(int), s));
    WR_CUDA(dmalloc(&d_ids, (size_t)count * stride * sizeof(uint32_t), s));
    WR_CUDA(dmalloc(&d_dirs, (size_t)count * stride, s));
    int rc = WR_OK;
    for (int p = 0; p < count && rc == WR_OK; p++) {
        a->start = start_ids[first + p]; a->goal = goal_ids[first + p];
        rc = wr_acs_begin(a, predict);
        if (rc == WR_OK) rc = wr_acs_iterate(a, n_iterations);
        if (rc != WR_OK) break;
        k_save_result<<<4, 256, 0, s>>>(a->d_state, a->d_best_n, a->d_best_ids, a->d_best_dirs, p, (int)stride, d_L, d_n, d_ids, d_dirs);
        rc = wr_acs_reset(a);
    }
    if (rc == WR_OK) rc = collect_results(a, count, d_ids, d_dirs, stride, d_L, d_n);
    else cudaStreamSynchronize(s);
    pool_free(d_L, s); pool_free(d_n, s); pool_free(d_ids, s); pool_free(d_dirs, s);
    return rc;
}

static int check_queries(wr_acs* a, const char* who, const int64_t* start_ids, const int64_t* goal_ids, int n)
{
    for (int p = 0; p < n; p++) {
        if (start_ids[p] < 0 || goal_ids[p] < 0) { set_error("%s: pair %d has an endpoint that did not snap to a free node", who, p); return WR_ERR_NOTFOUND; }
        if ((size_t)start_ids[p] >= a->N || (size_t)goal_ids[p] >= a->N) { set_error("%s: id out of range", who); return WR_ERR_INVALID; }
    }
    return WR_OK;
}

// cache -> the caller's arrays
static void export_results(const wr_acs* a, int n, float* L, int* path_nodes, int64_t* path_ids, int* path_dirs, int path_cap)
{
    for (int p = 0; p < n; p++) {
        L[p] = a->res_L[p]; path_nodes[p] = a->res_n[p];
        const int m = std::min(a->res_n[p], path_cap);
        for (int i = 0; i < m; i++) path_ids[(size_t)p * path_cap + i] = a->res_ids[a->res_off[p] + i];
        for (int i = 0; i + 1 < m; i++) path_dirs[(size_t)p * path_cap + i] = a->res_dirs[a->res_off[p] + i];
    }
}
static void clear_results(wr_acs* a) { a->res_L.clear(); a->res_n.clear(); a->res_off.clear(); a->res_ids.clear(); a->res_dirs.clear(); }

extern "C" int wr_acs_search_pairs(wr_acs* a, const int64_t* start_ids, const int64_t* goal_ids, int npairs, float predict, int n_iterations,
                                   float* L, int* path_nodes, int64_t* path_ids, int* path_dirs, int path_cap)
{
    WR_REQUIRE(a && start_ids && goal_ids && L && path_nodes && npairs >= 0 && n_iterations >= 0, WR_ERR_INVALID, "wr_acs_search_pairs: bad argument");
    WR_REQUIRE(a->nranks == 1, WR_ERR_STATE, "wr_acs_search_pairs: independent searches are sharded by giving each rank its own pairs");
    WR_REQUIRE(path_cap >= 0 && (path_cap == 0 || (path_ids && path_dirs)), WR_ERR_INVALID, "wr_acs_search_pairs: path buffers missing");
    int rc = check_queries(a, "wr_acs_search_pairs", start_ids, goal_ids, npairs);
    if (rc != WR_OK) return rc;
    clear_results(a);
    if (npairs == 0) return WR_OK;
    WR_CUDA(cudaSetDevice(a->device));
    rc = run_pairs_sequential(a, start_ids, goal_ids, 0, npairs, predict, n_iterations);
    if (rc == WR_OK) export_results(a, npairs, L, path_nodes, path_ids, path_dirs, path_cap);
    return rc;
}

extern "C" int wr_acs_result_path(wr_acs* a, int index, int64_t* ids, int* dirs, int cap, int* n, float* L)
{
    WR_REQUIRE(a && n && L, WR_ERR_INVALID, "wr_acs_result_path: null");
    WR_REQUIRE(index >= 0 && (size_t)index < a->res_L.size(), WR_ERR_INVALID, "wr_acs_result_path: no such result (run wr_acs_search_pairs / wr_acs_search_batch first)");
    *n = a->res_n[index]; *L = a->res_L[index];
    const int m = std::min(*n, cap);
    if (ids) for (int i = 0; i < m; i++) ids[i] = a->res_ids[a->res_off[index] + i];
    if (dirs) for (int i = 0; i + 1 < m; i++) dirs[i] = a->res_dirs[a->res_off[index] + i];
    return WR_OK;
}

// ---- the same searches advanced CONCURRENTLY (batch.cuh) ---------------------------------------------------------------
struct wr_batch {   // buffers of the batch path, kept by the handle between calls
    BatchTable tab = {};
    size_t T = 0;
    BatchQuery* qs = nullptr;
    long long *d_starts = nullptr, *d_goals = nullptr;
    int* steps = nullptr;
    uint32_t* path_ids = nullptr; uint8_t* path_dirs = nullptr;
    uint32_t* ranked_keys = nullptr; uint16_t* ranked_vals = nullptr;
    uint32_t* best_ids = nullptr; uint8_t* best_dirs = nullptr;
    float* res_L = nullptr; int* res_n = nullptr;
    uint32_t* overflow_list = nullptr; unsigned long long* gtab = nullptr; int4* resume = nullptr;
    uint32_t* gkeys = nullptr;   // K = 26: tile keys of the HBM visited tables (gtab holds their masks)
    float* ant_L = nullptr;      // K = 26: [qc][cm] length of every ant
    unsigned long long* cnt_save = nullptr;
    uint32_t pool = 0;
    int qc = 0, cm = 0, K = 6;   // queries per chunk / colony / neighbourhood the buffers were sized for
    bool mem_limited = false;   // qc is what fits into memory, not what was asked for
};

static void free_batch(wr_acs* a)
{
    wr_batch* b = a->batch;
    if (!b) return;
    cudaStream_t s = a->stream;
    cudaStreamSynchronize(s);
    cudaFree(b->tab.ent); cudaFree(b->tab.list); cudaFree(b->tab.count);
    void* ptrs[] = {b->qs, b->d_starts, b->d_goals, b->steps, b->path_ids, b->path_dirs, b->ranked_keys, b->ranked_vals, b->best_ids, b->best_dirs, b->res_L, b->res_n,
                    b->overflow_list, b->gtab, b->resume, b->gkeys, b->ant_L, b->cnt_save};
    for (void* p : ptrs) cudaFree(p);
    delete b;
    a->batch = nullptr;
}

// the table kernels of a batch for its entries of EW words: kBatchEntryWords (K = 6) or kBatchEntryWords26 (K = 26)
template <int EW>
static void batch_table_fill(const wr_batch* b, cudaStream_t s) { k_batch_fill<EW><<<kNumSMs * 8, 256, 0, s>>>(reinterpret_cast<uint4*>(b->tab.ent), b->T); }
static void launch_batch_fill(const wr_batch* b, cudaStream_t s)
{
    if (b->K == kK26) batch_table_fill<kBatchEntryWords26>(b, s);
    else batch_table_fill<kBatchEntryWords>(b, s);
}
static void launch_batch_wipe(const wr_batch* b, cudaStream_t s)
{
    if (b->K == kK26) k_batch_wipe<kBatchEntryWords26><<<kNumSMs * 4, 256, 0, s>>>(b->tab);
    else k_batch_wipe<kBatchEntryWords><<<kNumSMs * 4, 256, 0, s>>>(b->tab);
}
// ranking, evaporation and deposits of one iteration of every query of a chunk of n
template <int EW>
static void batch_rank_update(const wr_acs* a, const wr_batch* b, int n, int maxn, size_t rank_smem, cudaStream_t s)
{
    const int cm = b->cm;
    k_batch_rank<EW><<<n, kRankSmallThreads, rank_smem, s>>>(a->d_state, b->qs, b->tab, b->steps, b->ant_L, cm, maxn, a->cap, a->rank_bits, a->d_Ltab, b->ranked_keys,
                                                              b->ranked_vals, b->path_ids, b->path_dirs, b->best_ids, b->best_dirs);
    k_batch_evaporate<EW><<<kNumSMs * 8, 256, 0, s>>>(b->tab, a->p.rho);
    k_batch_deposit<EW><<<n, kBatchDepThreads, 0, s>>>(a->d_state, b->qs, b->tab, b->ranked_keys, b->ranked_vals, cm, b->path_ids, b->path_dirs, a->cap, a->d_Ltab,
                                                       a->p.rho, b->steps);
}

static int batch_table_entries(int table_env_default)
{
    if (const char* e = getenv("WR_BATCH_TABLE")) return std::max(16, std::min(2048, atoi(e)));
    return table_env_default;
}

// sizes the batch buffers for chunks of up to `want_q` queries of `cm` ants; *qc = queries per chunk that fit
static int alloc_batch(wr_acs* a, int want_q, int cm, int* qc_out)
{
    const size_t cap = a->cap;
    const bool k26 = a->K == kK26;
    if (a->batch && a->batch->cm == cm && a->batch->K == a->K && (a->batch->qc >= want_q || a->batch->mem_limited)) { *qc_out = a->batch->qc; return WR_OK; }
    free_batch(a);
    size_t free_b = 0, total_b = 0;
    WR_CUDA(cudaMemGetInfo(&free_b, &total_b));
    if (const char* e = getenv("WR_BATCH_MEM_MB")) free_b = std::min(free_b, (size_t)atoll(e) << 20);
    const size_t per_q = (size_t)cm * cap * 5 + (size_t)cm * (k26 ? 14 : 10) + (cap + 1) * 5 + sizeof(BatchQuery) + 64;
    const size_t fit = std::min<size_t>(std::max<size_t>(1, (free_b / 2) / per_q), (size_t)1 << 16);
    const int qc = (int)std::min<size_t>((size_t)want_q, fit);
    wr_batch* b = new wr_batch();
    a->batch = b;
    b->qc = qc; b->cm = cm; b->K = a->K; b->mem_limited = (size_t)want_q > fit;
    // pheromone table: one for the whole chunk.  A quarter of the free memory at most, 2^17 entries (4 MB; K = 26: 16 MB) per
    // query at most
    const int ew = k26 ? kBatchEntryWords26 : kBatchEntryWords;
    const size_t ebytes = (size_t)ew * sizeof(uint32_t);
    size_t T = (size_t)1 << 16;
    while (T < (size_t)qc << 17 && T * 2 * ebytes <= free_b / 4 && T < ((size_t)1 << 30)) T <<= 1;
    if (const char* e = getenv("WR_BATCH_LOG2")) T = (size_t)1 << std::max(8, std::min(30, atoi(e)));
    b->T = T;
    b->tab.tmask = (uint32_t)(T - 1); b->tab.shift = 32 - ceil_log2(T); b->tab.limit = (uint32_t)(T / 2);
    WR_CUDA(cudaMalloc(&b->tab.ent, T * ebytes));
    WR_CUDA(cudaMalloc(&b->tab.list, (size_t)b->tab.limit * sizeof(uint32_t)));
    WR_CUDA(cudaMalloc(&b->tab.count, 4 * sizeof(uint32_t)));
    launch_batch_fill(b, a->stream);
    WR_CUDA(cudaMemsetAsync(b->tab.count, 0, 4 * sizeof(uint32_t), a->stream));
    const size_t nq = qc;
    WR_CUDA(cudaMalloc(&b->qs, nq * sizeof(BatchQuery)));
    WR_CUDA(cudaMalloc(&b->d_starts, nq * sizeof(long long)));
    WR_CUDA(cudaMalloc(&b->d_goals, nq * sizeof(long long)));
    WR_CUDA(cudaMalloc(&b->steps, nq * cm * sizeof(int)));
    WR_CUDA(cudaMalloc(&b->path_ids, nq * cm * cap * sizeof(uint32_t)));
    WR_CUDA(cudaMalloc(&b->path_dirs, nq * cm * cap));
    WR_CUDA(cudaMalloc(&b->ranked_keys, nq * cm * sizeof(uint32_t)));
    WR_CUDA(cudaMalloc(&b->ranked_vals, nq * cm * sizeof(uint16_t)));
    WR_CUDA(cudaMalloc(&b->best_ids, nq * (cap + 1) * sizeof(uint32_t)));
    WR_CUDA(cudaMalloc(&b->best_dirs, nq * (cap + 1)));
    WR_CUDA(cudaMalloc(&b->res_L, nq * sizeof(float)));
    WR_CUDA(cudaMalloc(&b->res_n, nq * sizeof(int)));
    if (k26) WR_CUDA(cudaMalloc(&b->ant_L, nq * cm * sizeof(float)));
    // HBM visited tables for ants whose shared-memory table fills up: a pool (2 GB at most), handed out on demand.  K = 6:
    // k_walk_batch's 64-bit key|mask entries; K = 26: k_walk26's format, u32 tile keys + u64 masks
    const size_t Eg = (size_t)1 << a->gtable_log2_for_cap();
    const size_t gbytes = k26 ? 12 : 8;
    size_t pool = std::min<size_t>(nq * cm, std::max<size_t>(16, ((size_t)2 << 30) / (Eg * gbytes)));
    b->pool = (uint32_t)pool;
    WR_CUDA(cudaMalloc(&b->overflow_list, pool * sizeof(uint32_t)));
    WR_CUDA(cudaMalloc(&b->gtab, pool * Eg * sizeof(unsigned long long)));
    if (k26) WR_CUDA(cudaMalloc(&b->gkeys, pool * Eg * sizeof(uint32_t)));
    WR_CUDA(cudaMalloc(&b->resume, pool * sizeof(int4)));
    WR_CUDA(cudaMalloc(&b->cnt_save, 16 * sizeof(unsigned long long)));
    WR_CUDA(cudaGetLastError());
    *qc_out = qc;
    return WR_OK;
}

extern "C" int wr_acs_search_batch(wr_acs* a, const int64_t* start_ids, const int64_t* goal_ids, int nq, float predict, int n_iterations,
                                   float* L, int* path_nodes, int64_t* path_ids, int* path_dirs, int path_cap)
{
    WR_REQUIRE(a && start_ids && goal_ids && L && path_nodes && nq >= 0 && n_iterations >= 0, WR_ERR_INVALID, "wr_acs_search_batch: bad argument");
    WR_REQUIRE(a->nranks == 1, WR_ERR_STATE, "wr_acs_search_batch: independent searches are sharded by giving each rank its own queries");
    WR_REQUIRE(path_cap >= 0 && (path_cap == 0 || (path_ids && path_dirs)), WR_ERR_INVALID, "wr_acs_search_batch: path buffers missing");
    int rc = check_queries(a, "wr_acs_search_batch", start_ids, goal_ids, nq);
    if (rc != WR_OK) return rc;
    clear_results(a);
    if (nq == 0) return WR_OK;
    WR_CUDA(cudaSetDevice(a->device));
    cudaStream_t s = a->stream;
    const int cm = a->p.fixed_colony > 0 ? a->p.fixed_colony : (int)(0.35 * (double)predict / (double)a->g->precision);   // :247 with best = inf
    WR_REQUIRE(cm >= 0 && cm < (1 << 24), WR_ERR_INVALID, "wr_acs_search_batch: colony size out of range");
    // What the batch path does not cover runs as the sequential loop (same results by definition): colonies that fill the
    // GPU on their own, the unordered atomic mode, a pheromone field that is not in its initial state
    const bool batchable = cm >= 1 && cm <= kBatchMaxColony && a->p.update_mode != WR_UPDATE_ATOMIC && a->field_clean && nq > 1 && batch_enabled();
    const bool k26 = a->K == kK26;
    const uint32_t first_search = a->next_search;
    if (!batchable) {
        rc = run_pairs_sequential(a, start_ids, goal_ids, 0, nq, predict, n_iterations);
        if (rc == WR_OK) export_results(a, nq, L, path_nodes, path_ids, path_dirs, path_cap);
        return rc;
    }
    if (!k26) {
        rc = grid_ensure_open6(a->g, s);
        if (rc != WR_OK) return rc;
    }
    int qc = 0;
    rc = alloc_batch(a, nq, cm, &qc);
    if (rc != WR_OK) return rc;
    wr_batch* b = a->batch;
    const int entries = batch_table_entries(320);   // 42 KB per CTA: five CTAs per SM, like the register bound (C5: 256 -> 1898, 320 -> 2095, 384 -> 1989, 512 -> 1636 queries/s)
    // K = 26: four ants per CTA, each with k_walk26's shared-memory visited table of 1 << walk_table_log2 entries (12 B each)
    const size_t smem1 = k26 ? ((size_t)kWalk26Ants << a->table_log2) * 12 : kWalk2Lut + 128 + (size_t)kAntsPerCta * entries * sizeof(unsigned long long);
    WR_REQUIRE(smem1 <= 227 * 1024, WR_ERR_INVALID, "wr_acs_search_batch: WR_BATCH_TABLE too large");
    const bool alpha1 = a->p.alpha == 1;
    const int maxn = (std::max(cm, 32) + 31) / 32 * 32;
    const size_t rank_smem = (size_t)12 * maxn + 32 * 256 * sizeof(uint32_t);
    if (k26) {
        WR_CUDA(cudaFuncSetAttribute(k_walk_batch26<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
    } else {
        WR_CUDA(cudaFuncSetAttribute(k_walk_batch3<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
        WR_CUDA(cudaFuncSetAttribute(k_walk_batch3<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
    }
    if (k26) WR_CUDA(cudaFuncSetAttribute(k_batch_rank<kBatchEntryWords26>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rank_smem));
    else WR_CUDA(cudaFuncSetAttribute(k_batch_rank<kBatchEntryWords>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rank_smem));
    const int per_sm = std::max(1, std::min(16, (int)((227 * 1024) / (smem1 + 1024))));
    BatchArgs w;
    w.st = a->d_state; w.qs = b->qs; w.colony_max = cm; w.items_per_query = k26 ? cm : (cm + 3) / 4;   // K = 26: one ant per work item
    w.tab = b->tab; w.open6 = a->g->d_open6; w.occ = a->g->d_bits; w.coords = a->g->d_coords; w.rx = a->g->rx; w.ry = a->g->ry; w.rz = a->g->rz;
    w.seed_lo = (uint32_t)a->p.seed; w.seed_hi = (uint32_t)(a->p.seed >> 32); w.alpha = a->p.alpha; w.beta = a->p.beta; w.cap = a->cap;
    w.ant_steps = b->steps; w.path_ids = b->path_ids; w.path_dirs = b->path_dirs; w.table_entries = entries;
    w.overflow_list = b->overflow_list; w.gtab = b->gtab; w.gtable_log2 = a->gtable_log2_for_cap(); w.resume = b->resume; w.pool = b->pool;
    w.table_log2 = a->table_log2; w.gkeys = b->gkeys; w.precision = a->g->precision; w.ant_L = b->ant_L;
    for (int c0 = 0; c0 < nq && rc == WR_OK; c0 += qc) {
        const int n = std::min(qc, nq - c0);
        w.nq = n;
        std::vector<long long> hs(n), hg(n);
        for (int q = 0; q < n; q++) { hs[q] = start_ids[c0 + q]; hg[q] = goal_ids[c0 + q]; }
        WR_CUDA(cudaMemcpyAsync(b->d_starts, hs.data(), (size_t)n * sizeof(long long), cudaMemcpyHostToDevice, s));
        WR_CUDA(cudaMemcpyAsync(b->d_goals, hg.data(), (size_t)n * sizeof(long long), cudaMemcpyHostToDevice, s));
        WR_CUDA(cudaStreamSynchronize(s));   // hs / hg are on this frame
        // counters as they are before this chunk: a chunk that has to be re-run sequentially must not count twice
        unsigned long long* d_cnt = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(a->d_state) + offsetof(IterState, cnt));
        WR_CUDA(cudaMemcpyAsync(b->cnt_save, d_cnt, sizeof(unsigned long long) * 9, cudaMemcpyDeviceToDevice, s));
        k_batch_begin<<<(n + 255) / 256, 256, 0, s>>>(a->d_state, b->qs, n, b->d_starts, b->d_goals, first_search + (uint32_t)c0, predict, a->p.tau0, b->tab.count);
        const int items = n * w.items_per_query;
        const int blocks1 = std::max(1, std::min((items + 3) / 4, kNumSMs * per_sm));   // four work items per CTA for either K
        const int pass2_ants = k26 ? kWalk26Ants : kAntsPerCta;
        const int blocks2 = std::max(1, std::min((int)((b->pool + pass2_ants - 1) / pass2_ants), kNumSMs * 4));
        for (int it = 0; it < n_iterations; it++) {
            k_batch_iter_begin<<<(n + 255) / 256, 256, 0, s>>>(a->d_state, b->qs, n, a->p.fixed_colony, cm, a->g->precision, a->p.tau0, it > 0 ? 1 : 0, a->p.rho);
            if (k26) {
                k_walk_batch26<false><<<blocks1, kWalk26Threads, smem1, s>>>(w);
                k_walk_batch26<true><<<blocks2, kWalk26Threads, 0, s>>>(w);
            } else if (alpha1) {
                k_walk_batch3<true><<<blocks1, kWalkThreads, smem1, s>>>(w);
                k_walk_batch<true><<<blocks2, kWalkThreads, kWalk2Lut, s>>>(w);
            } else {
                k_walk_batch3<false><<<blocks1, kWalkThreads, smem1, s>>>(w);
                k_walk_batch<false><<<blocks2, kWalkThreads, kWalk2Lut, s>>>(w);
            }
            if (k26) batch_rank_update<kBatchEntryWords26>(a, b, n, maxn, rank_smem, s);
            else batch_rank_update<kBatchEntryWords>(a, b, n, maxn, rank_smem, s);
        }
        k_batch_results<<<(n + 255) / 256, 256, 0, s>>>(b->qs, n, b->res_L, b->res_n);
        WR_CUDA(cudaGetLastError());
        uint32_t cnt[4] = {0, 0, 0, 0};
        WR_CUDA(cudaMemcpyAsync(cnt, b->tab.count, sizeof cnt, cudaMemcpyDeviceToHost, s));
        WR_CUDA(cudaStreamSynchronize(s));
        launch_batch_wipe(b, s);
        a->batch_last_entries = cnt[0];
        if (cnt[1]) {   // pheromone table or overflow-table pool exhausted: this chunk's searches run one after the other instead
            a->batch_fallbacks++;
            launch_batch_fill(b, s);   // entries claimed beyond the list
            WR_CUDA(cudaMemcpyAsync(d_cnt, b->cnt_save, sizeof(unsigned long long) * 9, cudaMemcpyDeviceToDevice, s));
            k_set_base<<<1, 1, 0, s>>>(a->d_state, a->p.tau0);   // the batch advanced the handle's scalar; the dense field itself is untouched
            a->next_search = first_search + (uint32_t)c0;
            rc = run_pairs_sequential(a, start_ids, goal_ids, c0, n, predict, n_iterations);
        } else {
            rc = collect_results(a, n, b->best_ids, b->best_dirs, (size_t)a->cap + 1, b->res_L, b->res_n);
        }
    }
    a->next_search = first_search + (uint32_t)nq;
    a->begun = false;
    if (rc == WR_OK) rc = wr_acs_reset(a);   // the sequential loop ends every search with reset() (:481)
    if (rc == WR_OK) export_results(a, nq, L, path_nodes, path_ids, path_dirs, path_cap);
    return rc;
}

extern "C" int wr_acs_batch_stats(wr_acs* a, uint64_t out[4])
{
    WR_REQUIRE(a && out, WR_ERR_INVALID, "wr_acs_batch_stats: null");
    out[0] = a->batch ? (uint64_t)a->batch->qc : 0; out[1] = a->batch ? (uint64_t)a->batch->T : 0;
    out[2] = a->batch_last_entries; out[3] = a->batch_fallbacks;
    return WR_OK;
}

// ---- ant sharding across ranks ------------------------------------------------------------------
// CUDA loads a kernel's code the first time it is launched (lazy module loading), and loading may have to wait for running
// kernels.  A sharded iteration contains kernels that WAIT for other handles' kernels (k_peer_barrier); if those handles live
// in this process (several shards driven from one host thread) a first-time load behind a spinning barrier would wait for a
// signal that this very thread has not enqueued yet.  So everything an iteration can launch is loaded up front.
static int preload_iteration_kernels()
{
    static unsigned long long done = 0;   // one bit per device (modules are loaded per context)
    int dev = 0;
    WR_CUDA(cudaGetDevice(&dev));
    if (done >> (dev & 63) & 1ull) return WR_OK;
    cudaFuncAttributes at;
#define WR_PRELOAD(f) WR_CUDA(cudaFuncGetAttributes(&at, f))
    WR_PRELOAD(k_gather_steps); WR_PRELOAD(k_rank_small); WR_PRELOAD(k_rank_chunks); WR_PRELOAD(k_rank_merge);
    WR_PRELOAD(k_rank_finish_prefix); WR_PRELOAD(k_best_copy_peer); WR_PRELOAD(k_best_copy); WR_PRELOAD(k_rankset_gen); WR_PRELOAD(k_rankset_publish);
    WR_PRELOAD(k_rankset_merge); WR_PRELOAD(k_evaporate_tiles); WR_PRELOAD(k_rankset_apply); WR_PRELOAD(k_rankset_clear); WR_PRELOAD(k_deposit_serial);
    WR_PRELOAD((k_deposit_gen<false, true>)); WR_PRELOAD(k_tile_offsets); WR_PRELOAD(k_update_fused<true>); WR_PRELOAD(k_update_fused<false>);
    WR_PRELOAD(k_pull_finals); WR_PRELOAD(k_iter_begin); WR_PRELOAD(k_iter_end); WR_PRELOAD(k_path_warm); WR_PRELOAD(k_rankset_warm);
    WR_PRELOAD((k_walk3<true, 0>)); WR_PRELOAD((k_walk3<true, 1>)); WR_PRELOAD((k_walk3<false, 0>)); WR_PRELOAD((k_walk3<false, 1>));
    WR_PRELOAD((k_walk2<true>)); WR_PRELOAD((k_walk2<false>));
#undef WR_PRELOAD
    int rc = sort_preload();
    if (rc != WR_OK) return rc;
    done |= 1ull << (dev & 63);
    return WR_OK;
}

extern "C" int wr_acs_set_shard(wr_acs* a, int rank, int nranks)
{
    WR_REQUIRE(a && nranks >= 1 && rank >= 0 && rank < nranks, WR_ERR_INVALID, "wr_acs_set_shard: bad argument");
    WR_REQUIRE(!a->begun || (a->rank == rank && a->nranks == nranks), WR_ERR_STATE, "wr_acs_set_shard: set the shard before wr_acs_begin");
    WR_REQUIRE(nranks == 1 || a->p.update_mode != WR_UPDATE_ATOMIC, WR_ERR_INVALID, "wr_acs_set_shard: sharded colonies use the rank-ordered update modes");
    WR_REQUIRE(nranks == 1 || a->K == 6, WR_ERR_INVALID, "wr_acs_set_shard: the K = 26 extension runs on one GPU (ranks would have to exchange lengths as well as step counts)");
    WR_REQUIRE(nranks <= 256, WR_ERR_INVALID, "wr_acs_set_shard: at most 256 ranks");
    if (nranks > 1) { WR_CUDA(cudaSetDevice(a->device)); int rc = preload_iteration_kernels(); if (rc != WR_OK) return rc; }
    WR_REQUIRE(nranks == 1 || a->p.update_mode == WR_UPDATE_FUSED, WR_ERR_INVALID, "wr_acs_set_shard: sharded colonies use WR_UPDATE_FUSED or WR_UPDATE_RANKSET");
    a->rank = rank; a->nranks = nranks;
    return WR_OK;
}

// ---- sharded colonies over NVLink peer memory -------------------------------------------------------------------------
extern "C" int wr_acs_peer_export(wr_acs* a, void* ipc_handle, void** raw_pointer)
{
    WR_REQUIRE(a && a->begun && a->nranks > 1 && a->d_slab, WR_ERR_STATE, "wr_acs_peer_export: sharded handle after wr_acs_begin only");
    // the barrier epochs restart with every exchange: this rank's flag words and its epoch go back to 0 BEFORE the handle
    // leaves (the exchange itself is a host-side barrier, so no peer can signal before every rank has done this)
    WR_CUDA(cudaMemsetAsync(a->d_slab + a->off_flags, 0, 4096, a->stream));
    WR_CUDA(cudaMemsetAsync(a->d_epoch, 0, 2 * sizeof(uint32_t), a->stream));
    WR_CUDA(cudaStreamSynchronize(a->stream));
    a->peers_set = false;
    if (ipc_handle) WR_CUDA(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(ipc_handle), a->d_slab));
    if (raw_pointer) *raw_pointer = a->d_slab;
    return WR_OK;
}

static int install_peers(wr_acs* a, const std::vector<const unsigned char*>& slabs)
{
    std::vector<const void*> tab((size_t)wr_acs::kTabKinds * 2 * a->nranks);
    for (int r = 0; r < a->nranks; r++)
        for (int b = 0; b < 2; b++) {
            tab[((size_t)0 * 2 + b) * a->nranks + r] = slabs[r] + a->off_ids[b];
            tab[((size_t)1 * 2 + b) * a->nranks + r] = slabs[r] + a->off_dirs[b];
            tab[((size_t)2 * 2 + b) * a->nranks + r] = slabs[r] + a->off_fin[b];
            tab[((size_t)3 * 2 + b) * a->nranks + r] = slabs[r] + a->off_steps[b];
            tab[((size_t)4 * 2 + b) * a->nranks + r] = slabs[r] + a->off_pub;
            tab[((size_t)5 * 2 + b) * a->nranks + r] = slabs[r] + a->off_flags;
        }
    WR_CUDA(cudaMemcpyAsync(a->d_tabs, tab.data(), tab.size() * sizeof(void*), cudaMemcpyHostToDevice, a->stream));
    WR_CUDA(cudaStreamSynchronize(a->stream));
    a->peers_set = true;
    return WR_OK;
}

extern "C" int wr_acs_peer_import(wr_acs* a, const void* all_ipc_handles)
{
    WR_REQUIRE(a && all_ipc_handles && a->begun && a->nranks > 1 && a->d_slab, WR_ERR_STATE, "wr_acs_peer_import: sharded handle after wr_acs_begin only");
    WR_CUDA(cudaSetDevice(a->device));
    const cudaIpcMemHandle_t* h = reinterpret_cast<const cudaIpcMemHandle_t*>(all_ipc_handles);
    std::vector<const unsigned char*> slabs(a->nranks);
    for (int r = 0; r < a->nranks; r++) {
        if (r == a->rank) { slabs[r] = a->d_slab; continue; }
        void* p = nullptr;
        {
            std::lock_guard<std::mutex> lock(g_rs_cache_mu);
            if (g_ipc_maps.size() < (size_t)a->nranks) g_ipc_maps.resize(a->nranks);
            IpcMapping& m = g_ipc_maps[r];
            if (m.ptr && memcmp(&m.handle, &h[r], sizeof(cudaIpcMemHandle_t)) == 0) p = m.ptr;   // the peer re-used its parked slab
            else {
                if (m.ptr) { cudaIpcCloseMemHandle(m.ptr); m.ptr = nullptr; }
                WR_CUDA(cudaIpcOpenMemHandle(&p, h[r], cudaIpcMemLazyEnablePeerAccess));
                m.handle = h[r]; m.ptr = p;
            }
        }
        slabs[r] = static_cast<const unsigned char*>(p);
    }
    return install_peers(a, slabs);
}

extern "C" int wr_acs_peer_set_pointers(wr_acs* a, void* const* all_raw_pointers)
{
    WR_REQUIRE(a && all_raw_pointers && a->begun && a->nranks > 1 && a->d_slab, WR_ERR_STATE, "wr_acs_peer_set_pointers: sharded handle after wr_acs_begin only");
    std::vector<const unsigned char*> slabs(a->nranks);
    for (int r = 0; r < a->nranks; r++) slabs[r] = r == a->rank ? a->d_slab : static_cast<const unsigned char*>(all_raw_pointers[r]);
    // Shards that live in one process wait for each other's kernels ON THE SAME GPU: every barrier kernel needs the other shards'
    // kernels to be scheduled beside it.  Such handles spin with small grids (barrier_grid) and use plain launches on one stream
    // each — no whole-iteration graphs, no forked evaporation stream — so that as little as possible must be resident at once.
    // One process per GPU — the product layout — waits for OTHER GPUs only and keeps full grids, graphs and the overlap.
    a->in_process_peers = true;
    return install_peers(a, slabs);
}

extern "C" int wr_acs_sync(wr_acs* a)
{
    WR_REQUIRE(a, WR_ERR_INVALID, "wr_acs_sync: null");
    WR_CUDA(cudaStreamSynchronize(a->stream));
    if (a->timer.enabled) a->timer.resolve();
    if (a->d_peer_err) {
        uint32_t err = 0;
        WR_CUDA(cudaMemcpy(&err, a->d_peer_err, sizeof err, cudaMemcpyDeviceToHost));
        if (err) { set_error("wr_acs_sync: a peer rank did not reach a barrier within %.1f s (results of this search are invalid)", a->barrier_timeout_ns * 1e-9); return WR_ERR_CUDA; }
    }
    return WR_OK;
}

extern "C" int wr_acs_reset(wr_acs* a)
{   // reset() :307-315: every slot (out-of-bounds ones included) back to tau0
    WR_REQUIRE(a, WR_ERR_INVALID, "wr_acs_reset: null");
    WR_CUDA(cudaSetDevice(a->device));
    if (a->lazy) {   // clean-tile field: back to all-sentinel with base = tau0; after the first reset only the dirty tiles need rewriting
        k_tau_reset_tiles<<<kNumSMs * 8, 256, 0, a->stream>>>(reinterpret_cast<float4*>(a->d_tau), a->ntiles, a->d_dirty, a->oob_zero ? 1 : 0);
        a->oob_zero = false;
    } else {
        k_tau_fill<<<kNumSMs * 8, 256, 0, a->stream>>>(a->d_tau, a->n_slots, a->p.tau0);
    }
    k_set_base<<<1, 1, 0, a->stream>>>(a->d_state, a->p.tau0);
    WR_CUDA(cudaGetLastError());
    a->field_clean = true;
    return WR_OK;
}

extern "C" int wr_acs_best(wr_acs* a, int64_t* ids, int* dirs, int cap, int* n, float* L)
{
    WR_REQUIRE(a && n && L, WR_ERR_INVALID, "wr_acs_best: null");
    WR_CUDA(cudaStreamSynchronize(a->stream));
    IterState st;
    WR_CUDA(cudaMemcpy(&st, a->d_state, sizeof st, cudaMemcpyDeviceToHost));
    *L = st.best_L;
    if (st.best_steps == INT_MAX) { *n = 0; return WR_OK; }
    const int nodes = st.best_steps + 1;
    *n = nodes;
    if (ids && cap > 0) {
        std::vector<uint32_t> h(nodes);
        WR_CUDA(cudaMemcpy(h.data(), a->d_best_ids, nodes * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        for (int i = 0; i < nodes && i < cap; i++) ids[i] = h[i];
    }
    if (dirs && cap > 0 && nodes > 1) {
        std::vector<uint8_t> h(nodes - 1);
        WR_CUDA(cudaMemcpy(h.data(), a->d_best_dirs, nodes - 1, cudaMemcpyDeviceToHost));
        for (int i = 0; i < nodes - 1 && i < cap; i++) dirs[i] = h[i];
    }
    return WR_OK;
}

extern "C" int wr_acs_download_pheromone(wr_acs* a, float* tau, size_t n)
{
    WR_REQUIRE(a && tau, WR_ERR_INVALID, "wr_acs_download_pheromone: null");
    WR_REQUIRE(n >= a->n_slots, WR_ERR_CAPACITY, "wr_acs_download_pheromone: buffer too small");
    WR_CUDA(cudaStreamSynchronize(a->stream));
    WR_CUDA(cudaMemcpy(tau, a->d_tau, a->n_slots * sizeof(float), cudaMemcpyDeviceToHost));
    if (a->lazy) {   // clean-tile field: a sentinel stands for the value every never-deposited slot holds now
        IterState st;
        WR_CUDA(cudaMemcpy(&st, a->d_state, sizeof st, cudaMemcpyDeviceToHost));
        uint32_t* w = reinterpret_cast<uint32_t*>(tau);
        uint32_t basebits;
        memcpy(&basebits, &st.base, sizeof basebits);
        for (size_t i = 0; i < a->n_slots; i++) if (w[i] == kSentinelBits) w[i] = basebits;
    }
    return WR_OK;
}
extern "C" int wr_acs_upload_pheromone(wr_acs* a, const float* tau, size_t n)
{
    WR_REQUIRE(a && tau, WR_ERR_INVALID, "wr_acs_upload_pheromone: null");
    WR_REQUIRE(n == a->n_slots, WR_ERR_INVALID, "wr_acs_upload_pheromone: size mismatch");
    WR_CUDA(cudaStreamSynchronize(a->stream));
    if (a->lazy) {
        // clean-tile field: the bit pattern of -0.0f is the "never deposited" sentinel, which every kernel replaces by
        // IterState::base.  An uploaded -0.0f is a VALUE (it compares equal to 0 and evaporates to -0 like +0 to +0), so it
        // is stored as +0.0f: the same number in every comparison and product the search performs on it.
        std::vector<float> h(tau, tau + a->n_slots);
        uint32_t* w = reinterpret_cast<uint32_t*>(h.data());
        for (size_t i = 0; i < a->n_slots; i++) if (w[i] == kSentinelBits) w[i] = 0u;
        WR_CUDA(cudaMemcpy(a->d_tau, h.data(), a->n_slots * sizeof(float), cudaMemcpyHostToDevice));
    } else {
        WR_CUDA(cudaMemcpy(a->d_tau, tau, a->n_slots * sizeof(float), cudaMemcpyHostToDevice));
    }
    WR_CUDA(cudaMemset(a->d_dirty, 1, (size_t)a->ntiles + 1));   // explicit values everywhere: every tile takes part in the evaporation
    a->field_clean = false;
    return WR_OK;
}

extern "C" int wr_acs_last_colony(wr_acs* a, int* colony, float* lambda, float* Q)
{
    WR_REQUIRE(a, WR_ERR_INVALID, "wr_acs_last_colony: null");
    WR_CUDA(cudaStreamSynchronize(a->stream));
    IterState st;
    WR_CUDA(cudaMemcpy(&st, a->d_state, sizeof st, cudaMemcpyDeviceToHost));
    if (colony) *colony = st.colony;
    if (lambda) *lambda = st.lambda;
    if (Q) *Q = st.Q;
    return WR_OK;
}

extern "C" int wr_acs_last_ant(wr_acs* a, int k, int64_t* ids, int* dirs, int cap, int* n, float* L, int* order)
{
    WR_REQUIRE(a && n && L, WR_ERR_INVALID, "wr_acs_last_ant: null");
    WR_REQUIRE(a->begun, WR_ERR_STATE, "wr_acs_last_ant: no iteration yet");
    WR_CUDA(cudaStreamSynchronize(a->stream));
    IterState st;
    WR_CUDA(cudaMemcpy(&st, a->d_state, sizeof st, cudaMemcpyDeviceToHost));
    WR_REQUIRE(k >= 0 && k < st.colony, WR_ERR_INVALID, "wr_acs_last_ant: ant index out of range");
    const int first = a->rank * a->chunk;
    WR_REQUIRE(k >= first && k < first + a->chunk, WR_ERR_INVALID, "wr_acs_last_ant: ant lives on another rank");
    int steps = 0, ord = 0;
    WR_CUDA(cudaMemcpy(&steps, a->d_ant_steps + k, sizeof(int), cudaMemcpyDeviceToHost));
    WR_CUDA(cudaMemcpy(&ord, a->d_order + k, sizeof(int), cudaMemcpyDeviceToHost));
    if (order) *order = ord;
    if (steps < 0) { *L = INFINITY; *n = 0; return WR_OK; }   // the trail of a dead ant is not kept
    *L = a->h_Ltab[steps];
    if (a->K == kK26) WR_CUDA(cudaMemcpy(L, a->d_ant_L + (k - first), sizeof(float), cudaMemcpyDeviceToHost));
    *n = steps + 1;
    const size_t off = (size_t)(k - first) * a->cap;
    if (ids && cap > 0) {
        std::vector<uint32_t> h(steps);
        WR_CUDA(cudaMemcpy(h.data(), a->d_path_ids + off, steps * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        for (int i = 0; i < steps && i < cap; i++) ids[i] = h[i];
        if (steps < cap) ids[steps] = a->goal;
    }
    if (dirs && cap > 0) {
        std::vector<uint8_t> h(steps);
        WR_CUDA(cudaMemcpy(h.data(), a->d_path_dirs + off, steps, cudaMemcpyDeviceToHost));
        for (int i = 0; i < steps && i < cap; i++) dirs[i] = h[i];
    }
    return WR_OK;
}

extern "C" int wr_acs_counters(wr_acs* a, uint64_t out[9])
{
    WR_REQUIRE(a && out, WR_ERR_INVALID, "wr_acs_counters: null");
    WR_CUDA(cudaStreamSynchronize(a->stream));
    IterState st;
    WR_CUDA(cudaMemcpy(&st, a->d_state, sizeof st, cudaMemcpyDeviceToHost));
    for (int i = 0; i < 9; i++) out[i] = st.cnt[i];
    return WR_OK;
}

extern "C" int wr_acs_set_timing(wr_acs* a, int enabled)
{
    WR_REQUIRE(a, WR_ERR_INVALID, "wr_acs_set_timing: null");
    WR_CUDA(cudaStreamSynchronize(a->stream));
    a->timer.resolve();
    a->timer.enabled = enabled != 0;
    return WR_OK;
}
extern "C" int wr_acs_kernel_ms(wr_acs* a, float out[5])
{
    WR_REQUIRE(a && out, WR_ERR_INVALID, "wr_acs_kernel_ms: null");
    WR_CUDA(cudaStreamSynchronize(a->stream));
    a->timer.resolve();
    for (int i = 0; i < 5; i++) out[i] = a->timer.ms[i];
    return WR_OK;
}

extern "C" int wr_acs_update_stats(wr_acs* a, uint32_t out[4])
{
    WR_REQUIRE(a && out, WR_ERR_INVALID, "wr_acs_update_stats: null");
    WR_CUDA(cudaStreamSynchronize(a->stream));
    IterState st;
    WR_CUDA(cudaMemcpy(&st, a->d_state, sizeof st, cudaMemcpyDeviceToHost));
    out[0] = (uint32_t)st.use_rankset; out[1] = st.spread_tiles; out[2] = st.spread_slots; out[3] = st.rankset_iters;
    return WR_OK;
}

extern "C" int wr_acs_stream_kernel_ms(wr_acs* a, float* ms, int* launches)
{
    WR_REQUIRE(a && ms && launches, WR_ERR_INVALID, "wr_acs_stream_kernel_ms: null");
    WR_CUDA(cudaStreamSynchronize(a->stream));
    a->sk_resolve();
    *ms = a->sk_ms; *launches = a->sk_launches;
    return WR_OK;
}

extern "C" int wr_acs_field_stats(wr_acs* a, uint64_t out[2])
{
    WR_REQUIRE(a && out, WR_ERR_INVALID, "wr_acs_field_stats: null");
    WR_CUDA(cudaStreamSynchronize(a->stream));
    std::vector<uint8_t> h(a->ntiles);
    WR_CUDA(cudaMemcpy(h.data(), a->d_dirty, a->ntiles, cudaMemcpyDeviceToHost));
    uint64_t n = 0;
    for (uint8_t v : h) n += v ? 1 : 0;
    out[0] = n; out[1] = a->ntiles;
    return WR_OK;
}

extern "C" int wr_acs_bench_kernel(wr_acs* a, int which, int reps, float* ms_per_launch)
{
    WR_REQUIRE(a && ms_per_launch && reps > 0 && which >= 0 && which <= 2, WR_ERR_INVALID, "wr_acs_bench_kernel: bad argument");
    WR_REQUIRE(a->begun, WR_ERR_STATE, "wr_acs_bench_kernel: call wr_acs_begin first");
    WR_CUDA(cudaSetDevice(a->device));
    cudaStream_t s = a->stream;
    cudaEvent_t e0, e1;
    WR_CUDA(cudaEventCreate(&e0));
    WR_CUDA(cudaEventCreate(&e1));
    float* scratch = nullptr;
    if (which == 2) WR_CUDA(dmalloc(&scratch, a->n_slots_pad * sizeof(float), s));
    const uint32_t* ck = a->recs_in_b ? a->sort_recs.keys_b : a->sort_recs.keys_a;
    const uint32_t* cv = a->recs_in_b ? a->sort_recs.vals_b : a->sort_recs.vals_a;
    const int* d_n = a->dptr_nrec();
    if (a->rankset) {   // no record list in this mode: the fused kernels run with zero records (count[2] stays 0)
        ck = cv = a->rs.list;
        d_n = reinterpret_cast<const int*>(a->rs.count + 2);
    }
    for (int r = -1; r < reps; r++) {   // one untimed warm-up launch
        if (r == 0) WR_CUDA(cudaEventRecord(e0, s));
        if (which == 0) {
            int rc = launch_fused(a, ck, cv, d_n);
            if (rc != WR_OK) return rc;
        } else if (which == 1) {
            k_evaporate<<<kNumSMs * 8, 256, 0, s>>>(reinterpret_cast<float4*>(a->d_tau), a->n_slots_pad / 4, a->p.rho);
        } else {
            WR_CUDA(cudaMemcpyAsync(scratch, a->d_tau, a->n_slots_pad * sizeof(float), cudaMemcpyDeviceToDevice, s));
        }
    }
    WR_CUDA(cudaEventRecord(e1, s));
    WR_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    WR_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    *ms_per_launch = ms / reps;
    cudaEventDestroy(e0); cudaEventDestroy(e1); pool_free(scratch, s);
    WR_CUDA(cudaGetLastError());
    return WR_OK;
}

