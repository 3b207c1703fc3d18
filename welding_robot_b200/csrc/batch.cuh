// Batched concurrent searches: the all-pairs loop of searchBestPathOfPoints (core/ACSRank_3D.hpp:472-499) and independent
// start/goal queries (BASELINE config 5) as ONE colony-of-colonies.  A 35- or 256-ant search is 9-64 warps on a machine
// that holds 9472; run one after the other (wr_acs_search_pairs) such searches leave the GPU 97 % idle.  Here up to
// thousands of searches advance in lockstep, one launch per phase covering every (query, ant):
//
//   k_batch_iter_begin   colony size, lambda, Q of every query (:247-249)
//   k_walk_batch3        K2 over (query, 4-ant group) work items, pass 1; pass 2 (parked ants) is k_walk2<Batch6>.  The step
//                        is walk2.cuh's with two differences forced by memory — 1024 dense pheromone + heuristic fields would
//                        need 800 MB (256^3) to 6.4 GB (512^3) EACH — both behind the input type Batch6:
//                          * pheromone lives in ONE hash table for the whole batch, keyed by (query, node): an entry holds the
//                            node's six directed slots (32 B = one sector, read by the ant's six lanes in one request); a node
//                            without an entry has never received a deposit and is worth the scalar `base` — the clean-tile
//                            argument of acs_kernels.cuh at node granularity, bit-exact for the same reason;
//                          * the geometric factor 1 + beta*cos is computed per step from the three axis tables (heur6, the
//                            function k_heuristic tabulates) while the pheromone gather is in flight, and
//                            the open-neighbour mask comes from the grid's one byte per node (grid.cu k_open6);
//   k_batch_rank         one CTA per query: stable sort by (steps, ant), best decision (:263-264), eligibility (:200), new
//                        best path and its node-membership flags (isOnBestPath, :209)
//   k_batch_evaporate    tau *= rho over the entries claimed so far (:268-272; every query is at the same iteration)
//   k_batch_deposit      one CTA per query: the reference's own loop order (:275-280) — eligible ants front to back, a CTA
//                        barrier per ant; within an ant every slot occurs once, so its steps run in parallel.  The colonies
//                        are small (<= 4096 ants), the parallelism comes from the number of queries.
// Every query draws from its own Philox search index (wr_common.cuh), so a batch equals the same searches run one after
// the other through wr_acs_search_pairs bit for bit — and those equal the oracle's.
// K = 26 (batch26.cuh) shares the table code — templated on the entry's words EW, so the K = 6 kernels keep a constant
// stride — with a 128-byte entry, ranking by the bits of L and deposits with the ant's own L; its walk is k_walk26<Batch26>.
#pragma once
#include "rank_small.cuh"
#include "walk2.cuh"
#include "walk3.cuh"

namespace wr {

constexpr int kBatchMaxColony = 4096;       // larger colonies fill the GPU on their own: wr_acs_search_pairs
constexpr int kBatchEntryWords = 8;         // K = 6: key (2 words: node+1 | query << 32 | on-best << 63), tau[6]
constexpr int kBatchEntryWords26 = 32;      // K = 26: the same key, tau[26] in the slot26 enumeration, 4 unused words (one 128 B line)
constexpr unsigned long long kBatchFlagBit = 1ull << 63;

struct BatchQuery {   // device-side state of one query (the part of IterState that differs between queries)
    int start, goal;
    uint32_t stream_word, block_hi;   // Philox counter words of its search index
    int colony;
    float lambda, Q;
    int best_steps;      // INT_MAX: none yet
    float best_L;        // +inf: none yet
    int best_changed, best_ant;
    int n_eligible;
    int best_n;          // nodes of the stored best path
    int pad;
};

struct BatchTable {
    uint32_t* ent;       // [T][EW]: kBatchEntryWords (K = 6) or kBatchEntryWords26 words per entry
    uint32_t* list;      // [limit] entries claimed since the batch began
    uint32_t* count;     // [0] claimed entries [1] failure flag (table or overflow-table pool exhausted: the batch is re-run) [2] pool tables in use
    uint32_t tmask;
    int shift;           // 32 - log2(T)
    uint32_t limit;      // claims allowed (T/2)
};

__device__ __forceinline__ uint32_t batch_hash(uint32_t node, uint32_t q) { return (node * 2654435761u) ^ (q * 0x85EBCA6Bu + (q << 13)); }

// entry of (query, node), or 0xFFFFFFFF if it has none
template <int EW>
__device__ __forceinline__ uint32_t batch_find(const BatchTable& t, uint32_t node, uint32_t q)
{
    const unsigned long long want = (unsigned long long)(node + 1u) | ((unsigned long long)q << 32);
    uint32_t h = batch_hash(node, q) >> t.shift;
    for (uint32_t probes = 0; probes <= t.tmask; probes++) {   // bounded: a failing batch (claims raced past the limit) may have filled a tiny table
        const unsigned long long k = *reinterpret_cast<const volatile unsigned long long*>(t.ent + (size_t)h * EW);
        if ((k & ~kBatchFlagBit) == want) return h;
        if (k == 0ull) return 0xFFFFFFFFu;
        h = (h + 1) & t.tmask;
    }
    return 0xFFFFFFFFu;
}

// ... created if missing (its slots hold the sentinel: the table is filled with sentinels, keys zero)
template <int EW>
__device__ __forceinline__ uint32_t batch_find_or_insert(const BatchTable& t, uint32_t node, uint32_t q)
{
    const unsigned long long want = (unsigned long long)(node + 1u) | ((unsigned long long)q << 32);
    uint32_t h = batch_hash(node, q) >> t.shift;
    volatile uint32_t* fail = t.count + 1;
    for (uint32_t probes = 0; probes <= t.tmask; probes++) {
        unsigned long long* kp = reinterpret_cast<unsigned long long*>(t.ent + (size_t)h * EW);
        unsigned long long k = *reinterpret_cast<volatile unsigned long long*>(kp);
        if (k == 0ull) {
            if (*fail) return 0xFFFFFFFFu;
            k = atomicCAS(kp, 0ull, want);
            if (k == 0ull) {
                const uint32_t at = atomicAdd(t.count, 1u);
                if (at < t.limit) t.list[at] = h; else *fail = 1u;
                return h;
            }
        }
        if ((k & ~kBatchFlagBit) == want) return h;
        h = (h + 1) & t.tmask;
    }
    *fail = 1u;
    return 0xFFFFFFFFu;
}

struct BatchArgs {
    IterState* st;            // the handle's state: iteration counter, base, work queues, counters
    BatchQuery* qs;
    int nq, colony_max, items_per_query;
    BatchTable tab;
    const uint8_t* open6;     // per node: bit k <=> neighbour k in bounds and free (K = 6)
    const uint32_t* occ;      // K = 26: the grid's occupancy, one bit per node, 1 = occupied
    const float* coords;      // xs | ys | zs
    int rx, ry, rz;
    uint32_t seed_lo, seed_hi;
    int alpha;
    float beta;
    int cap;
    int* ant_steps;           // [nq][colony_max]
    uint32_t* path_ids;       // [nq][colony_max][cap]
    uint8_t* path_dirs;
    int table_entries;        // shared-memory visited-tile entries per ant (pass 1)
    uint32_t* overflow_list;  // [pool] (query * colony_max + ant) of the parked ants
    unsigned long long* gtab; // [pool][1 << gtable_log2] HBM visited tables (K = 26: their masks)
    int gtable_log2;
    int4* resume;             // [pool]
    uint32_t pool;
    // K = 26 (batch26.cuh)
    int table_log2;           // shared-memory visited-tile table of an ant: 1 << table_log2 entries (pass 1)
    uint32_t* gkeys;          // [pool][1 << gtable_log2] tile keys of the HBM visited tables (masks in gtab)
    float precision;          // step lengths precision, precision*1.414f, precision*1.732f
    float* ant_L;             // [nq][colony_max] length of every ant, +inf if it died
};

// Inputs of a K = 6 walk over a batch: k_walk_batch3 (pass 1) and k_walk2<Batch6> (pass 2, the parked ants).
//   * tau: the node's (query, node) entry, or the scalar if it has none;
//   * the geometric factor: heur6 from the three axis tables, per step;
//   * open: the grid's one byte per node (grid.cu k_open6).
// issue() sends the loads of a step (first probe of the entry, open byte, coordinates) out as soon as the node is known,
// resolve() finishes them when the step needs them.
struct Batch6 {
    using Args = BatchArgs;
    // this lane
    int k, kk6;
    int axis_k, dk, axis_len;         // axis of the slot: 0 = x (slots 2, 3), 1 = y (slots 1, 4), 2 = z (slots 0, 5); -1 / +1 along it (0 for the idle lanes)
    const float *xs, *ys, *zs, *axis_tab;
    const uint32_t* ent;
    const uint8_t* open6;
    int shift;
    uint32_t tmask;
    float beta;
    int rx, rxy;
    // the bound query and ant
    uint32_t qi, qhash;
    float gxv, gyv, gzv;              // goal coordinates (vector_a = goal - node, :151)
    int start, goal;
    uint32_t ant, stream_word, block_hi;
    size_t row;
    // the current step
    uint32_t want0, eh, etau, omask;
    uint2 ekey;
    float cxv, cyv, czv, nbv;

    __device__ __forceinline__ Batch6(const BatchArgs& a, int k_)
        : k(k_), kk6(k_ < 6 ? k_ : 5), ent(a.tab.ent), open6(a.open6), shift(a.tab.shift), tmask(a.tab.tmask), beta(a.beta), rx(a.rx), rxy(a.rx * a.ry)
    {
        const int dxk = (k == 3) - (k == 2), dyk = (k == 4) - (k == 1), dzk = (k == 5) - (k == 0);
        axis_k = (k == 2 || k == 3) ? 0 : ((k == 1 || k == 4) ? 1 : 2);
        dk = dxk + dyk + dzk;
        xs = a.coords;
        ys = xs + a.rx;
        zs = ys + a.ry;
        axis_tab = axis_k == 0 ? xs : (axis_k == 1 ? ys : zs);
        axis_len = axis_k == 0 ? a.rx : (axis_k == 1 ? a.ry : a.rz);
    }
    __device__ __forceinline__ const BatchQuery& query(const BatchArgs& a, uint32_t q)
    {
        qi = q;
        qhash = q * 0x85EBCA6Bu + (q << 13);
        const BatchQuery& bq = a.qs[q];
        const int g = bq.goal;
        gxv = __ldg(xs + g % rx); gyv = __ldg(ys + (g % rxy) / rx); gzv = __ldg(zs + g / rxy);
        return bq;
    }
    // parked ants to resume: those beyond the pool got no table (the batch has failed and will be re-run), as Batch26::items
    __device__ __forceinline__ unsigned items(const BatchArgs& a, const IterState* st) const { return min(st->overflow_n, a.pool); }
    // entry q of the parked-ant list (has = false: no ant, the group idles)
    __device__ __forceinline__ void bind(const BatchArgs& a, unsigned q, bool has)
    {
        const uint32_t ga = has ? a.overflow_list[q] : 0u;   // query * colony_max + ant
        const uint32_t qq = ga / (uint32_t)a.colony_max;
        ant = ga - qq * (uint32_t)a.colony_max;
        const BatchQuery& bq = query(a, qq);
        start = bq.start; goal = bq.goal;
        stream_word = bq.stream_word; block_hi = bq.block_hi;
        row = (size_t)qq * a.colony_max + ant;
    }
    __device__ __forceinline__ void issue(int cur, uint32_t P)
    {
        want0 = (uint32_t)cur + 1u;
        eh = (((uint32_t)cur * 2654435761u) ^ qhash) >> shift;
        const uint32_t* e = ent + (size_t)eh * kBatchEntryWords;
        ekey = __ldg(reinterpret_cast<const uint2*>(e));
        etau = __ldg(e + 2 + kk6);
        omask = (uint32_t)__ldg(open6 + cur);
        const int x = (int)(P & 1023u), y = (int)((P >> 10) & 1023u), z = (int)((P >> 20) & 1023u);   // bits 30-31 may carry a key tag
        cxv = __ldg(xs + x); cyv = __ldg(ys + y); czv = __ldg(zs + z);
        const int ci = (axis_k == 0 ? x : (axis_k == 1 ? y : z)) + dk;
        nbv = __ldg(axis_tab + min(max(ci, 0), axis_len - 1));
    }
    __device__ __forceinline__ Slot6 resolve()
    {
        Slot6 s;
        s.open = k < 6 && ((omask >> k) & 1u);
        // ---- geometric factor of slot k, k_heuristic's expressions ----
        const float ax = __fsub_rn(gxv, cxv), ay = __fsub_rn(gyv, cyv), az = __fsub_rn(gzv, czv);
        const float na = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(ax, ax), __fmul_rn(ay, ay)), __fmul_rn(az, az)));
        const float cc = axis_k == 0 ? cxv : (axis_k == 1 ? cyv : czv);
        const float ac = axis_k == 0 ? ax : (axis_k == 1 ? ay : az);
        s.heur = heur6(ac, __fsub_rn(nbv, cc), na, beta);
        // ---- pheromone of slot k: the node's entry, or the scalar if it has none ----
        uint32_t probes = 0;
        while ((ekey.x != want0 || (ekey.y & 0x7FFFFFFFu) != qi) && (ekey.x | ekey.y) != 0u) {   // rare: linear probing at load <= 1/2
            if (++probes > tmask) { ekey = make_uint2(0u, 0u); break; }   // a full table: only in a batch that has already failed and will be re-run
            eh = (eh + 1) & tmask;
            const uint32_t* e = ent + (size_t)eh * kBatchEntryWords;
            ekey = __ldg(reinterpret_cast<const uint2*>(e));
            etau = __ldg(e + 2 + kk6);
        }
        s.tau = (ekey.x | ekey.y) != 0u ? __uint_as_float(etau) : __uint_as_float(kSentinelBits);
        return s;
    }
};

template <int EW>
__global__ void k_batch_fill(uint4* __restrict__ ent4, size_t n_entries)
{   // keys 0, every slot (and the unused words of a K = 26 entry) the sentinel
    const uint4 a = make_uint4(0u, 0u, kSentinelBits, kSentinelBits), b = make_uint4(kSentinelBits, kSentinelBits, kSentinelBits, kSentinelBits);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_entries; i += (size_t)gridDim.x * blockDim.x) {
        ent4[EW / 4 * i] = a;
#pragma unroll
        for (int j = 1; j < EW / 4; j++) ent4[EW / 4 * i + j] = b;
    }
}
// after a batch: only the claimed entries need restoring
template <int EW>
__global__ void k_batch_wipe(BatchTable t)
{
    const uint32_t n = min(t.count[0], t.limit);
    const uint4 a = make_uint4(0u, 0u, kSentinelBits, kSentinelBits), b = make_uint4(kSentinelBits, kSentinelBits, kSentinelBits, kSentinelBits);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint4* e = reinterpret_cast<uint4*>(t.ent + (size_t)t.list[i] * EW);
        e[0] = a;
#pragma unroll
        for (int j = 1; j < EW / 4; j++) e[j] = b;
    }
}

__global__ void k_batch_begin(IterState* st, BatchQuery* qs, int nq, const long long* __restrict__ starts, const long long* __restrict__ goals, uint32_t first_search,
                              float predict, float tau0, uint32_t* count)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q == 0) {
        st->iter = 0; st->predict = predict; st->base = tau0;
        st->queue = 0; st->queue2 = 0; st->overflow_n = 0;
        count[0] = 0; count[1] = 0; count[2] = 0;
    }
    if (q >= nq) return;
    BatchQuery b;
    b.start = (int)starts[q]; b.goal = (int)goals[q];
    const uint32_t search = first_search + (uint32_t)q;
    b.stream_word = kStreamAcs3D + (search & 0xFFFFu); b.block_hi = (search >> 16) << 16;
    b.colony = 0; b.lambda = 0; b.Q = 0;
    b.best_steps = INT_MAX; b.best_L = INFINITY; b.best_changed = 0; b.best_ant = -1; b.n_eligible = 0; b.best_n = 0; b.pad = 0;
    qs[q] = b;
}

__global__ void k_batch_iter_begin(IterState* st, BatchQuery* qs, int nq, int fixed_colony, int colony_max, float precision, float tau0, int advance, float rho)
{   // :247-249 per query (the expressions of k_iter_begin)
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q == 0) {
        if (advance) { st->iter++; st->base = __fmul_rn(st->base, rho); }
        st->cnt[6] += (unsigned long long)nq;   // one ACS iteration per query
        st->queue = 0; st->queue2 = 0; st->overflow_n = 0;
    }
    if (q >= nq) return;
    BatchQuery& b = qs[q];
    const float best_L = b.best_L, predict = st->predict;
    int colony = fixed_colony > 0 ? fixed_colony : (int)(0.35 * (double)(best_L < predict ? best_L : predict) / (double)precision);
    colony = max(0, min(colony, colony_max));
    const float lambda = (float)(0.2 * (double)colony);
    b.colony = colony; b.lambda = lambda;
    b.Q = __fmul_rn(__fdiv_rn(tau0, lambda), (best_L == INFINITY ? predict : best_L));
    b.best_changed = 0; b.n_eligible = 0;
}

// ------------------------------------------------------------------------------------------
// Pass 1 of K2 over a batch, restructured like k_walk3 (walk3.cuh): the four ants of a warp are at the same step index, so
// four steps per trip with the draw chosen at compile time, Philox for the next four steps computed in slices beside them, the
// trail kept in registers and written eight steps at a time, the visited insert a predicated store by the lane whose pick is
// the highest, the tile count fed by one vote, outcomes reconstructed after the loop.  Its inputs — pheromone entry or scalar,
// geometric factor, open mask — come from Batch6, as in pass 2 (k_walk2<Batch6>, parked ants), so every ant is bit-identical.
// This kernel is issue-bound once a few hundred queries are in flight (60 % of the issue
// slots), so the shorter instruction stream is throughput.
// ------------------------------------------------------------------------------------------
// Register allocation bounded for five CTAs per SM (102 registers): measured best on C5 — 2027 queries/s, against 1934 with six
// (80 registers, spills) and 1854 with four (120).
template <bool ALPHA1>
__global__ void __launch_bounds__(kWalkThreads, 5) k_walk_batch3(BatchArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    int4* move_lut = reinterpret_cast<int4*>(smem_raw);
    unsigned long long* tab_s = reinterpret_cast<unsigned long long*>(smem_raw + kWalk2Lut + 128);
    if (threadIdx.x < 64) {
        const int pbv = threadIdx.x;
        const int c = pbv ? 31 - __clz(pbv) : 0;
        const int dx = (c == 3) - (c == 2), dy = (c == 4) - (c == 1), dz = (c == 5) - (c == 0);
        move_lut[pbv] = pbv ? make_int4(dx + dy * a.rx + dz * a.rx * a.ry, dx + dy * 1024 + dz * 1048576, c, 0) : make_int4(0, 0, 0, 0);
    }
    __syncthreads();

    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int gbase = lane & 24;
    const int k = lane & 7;
    const int g = threadIdx.x >> 3;
    const int E = a.table_entries;
    uint32_t lut_sa = (uint32_t)__cvta_generic_to_shared(move_lut);
    TabRef<false> tab;
    tab.gp = nullptr;
    tab.sa = (uint32_t)__cvta_generic_to_shared(tab_s + (size_t)g * E);
    uint32_t gmask = 0xFFu << gbase;
    uint32_t lut_rot = (uint32_t)(gbase - 4) & 31u;
    asm volatile("" : "+r"(lut_sa), "+r"(tab.sa), "+r"(gmask), "+r"(lut_rot));

    const int rx = a.rx, rxy = a.rx * a.ry;
    const int dxk = (k == 3) - (k == 2), dyk = (k == 4) - (k == 1), dzk = (k == 5) - (k == 0);
    const uint32_t dPk = (uint32_t)(dxk + dyk * 1024 + dzk * 1048576);
    Batch6 in(a, k);
    uint32_t m4 = k <= 4 ? ~0u : 0u, m3 = k <= 3 ? ~0u : 0u, m2 = k <= 2 ? ~0u : 0u, m1 = k <= 1 ? ~0u : 0u, m0 = k <= 0 ? ~0u : 0u;
    asm volatile("" : "+r"(m4), "+r"(m3), "+r"(m2), "+r"(m1), "+r"(m0));
    constexpr uint32_t kKeyMask = kPackKey | kKeyTag;

    IterState* st = a.st;
    const uint32_t iter = (uint32_t)st->iter;
    const float base_now = st->base;
    const unsigned n_items = (unsigned)(a.nq * a.items_per_query);
    const uint32_t limit = (uint32_t)((E >> 2) * 3);
    const int cap = a.cap;
    int cap_k = k < 6 ? cap : 0;   // the two idle lanes of a group are never alive
    asm volatile("" : "+r"(cap_k));

    unsigned long long c_steps = 0, c_ants = 0, c_arrived = 0, c_nocand = 0, c_fall = 0, c_cap = 0, c_over = 0;

    while (true) {
        unsigned q0 = 0;
        if (lane == 0) q0 = atomicAdd(&st->queue, 1u);
        q0 = __shfl_sync(FULL, q0, 0);
        if (q0 >= n_items) break;                                    // warp-uniform
        const uint32_t qi = q0 / (unsigned)a.items_per_query;        // work item = (query, group of four ants)
        const int ant = (int)(q0 - qi * (unsigned)a.items_per_query) * 4 + (lane >> 3);
        const BatchQuery& bq = in.query(a, qi);
        const bool has = ant < bq.colony;
        const int start = bq.start, goal = bq.goal;
        const uint32_t stream_word = bq.stream_word, block_hi = bq.block_hi;

        const uint32_t Pstart = pack_xyz(start % rx, (start % rxy) / rx, start / rxy) | kKeyTag;   // bit 31: the key tag rides along
        for (int i = k; i < E; i += kGroup) tab.store(i, 0ull);
        __syncwarp();
        if (k == 0) {   // addStartNode :81-86
            const uint32_t key = Pstart & kKeyMask;
            const uint32_t bit = (((Pstart & kPackLow) * kPackMul) >> 20) & 31u;
            tab.store(tile_hash(key, (uint32_t)E), ((unsigned long long)key << 32) | (unsigned long long)(1u << bit));
        }
        __syncwarp();

        int cur = start, steps = 0;
        uint32_t P = Pstart;
        uint32_t ntiles = 1u, lastcb = 1u;
        bool parked = false;
        bool live = has && cap_k > 0;
        uint32_t T = 0, kt = (uint32_t)k;
        uint32_t rec_id = 0, rec_dir = 0;
        const size_t ant_row = ((size_t)qi * a.colony_max + (size_t)(has ? ant : 0)) * cap;
        uint32_t* pid = a.path_ids + ant_row;
        uint8_t* pdir = a.path_dirs + ant_row;

        float u0, u1, u2, u3;
        {
            uint32_t w0, w1, w2, w3;
            philox4(iter, (uint32_t)ant, block_hi, stream_word, a.seed_lo, a.seed_hi, w0, w1, w2, w3);
            u0 = __fmul_rn(__int2float_rn((int)(w0 >> 1)), 4.656612873077392578125e-10f);
            u1 = __fmul_rn(__int2float_rn((int)(w1 >> 1)), 4.656612873077392578125e-10f);
            u2 = __fmul_rn(__int2float_rn((int)(w2 >> 1)), 4.656612873077392578125e-10f);
            u3 = __fmul_rn(__int2float_rn((int)(w3 >> 1)), 4.656612873077392578125e-10f);
        }
        uint32_t pc0 = 0, pc1 = 0, pc2 = 0, pc3 = 0;
        auto rounds = [&](auto r0, auto r1) { philox_rounds<decltype(r0)::value, decltype(r1)::value>(pc0, pc1, pc2, pc3, a.seed_lo, a.seed_hi); };

        in.issue(cur, P);   // the loads of a step go out as soon as the node is known

        auto step = [&](const uint32_t J, const float u) {
            // ---- open, factor and pheromone of slot k ------------------------------------------------------------------
            const Slot6 sl = in.resolve();
            const bool open_k = sl.open;
            // ---- neighbour k: tabu probe -------------------------------------------------------------------------------
            const uint32_t Pk = P + dPk;
            const uint32_t key = Pk & kKeyMask;
            const uint32_t bitm = 1u << ((((Pk & kPackLow) * kPackMul) >> 20) & 31u);
            unsigned slot = tile_hash(key, (uint32_t)E);
            unsigned long long e = tab.load(slot);
            while (open_k && (uint32_t)(e >> 32) != key && (uint32_t)(e >> 32) != 0u) {
                slot = slot + 1 < (unsigned)E ? slot + 1 : 0u;
                e = tab.load(slot);
            }
            const bool found = (uint32_t)(e >> 32) == key;
            const uint32_t emask = found ? (uint32_t)e : 0u;
            const bool cand = live && open_k && !(emask & bitm);
            const float tau_now = tau_or_base(sl.tau, base_now);
            const float tpow = ALPHA1 ? tau_now : pow_int(tau_now, a.alpha);
            const float info = cand ? __fmul_rn(tpow, sl.heur) : 0.0f;
            // ---- roulette in the reference's order (:155, :172-181) ---------------------------------------------------
            const unsigned cb = __ballot_sync(FULL, cand) & gmask;
            const float v0 = __shfl_sync(FULL, info, 0, 8), v1 = __shfl_sync(FULL, info, 1, 8), v2 = __shfl_sync(FULL, info, 2, 8);
            const float v3 = __shfl_sync(FULL, info, 3, 8), v4 = __shfl_sync(FULL, info, 4, 8), v5 = __shfl_sync(FULL, info, 5, 8);
            const float total = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(0.0f, v0), v1), v2), v3), v4), v5);
            const float rnd = __fmul_rn(u, total);
            float mine = __fadd_rn(0.0f, v5);
            mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v4) & m4));
            mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v3) & m3));
            mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v2) & m2));
            mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v1) & m1));
            mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v0) & m0));
            const bool pick = cand && (mine >= rnd);
            const unsigned pball = __ballot_sync(FULL, pick);
            int4 mv;   // a dead or finished ant has no pick and the table's entry 0 moves nowhere
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(mv.x), "=r"(mv.y), "=r"(mv.z), "=r"(mv.w) : "r"(lut_sa + (__funnelshift_r(pball, pball, lut_rot) & 0x3F0u)) : "memory");
            const unsigned pb = (pball >> gbase) & 0x3Fu;
            const uint32_t prev = (uint32_t)cur;
            cur += mv.x;
            P += (uint32_t)mv.y;
            in.issue(cur, P);
            // ---- side effects, all predicated --------------------------------------------------------------------------
            const bool stepok = pb != 0u;
            const bool win = pick && (pb >> k) == 1u;
            if (win) tab.store(slot, ((unsigned long long)key << 32) | (unsigned long long)(emask | bitm));
            if (stepok && kt == J) { rec_id = prev; rec_dir = (uint32_t)mv.z; }
            const bool full = ntiles > limit;
            const unsigned nt = __ballot_sync(FULL, win && !found) & gmask;
            ntiles += nt ? 1u : 0u;
            lastcb = live ? cb : lastcb;
            steps = stepok ? (int)(T + J + 1u) : steps;
            const bool go = stepok && cur != goal;
            parked = parked || (go && full);
            live = go && !full && (int)(T + J + 1u) < cap_k;
            __syncwarp();
        };

        while (__any_sync(FULL, live)) {
            pc0 = iter; pc1 = (uint32_t)ant; pc2 = ((T >> 2) + 1u) | block_hi; pc3 = stream_word;
            step(0u, u0); rounds(IC<0>{}, IC<3>{});
            step(1u, u1); rounds(IC<3>{}, IC<6>{});
            step(2u, u2); rounds(IC<6>{}, IC<9>{});
            step(3u, u3); rounds(IC<9>{}, IC<10>{});
            u0 = __fmul_rn(__int2float_rn((int)(pc0 >> 1)), 4.656612873077392578125e-10f);
            u1 = __fmul_rn(__int2float_rn((int)(pc1 >> 1)), 4.656612873077392578125e-10f);
            u2 = __fmul_rn(__int2float_rn((int)(pc2 >> 1)), 4.656612873077392578125e-10f);
            u3 = __fmul_rn(__int2float_rn((int)(pc3 >> 1)), 4.656612873077392578125e-10f);
            if (T & 4u) {
                const int base8 = (int)T - 4;
                if (k < steps - base8) { pid[base8 + k] = rec_id; pdir[base8 + k] = (uint8_t)rec_dir; }
            }
            T += 4u;
            kt ^= 4u;
        }
        if (T & 4u) {
            const int base8 = (int)T - 4;
            if (k < steps - base8) { pid[base8 + k] = rec_id; pdir[base8 + k] = (uint8_t)rec_dir; }
        }
        const bool arrived = has && steps > 0 && cur == goal;
        const int result = arrived ? steps : (parked ? -2 : -1);
        int reason = 0;
        if (result == -1) reason = steps >= cap ? 3 : (lastcb == 0u ? 1 : 2);

        {   // park the ants whose shared-memory table filled up (k_walk2<Batch6> resumes them); HBM tables come from a pool
            const bool pk = has && parked && !arrived;
            const unsigned pm = __ballot_sync(FULL, pk && k == 0);
            if (pm) {
                int o = 0;
                if (pk && k == 0) o = (int)atomicAdd(&st->overflow_n, 1u);
                o = __shfl_sync(FULL, o, 0, 8);
                const bool fits = (uint32_t)o < a.pool;
                if (pk && !fits && k == 0) a.tab.count[1] = 1u;
                const int Eg = 1 << a.gtable_log2;
                for (unsigned rest = pm; rest; rest &= rest - 1) {
                    const int src = __ffs(rest) - 1;
                    const int oo = __shfl_sync(FULL, o, src);
                    if ((uint32_t)oo >= a.pool) continue;   // warp-uniform
                    uint4* z = reinterpret_cast<uint4*>(a.gtab + (size_t)oo * Eg);
                    for (int i = lane; i < Eg / 2; i += 32) z[i] = make_uint4(0u, 0u, 0u, 0u);
                }
                __syncwarp();
                if (pk && fits) {
                    unsigned long long* ntab = a.gtab + (size_t)o * Eg;
                    for (int i = k; i < E; i += kGroup) {
                        const unsigned long long t = tab.load(i);
                        if (t == 0ull) continue;
                        unsigned sl = tile_hash((uint32_t)(t >> 32), (uint32_t)Eg);
                        while (atomicCAS(&ntab[sl], 0ull, t) != 0ull) sl = (sl + 1) & (Eg - 1);
                    }
                    if (k == 0) {
                        a.resume[o] = make_int4(cur, steps, 0, 0);
                        a.overflow_list[o] = qi * (uint32_t)a.colony_max + (uint32_t)ant;
                    }
                }
                __syncwarp();
            }
        }
        if (has) {
            if (result == -2) {
                c_over++;
            } else {
                c_arrived += result >= 0 ? 1 : 0;
                c_nocand += reason == 1 ? 1 : 0;
                c_fall += reason == 2 ? 1 : 0;
                c_cap += reason == 3 ? 1 : 0;
                c_steps += (unsigned long long)steps; c_ants++;
            }
            if (k == 0) a.ant_steps[(size_t)qi * a.colony_max + ant] = result;
        }
        __syncwarp();
    }
    if (k == 0) {
        if (c_steps) atomicAdd(&st->cnt[0], c_steps);
        if (c_ants) atomicAdd(&st->cnt[1], c_ants);
        if (c_arrived) atomicAdd(&st->cnt[2], c_arrived);
        if (c_nocand) atomicAdd(&st->cnt[3], c_nocand);
        if (c_fall) atomicAdd(&st->cnt[4], c_fall);
        if (c_cap) atomicAdd(&st->cnt[5], c_cap);
        if (c_over) atomicAdd(&st->cnt[8], c_over);
    }
}

// ------------------------------------------------------------------------------------------
// Ranking, best decision and best path of every query: one CTA per query.
// dynamic shared memory: keys[2][maxn] (u32) + vals[2][maxn] (u16) + whist[32][256] (u32)
// ------------------------------------------------------------------------------------------
// EW = kBatchEntryWords26 (K = 26): keys are the bits of each query's ant_L row, as k_rank_small's K = 26 branch (ant_L is
// unused for K = 6).
template <int EW>
__global__ void __launch_bounds__(kRankSmallThreads) k_batch_rank(IterState* st, BatchQuery* qs, BatchTable tab, const int* __restrict__ ant_steps,
                                                                   const float* __restrict__ ant_L, int colony_max, int maxn,
                                                                   int cap, int key_bits, const float* __restrict__ Ltab, uint32_t* __restrict__ ranked_keys,
                                                                   uint16_t* __restrict__ ranked_vals, const uint32_t* __restrict__ path_ids,
                                                                   const uint8_t* __restrict__ path_dirs, uint32_t* __restrict__ best_ids, uint8_t* __restrict__ best_dirs)
{
    extern __shared__ __align__(16) uint32_t rs_smem[];
    uint32_t* kbuf[2] = {rs_smem, rs_smem + maxn};
    uint16_t* vbase = reinterpret_cast<uint16_t*>(rs_smem + 2 * maxn);
    uint16_t* vbuf[2] = {vbase, vbase + maxn};
    uint32_t* whist = rs_smem + 3 * maxn;
    __shared__ uint32_t warp_sum[32];
    __shared__ int s_elig, s_changed, s_old_n;
    const uint32_t q = blockIdx.x;
    BatchQuery& b = qs[q];
    const int n = b.colony;
    const int* steps_q = ant_steps + (size_t)q * colony_max;
    const float* L_q = EW == kBatchEntryWords26 ? ant_L + (size_t)q * colony_max : nullptr;
    const int src = rank_sort_chunk(kbuf, vbuf, whist, warp_sum, steps_q, L_q, 0, n, cap, key_bits);
    const uint32_t* keys = kbuf[src];
    const uint16_t* vals = vbuf[src];
    const float lambda = b.lambda;
    if (threadIdx.x == 0) {
        s_elig = 0; s_changed = 0; s_old_n = b.best_n;
        if (n > 0 && L_q) {
            const float L0 = __uint_as_float(keys[0]);
            if (L0 < b.best_L) {   // agentK.L < best.L  (:263) on the float lengths
                b.best_steps = steps_q[vals[0]]; b.best_L = L0; b.best_changed = 1; b.best_ant = (int)vals[0];
                s_changed = 1;
            }
        } else if (n > 0) {
            const int s = (int)keys[0];
            if (s <= cap && s < b.best_steps) {   // agentK.L < best.L  (:263); ties keep the earlier best, the first of equal ants wins
                b.best_steps = s; b.best_L = Ltab[s]; b.best_changed = 1; b.best_ant = (int)vals[0];
                s_changed = 1;
            }
        }
    }
    __syncthreads();
    int local = 0;
    for (int r = threadIdx.x; r < n; r += kRankSmallThreads) {
        const uint32_t key = keys[r];
        ranked_keys[(size_t)q * colony_max + r] = key;
        ranked_vals[(size_t)q * colony_max + r] = vals[r];
        const bool arrived = L_q ? key != 0x7F800000u : (int)key <= cap;
        local += (arrived && !((float)(r + 1) > __fsub_rn(lambda, 1.0f))) ? 1 : 0;   // :200
    }
    if (local) atomicAdd(&s_elig, local);
    __syncthreads();
    if (threadIdx.x == 0) {
        b.n_eligible = s_elig;
        unsigned long long recs = 0;
        for (int r = 0; r < s_elig; r++) recs += L_q ? (unsigned long long)steps_q[vals[r]] : keys[r];   // eligible ranks are a prefix of the sorted colony
        atomicAdd(&st->cnt[7], recs);
    }
    if (!s_changed) return;   // CTA-uniform
    // best = agentK (:264): the old path's nodes lose their membership flag, the new path's get it (entries are created for
    // nodes that have none: their slots stay sentinels, i.e. worth the scalar)
    uint32_t* bi = best_ids + (size_t)q * (cap + 1);
    uint8_t* bd = best_dirs + (size_t)q * (cap + 1);
    for (int i = threadIdx.x; i < s_old_n; i += kRankSmallThreads) {
        const uint32_t h = batch_find<EW>(tab, bi[i], q);
        if (h != 0xFFFFFFFFu) atomicAnd(reinterpret_cast<unsigned long long*>(tab.ent + (size_t)h * EW), ~kBatchFlagBit);
    }
    __syncthreads();
    const int steps = b.best_steps;
    const size_t off = ((size_t)q * colony_max + (size_t)b.best_ant) * cap;
    for (int i = threadIdx.x; i <= steps; i += kRankSmallThreads) {
        const uint32_t id = i < steps ? path_ids[off + i] : (uint32_t)b.goal;
        bi[i] = id;
        if (i < steps) bd[i] = path_dirs[off + i];
        const uint32_t h = batch_find_or_insert<EW>(tab, id, q);
        if (h != 0xFFFFFFFFu) atomicOr(reinterpret_cast<unsigned long long*>(tab.ent + (size_t)h * EW), kBatchFlagBit);
    }
    if (threadIdx.x == 0) b.best_n = steps + 1;
}

template <int EW>
__global__ void __launch_bounds__(256) k_batch_evaporate(BatchTable t, float rho)
{   // :268-272 for every slot that ever received a deposit (sentinels are -0: unchanged by the product)
    const uint32_t n = min(t.count[0], t.limit);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint32_t* e = t.ent + (size_t)t.list[i] * EW;
        constexpr int end = EW == kBatchEntryWords26 ? 2 + 26 : 2 + 6;   // slots are words [2, end): two, then groups of four
        float2 a = *reinterpret_cast<float2*>(e + 2);
        a.x = __fmul_rn(a.x, rho); a.y = __fmul_rn(a.y, rho);
        *reinterpret_cast<float2*>(e + 2) = a;
#pragma unroll
        for (int j = 4; j < end; j += 4) {
            float4 b = *reinterpret_cast<float4*>(e + j);
            b.x = __fmul_rn(b.x, rho); b.y = __fmul_rn(b.y, rho); b.z = __fmul_rn(b.z, rho); b.w = __fmul_rn(b.w, rho);
            *reinterpret_cast<float4*>(e + j) = b;
        }
    }
}

// update_pheromone (:198-215) of every query; value = (lambda - order)*Q/L_ant + float(onBest)*lambda*Q/L_best (:210-211)
// EW = kBatchEntryWords26 (K = 26): ranked_keys hold the bits of the ant's L, its step count is steps26[query][ant] (unused
// for K = 6)
constexpr int kBatchDepThreads = 256;
template <int EW>
__global__ void __launch_bounds__(kBatchDepThreads) k_batch_deposit(const IterState* st, const BatchQuery* __restrict__ qs, BatchTable tab,
                                                                     const uint32_t* __restrict__ ranked_keys, const uint16_t* __restrict__ ranked_vals, int colony_max,
                                                                     const uint32_t* __restrict__ path_ids, const uint8_t* __restrict__ path_dirs, int cap,
                                                                     const float* __restrict__ Ltab, float rho, const int* __restrict__ steps26 = nullptr)
{
    __shared__ uint8_t s_flag[kBatchDepThreads + 1];
    const uint32_t q = blockIdx.x;
    const BatchQuery& b = qs[q];
    const int n = b.n_eligible;
    if (n == 0) return;
    const float base_new = __fmul_rn(st->base, rho);   // what a slot without a deposit is worth after this iteration's evaporation
    const float lambda = b.lambda, Q = b.Q;
    const float elite = __fdiv_rn(__fmul_rn(__fmul_rn(1.0f, lambda), Q), b.best_L);
    const uint32_t goal = (uint32_t)b.goal;
    for (int r = 0; r < n; r++) {
        const int ant = (int)ranked_vals[(size_t)q * colony_max + r];
        const uint32_t key = ranked_keys[(size_t)q * colony_max + r];
        constexpr bool k26 = EW == kBatchEntryWords26;
        const int steps = k26 ? steps26[(size_t)q * colony_max + ant] : (int)key;
        const float L_ant = k26 ? __uint_as_float(key) : Ltab[steps];
        const float base = __fdiv_rn(__fmul_rn(__fsub_rn(lambda, (float)(r + 1)), Q), L_ant);
        const float with_elite = __fadd_rn(base, elite), without = __fadd_rn(base, 0.0f);
        const size_t off = ((size_t)q * colony_max + (size_t)ant) * cap;
        for (int i0 = 0; i0 < steps; i0 += kBatchDepThreads) {   // CTA-uniform trips
            const int i = i0 + (int)threadIdx.x;
            uint32_t h = 0xFFFFFFFFu;
            bool f = false;
            if (i < steps) {
                h = batch_find_or_insert<EW>(tab, path_ids[off + i], q);
                if (h != 0xFFFFFFFFu) f = (tab.ent[(size_t)h * EW + 1] >> 31) != 0u;
            }
            s_flag[threadIdx.x] = f ? 1 : 0;
            if (threadIdx.x == 0) {   // membership of the node that follows this trip's last step
                const int j = i0 + kBatchDepThreads;
                bool fn = false;
                if (j <= steps) {
                    const uint32_t hn = batch_find<EW>(tab, j < steps ? path_ids[off + j] : goal, q);
                    fn = hn != 0xFFFFFFFFu && (tab.ent[(size_t)hn * EW + 1] >> 31) != 0u;
                }
                s_flag[kBatchDepThreads] = fn ? 1 : 0;
            }
            __syncthreads();
            if (i < steps && h != 0xFFFFFFFFu) {
                bool next_on;
                if (i + 1 < i0 + kBatchDepThreads && i + 1 < steps) next_on = s_flag[threadIdx.x + 1] != 0;
                else if (i + 1 == i0 + kBatchDepThreads) next_on = s_flag[kBatchDepThreads] != 0;
                else {   // i + 1 == steps: the goal
                    const uint32_t hn = batch_find<EW>(tab, goal, q);
                    next_on = hn != 0xFFFFFFFFu && (tab.ent[(size_t)hn * EW + 1] >> 31) != 0u;
                }
                float* slot = reinterpret_cast<float*>(tab.ent + (size_t)h * EW + 2) + path_dirs[off + i];   // direction 0..5 or 0..25
                *slot = __fadd_rn(tau_or_base(*slot, base_new), (f && next_on) ? with_elite : without);
            }
            __syncthreads();   // the next ant (or trip) may touch the same node's entry
        }
    }
}

// results of every query: L and node count (the path itself is the query's row of best_ids / best_dirs)
__global__ void k_batch_results(const BatchQuery* __restrict__ qs, int nq, float* __restrict__ res_L, int* __restrict__ res_n)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const BatchQuery& b = qs[q];
    res_L[q] = b.best_L;
    res_n[q] = b.best_steps != INT_MAX ? b.best_n : 0;
}

}  // namespace wr
