// Device kernels of the rank-based 3-D ant colony search (ACS_Rank, core/ACSRank_3D.hpp).
//   K2  k_walk2 (walk2.cuh) ant construction (selectNext :134-193 + the ant loop :252-265)
//   --  k_rank_*          colony ranking, best tracking (:263-264, :273-274)
//   --  k_deposit_gen     deposit records of update_pheromone (:198-215)
//   K3  k_update_fused    evaporation (:268-272) + rank-ordered deposits in ONE HBM pass (TMA)
//       k_evaporate / k_deposit_apply / atomic: the split variants
// All float arithmetic that reaches a comparison or the pheromone field uses explicit
// round-to-nearest intrinsics in the reference's operation order (no FMA contraction).
#pragma once
#include <limits.h>
#include <math.h>

#include "tma.cuh"
#include "wr_common.cuh"

namespace wr {

constexpr int kWalkThreads = 128;
constexpr int kGroup = 8;                                  // lanes per ant (6 neighbour lanes + 2 idle) for K = 6
constexpr int kAntsPerCta = kWalkThreads / kGroup;         // 16
constexpr uint32_t kEmptyKey = 0xFFFFFFFFu;
constexpr int kUpdTile = 4096;                             // floats per TMA tile (16 KB)
constexpr int kUpdStages = 4;
constexpr int kUpdThreads = 256;

// ------------------------------------------------------------------------------------------
// Clean-tile pheromone field.  The reference multiplies EVERY slot by rho every iteration (:268-272) — its wall-clock
// bottleneck — but a slot that never received a deposit holds the same value as every other such slot: tau0 after
// initFromGridMap/reset(), then fmul(.., rho) once per iteration.  That one float sequence is kept in IterState::base, the
// slots themselves hold the sentinel -0.0f (which no real pheromone value can be, and which rho leaves unchanged:
// -0 * rho = -0), and a 16 KB tile that holds nothing but sentinels (and the exact zeros of out-of-bounds slots) is
// "clean": the evaporation pass skips it — no read, no write.  A reader substitutes base for the sentinel (one select per
// walk step); the first deposit on a slot starts its chain from the base of that iteration, exactly the value the
// reference's slot holds at that point, and marks the tile dirty for good.  Bits are identical by construction; what is
// saved is the traffic of every tile the colony never touched (most of a 512^3 field).
// The same rule holds per 128-byte line (32 slots), and that is the granule the passes skip at: a wandering colony leaves
// scattered single deposits in ~40 % of the tiles but only ~8 % of the lines, and the set stops growing once the colony
// converges.  Every writer of a non-sentinel value marks the slot's line AND its tile (plain byte stores of 1, no
// atomics); the tile byte is a summary (any of its lines dirty) that fieldStats() counts and the tile-level passes test.
// ------------------------------------------------------------------------------------------
constexpr uint32_t kSentinelBits = 0x80000000u;
__device__ __forceinline__ float tau_or_base(float v, float base) { return __float_as_uint(v) == kSentinelBits ? base : v; }

constexpr int kLineSlots = 32;                             // floats per 128-byte line
constexpr int kTileLines = kUpdTile / kLineSlots;          // 128 lines per tile
struct DirtyFlags {
    uint8_t* tile;   // [ntiles + 1]     1: some line of the tile is dirty
    uint8_t* line;   // [ntiles * 128]   1: the line holds (or held since the last reset()) a value that is not a sentinel
    __device__ __forceinline__ void mark(uint32_t slot) const { line[slot / (uint32_t)kLineSlots] = 1; tile[slot / (uint32_t)kUpdTile] = 1; }
};

struct WalkArgs {
    IterState* st;
    const float* tau;        // [N][6] node-major ("edge-major": a node's 6 directed slots are contiguous)
    const float* heur;       // [N][6]  1 + beta*cos(theta) per directed slot for the current goal (k_heuristic)
    const float* closed_marker;   // one float = kClosedSlot (k_walk2's idle lanes read it)
    const float* coords;     // xs | ys | zs
    int rx, ry, rz;
    int start, goal;
    uint32_t seed_lo, seed_hi;
    uint32_t stream_word;    // Philox counter word 3: kStreamAcs3D + (search & 0xFFFF)   (search = index of this computeSolution on the handle)
    uint32_t block_hi;       // OR-ed into counter word 2 (step >> 2): (search >> 16) << 16
    int alpha;
    float beta;
    int cap;                 // max steps per ant
    int shard_first, shard_chunk;  // this rank constructs global ants [first, first+chunk) /\ [0, colony)
    int* ant_steps;          // [chunk]  steps, -1 dead, -2 pending (table overflow -> pass 2)
    uint32_t* path_ids;      // [chunk][cap]   node the ant stood on before step i
    uint8_t* path_dirs;      // [chunk][cap]   slot chosen at step i
    int table_log2;          // K = 26: shared-memory visited-tile table size of pass 1 (pass 2's HBM tables have 1 << gtable_log2)
    int table_entries;       // k_walk2: shared-memory visited-tile entries per ant (any size; the HBM tables of pass 2 have 1 << gtable_log2)
    uint32_t* overflow_list; // [chunk]
    uint32_t* gkeys;         // K = 26: tile keys of the HBM visited tables, one per overflowed ant: [chunk][1 << gtable_log2]
    unsigned long long* gtab;   // HBM visited tables: K = 6 64-bit key|mask entries, K = 26 the masks beside gkeys
    int gtable_log2;
    int4* resume;            // [chunk] state of an overflowed ant: {cur, steps, ntiles, bits of L (K = 26)}
    float precision;         // K = 26 (walk26.cuh): step lengths precision, precision*1.414f, precision*1.732f
    float* ant_L;            // K = 26: [chunk] length of the finished ant, +inf if it died (for K = 6 L is a function of steps)
    const uint32_t* best_ids;   // k_walk3: nodes of the best path so far, [cap + 16], every entry a valid node id (gather prediction)
    const int* verify_dev;   // k_walk3<*, 0>: [chunk] steps each ant followed the best path (k_path_verify), nullptr: walk from the start
    const int2* verify_n;    // {verifiable prefix D, best_n - 1 if the whole path verified else -1} (k_path_thresholds)
};

__device__ __forceinline__ float pow_int(float x, int y)
{   // power<T>() ACSRank_3D.hpp:48-60 (square-and-multiply, same multiplication order)
    float ans = 1.0f;
    while (y) {
        if (y & 1) ans = __fmul_rn(ans, x);
        x = __fmul_rn(x, x);
        y >>= 1;
    }
    return ans;
}

// ------------------------------------------------------------------------------------------
// Barrier between the ranks of a sharded colony, in peer memory (NVLink): every rank owns an array of epoch words, one
// per source rank, in its slab.  Rank `me` writes the barrier's epoch into word `me` of every peer's array (system-scope
// release: everything this rank's earlier kernels wrote — trails, step counts, published row blocks, final values — is
// visible to whoever acquires the word), then waits until every peer's word in its own array has reached the epoch.
// No host involvement, no collective library in the iteration loop.  The epoch is a function of the iteration counter
// (two barriers per iteration: 2*iter + 1 after the walk, 2*iter + 2 before the deposits are merged), the words restart at
// 0 with every exchange of the slabs (wr_acs_peer_export) — so the barrier needs no state of its own and lives INSIDE the
// kernel that consumes what it protects: its first CTAs signal (idempotent), every CTA waits before it touches peer
// data.  A peer that never arrives (its process died) would spin forever: after `timeout_ns` the CTA gives up, sets *err
// and the host reports it at the next synchronisation.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long global_timer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

struct PeerBarrier {
    uint32_t* const* flags_tab;   // [rank] -> that rank's epoch words
    int me, nranks;
    uint32_t* err;
    unsigned long long timeout_ns;
};

// all threads of the CTA call it; `which` = 1 or 2 (the barrier of this iteration)
__device__ __forceinline__ void peer_barrier(const PeerBarrier& b, const IterState* st, uint32_t which)
{
    const uint32_t e = 2u * (uint32_t)st->iter + which;
    const bool signals = blockIdx.x < 4;   // the first CTAs to be dispatched signal (idempotent; four of them so that one is certainly resident early)
    if (signals) __threadfence_system();
    for (int t = threadIdx.x; t < b.nranks; t += blockDim.x) {
        if (t == b.me) continue;
        if (signals) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(b.flags_tab[t] + b.me), "r"(e) : "memory");
        const uint32_t* mine = b.flags_tab[b.me] + t;
        const unsigned long long t0 = global_timer_ns();
        while (true) {
            uint32_t v;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
            if ((int)(v - e) >= 0) break;
            if (global_timer_ns() - t0 > b.timeout_ns) { *b.err = 1u; break; }
            __nanosleep(100);
        }
    }
    __syncthreads();
}

__global__ void k_begin(IterState* st, float predict)
{   // computeSolution :229-233
    st->iter = 0;
    st->predict = predict;
    st->best_steps = INT_MAX;
    st->best_L = INFINITY;
    st->best_changed = 0;
    st->best_ant = -1;
    st->colony = 0; st->lambda = 0; st->Q = 0;
    st->n_eligible = 0; st->n_records = 0; st->n_records_sort = 0;
    st->use_rankset = 0; st->spread_tiles = 0xFFFFFFFFu; st->spread_slots = 0xFFFFFFFFu; st->rankset_iters = 0;
    st->grp_rep = -1; st->grp_steps = 0; st->grp_ranks = 0; st->grp_ranks_total = 0;
}

// advance: the previous iteration's k_iter_end folded in (iterations enqueued back to back); upd_q: the fused update's
// three queue words, zeroed here instead of by a memset launch in front of k_tile_offsets.
// rankset_count != nullptr: adaptive handle (WR_UPDATE_RANKSET).  use_rankset is the HOST's choice for this iteration: rank
// sets pay off once the colony has converged on a few hundred slots, sorted records while it still wanders over ~10^6.
// What the choice is based on — how concentrated the previous iteration's deposits were — is measured here and
// published to the host through mapped pinned memory (a ring of records {generation << 16 | iteration, path, tiles, row
// blocks}); the host reads the record of the iteration that started kRsAhead iterations before the one it is enqueueing
// (that iteration has finished: acs.cu keeps itself at most four iterations ahead of the device), and only enqueues
// the kernels of the path it chose.  The choice is therefore a pure function of the search: identical on every rank of a
// sharded colony (whose protocol depends on it) and in every run.  Either path gives the same bits.
__global__ void k_iter_begin(IterState* st, int fixed_colony, int colony_max, float precision, float tau0, int advance = 0, uint32_t* upd_q = nullptr,
                             uint32_t* rankset_count = nullptr, int use_rankset = 0, volatile uint32_t* feedback = nullptr, uint32_t generation = 0,
                             float rho = 1.0f)
{   // :247-249
    if (advance) { st->iter++; st->cnt[6]++; st->base = __fmul_rn(st->base, rho); }
    st->grp_ranks_total += st->grp_ranks; st->grp_ranks = 0;   // the previous iteration's group deposits (k_rank_small)
    if (rankset_count) {
        const int prev = st->use_rankset;
        if (st->iter > 0) { if (prev) st->spread_slots = rankset_count[1]; else if (upd_q) st->spread_tiles = upd_q[2]; }
        st->use_rankset = use_rankset;
        if (use_rankset) st->rankset_iters++;
        rankset_count[0] = 0; rankset_count[3] = 0;   // claimed blocks, overflow flag
        if (feedback) {   // record of the iteration that starts now, in its slot of the ring (acs.cu reads the record of ONE specific iteration)
            volatile uint32_t* f = feedback + 4 * ((uint32_t)st->iter & 7u);
            f[1] = (uint32_t)prev; f[2] = st->spread_tiles; f[3] = st->spread_slots;
            __threadfence_system();
            f[0] = (generation << 16) | ((uint32_t)st->iter & 0xFFFFu);
        }
    }
    if (upd_q) { upd_q[0] = 0; upd_q[1] = 0; upd_q[2] = 0; upd_q[3] = 0; }
    float best_L = st->best_L, predict = st->predict;
    int colony = fixed_colony > 0 ? fixed_colony : (int)(0.35 * (double)(best_L < predict ? best_L : predict) / (double)precision);
    colony = max(0, min(colony, colony_max));
    float lambda = (float)(0.2 * (double)colony);
    float Q = __fmul_rn(__fdiv_rn(tau0, lambda), (best_L == INFINITY ? predict : best_L));
    st->colony = colony; st->lambda = lambda; st->Q = Q;
    st->queue = 0; st->queue2 = 0; st->overflow_n = 0; st->best_changed = 0;
    st->n_eligible = 0; st->n_records = 0;
}

__global__ void k_iter_end(IterState* st, float rho)
{
    st->iter++;
    st->cnt[6]++;
    st->base = __fmul_rn(st->base, rho);   // the evaporation (:268-272) of every slot that never received a deposit
}
__global__ void k_set_base(IterState* st, float v) { st->base = v; }


// ------------------------------------------------------------------------------------------
// Heuristic table for the current goal: heur[node][k] = 1 + beta*cos(theta), theta between (goal - node) and
// (neighbour_k - node) — selectNext :151-154, evaluated once per (node, slot) instead of once per ant-step.
// vector_b has a single non-zero component d, so dot(a,b) = a_c*d and |b| = sqrt(d*d) = |d| exactly (the zero
// terms add exactly; sqrt(RN(d*d)) == |d| in binary floating point unless d*d leaves the normal range, which
// takes the slow path).  NaN on duplicate-coordinate planes (d = 0 -> 0/0) is produced here and propagates
// through the roulette exactly like in the reference (SURVEY.md section 0.5).  A slot whose neighbour is out of
// bounds or occupied gets the sentinel -1, so the walk needs no separate open-neighbour mask.
// ------------------------------------------------------------------------------------------
__device__ __noinline__ float slow_norm1(float d) { return __fsqrt_rn(__fmul_rn(d, d)); }

constexpr float kClosedSlot = -1.0f;   // heur value of a slot whose neighbour is out of bounds or occupied (a real factor is >= 1 - beta or NaN)

// The factor of one slot: ac = the goal vector's component along the slot's axis, d = neighbour minus node on that axis,
// na = |goal - node|.  k_heuristic tabulates it, Batch6 (batch.cuh) evaluates it per step: one function, so the two
// cannot drift apart.
__device__ __forceinline__ float heur6(float ac, float d, float na, float beta)
{
    float nb = fabsf(d);
    if (!(nb >= 1e-18f && nb <= 1e18f) && nb != 0.0f) nb = slow_norm1(d);
    const float cosv = __fdiv_rn(__fmul_rn(ac, d), __fmul_rn(na, nb));
    return __fadd_rn(1.0f, __fmul_rn(beta, cosv));
}

__global__ void __launch_bounds__(256) k_heuristic(float* __restrict__ heur, const float* __restrict__ coords, const uint32_t* __restrict__ occ_bits,
                                                    int rx, int ry, int rz, unsigned long long N, int goal, float beta)
{
    const unsigned long long id = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= N) return;
    const float* xs = coords;
    const float* ys = xs + rx;
    const float* zs = ys + ry;
    const unsigned long long rxy = (unsigned long long)rx * ry;
    const int z = (int)(id / rxy), y = (int)((id % rxy) / rx), x = (int)(id % rx);
    const int gz = (int)(goal / rxy), gy = (int)((goal % rxy) / rx), gx = (int)(goal % rx);
    const float cx = xs[x], cy = ys[y], cz = zs[z];
    const float ax = __fsub_rn(xs[gx], cx), ay = __fsub_rn(ys[gy], cy), az = __fsub_rn(zs[gz], cz);
    const float na = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(ax, ax), __fmul_rn(ay, ay)), __fmul_rn(az, az)));
    float h[6];
#pragma unroll
    for (int k = 0; k < 6; k++) {
        const int dx = (k == 3) - (k == 2), dy = (k == 4) - (k == 1), dz = (k == 5) - (k == 0);
        const int nx = x + dx, ny = y + dy, nz = z + dz;
        const bool inb = nx >= 0 && nx < rx && ny >= 0 && ny < ry && nz >= 0 && nz < rz;
        const unsigned long long nid = id + dx + (long long)dy * rx + (long long)dz * (long long)rxy;
        // the neighbour must exist (:391-393) and be free (:148); the open mask is folded into the table
        const bool open = inb && !((occ_bits[nid >> 5] >> (nid & 31)) & 1u);
        float v = kClosedSlot;
        if (open) {
            const float ac = dx ? ax : (dy ? ay : az);
            const float d = dx ? __fsub_rn(xs[nx], cx) : (dy ? __fsub_rn(ys[ny], cy) : __fsub_rn(zs[nz], cz));
            v = heur6(ac, d, na, beta);
        }
        h[k] = v;
    }
    float2* o = reinterpret_cast<float2*>(heur + id * 6);
    o[0] = make_float2(h[0], h[1]); o[1] = make_float2(h[2], h[3]); o[2] = make_float2(h[4], h[5]);
}

// ------------------------------------------------------------------------------------------
// Ranking (:273-280) and best tracking (:263-264)
// ------------------------------------------------------------------------------------------
// The ranking itself lives in rank_small.cuh: key = steps for an ant that arrived, cap+1 for a dead one; value = ant index.
// L is a strictly increasing function of steps (L = precision added `steps` times, :78), so ordering by (steps, ant) is
// ordering by (L, ant), the oracle's total order.  best = agentK (:264): the ranking kernels drop the old best path's
// membership bits ...
// ... then copy the new one (path + chosen slots) and set its bits.  src_ids/src_dirs: the path
// buffers of the ant that produced it (local ant index src_ant).
__global__ void k_best_copy(const IterState* st, int* best_n, uint32_t* best_ids, uint8_t* best_dirs, uint32_t* onbest,
                            const uint32_t* __restrict__ path_ids, const uint8_t* __restrict__ path_dirs, int cap, int shard_first, int goal)
{
    if (!st->best_changed) return;
    const int steps = st->best_steps;
    const size_t off = (size_t)(st->best_ant - shard_first) * cap;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= steps; i += gridDim.x * blockDim.x) {
        uint32_t id = i < steps ? path_ids[off + i] : (uint32_t)goal;
        best_ids[i] = id;
        if (i < steps) best_dirs[i] = path_dirs[off + i];
        atomicOr(&onbest[id >> 5], 1u << (id & 31));
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *best_n = steps + 1;
}

// Peer-memory variant (sharded colonies on NVLink): the trail is read straight from the HBM of the rank that walked
// the ant — ids_tab[r] / dirs_tab[r] are rank r's trail buffers (peer pointers), chunk ants per rank.
__global__ void k_best_copy_peer(const IterState* st, int* best_n, uint32_t* best_ids, uint8_t* best_dirs, uint32_t* onbest,
                                 const uint32_t* const* __restrict__ ids_tab, const uint8_t* const* __restrict__ dirs_tab, int cap, int chunk, int goal)
{
    if (!st->best_changed) return;
    const int steps = st->best_steps;
    const int owner = st->best_ant / chunk;
    const size_t off = (size_t)(st->best_ant - owner * chunk) * cap;
    const uint32_t* path_ids = ids_tab[owner];
    const uint8_t* path_dirs = dirs_tab[owner];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= steps; i += gridDim.x * blockDim.x) {
        uint32_t id = i < steps ? path_ids[off + i] : (uint32_t)goal;
        best_ids[i] = id;
        if (i < steps) best_dirs[i] = path_dirs[off + i];
        atomicOr(&onbest[id >> 5], 1u << (id & 31));
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *best_n = steps + 1;
}

// ------------------------------------------------------------------------------------------
// Deposit records (:198-215).  One CTA per eligible rank; record i of rank r goes to
// rec_off[r] + i, so records are emitted in (rank, step) order and a STABLE sort by slot keeps
// rank order inside every slot — the order the reference adds them in.
//   value = (lambda - order)*Q/L_ant + float(onBest)*lambda*Q/L_best      (:210-211)
// ------------------------------------------------------------------------------------------
// PEER: ids_tab / dirs_tab name every rank's trail buffers (peer pointers over NVLink), so each rank generates the
// records of ALL eligible ants itself, in global (rank, step) order — no record exchange, no host-sized collective.
template <bool ATOMIC, bool PEER = false>
__global__ void __launch_bounds__(128) k_deposit_gen(const IterState* st, const uint32_t* __restrict__ rank_keys,
                                                      const uint32_t* __restrict__ rank_vals, const uint32_t* __restrict__ rec_off,
                                                      const uint32_t* __restrict__ path_ids, const uint8_t* __restrict__ path_dirs, int cap,
                                                      int shard_first, int shard_chunk,
                                                      int goal, const float* __restrict__ Ltab, const uint32_t* __restrict__ onbest,
                                                      uint32_t* __restrict__ rec_keys, uint32_t* __restrict__ rec_vals, float* tau,
                                                      const uint32_t* const* __restrict__ ids_tab = nullptr,
                                                      const uint8_t* const* __restrict__ dirs_tab = nullptr, int K = 6,
                                                      const int* __restrict__ steps26 = nullptr)
{   // steps26 != nullptr (K = 26): rank_keys holds the bits of the ant's L, its step count is steps26[ant]
    const int r = blockIdx.x;
    if (r >= st->n_eligible || st->use_rankset) return;   // use_rankset: this iteration's deposits go through rank sets (rankset.cuh)
    const int ant_global = (int)rank_vals[r];
    const int steps = steps26 ? steps26[ant_global] : (int)rank_keys[r];
    const float L_ant = steps26 ? __uint_as_float(rank_keys[r]) : Ltab[steps];
    if (PEER) {
        const int owner = ant_global / shard_chunk;
        path_ids = ids_tab[owner]; path_dirs = dirs_tab[owner];
        shard_first = owner * shard_chunk;
    } else if (ant_global < shard_first || ant_global >= shard_first + shard_chunk) return;   // another rank holds this trail
    const size_t ant = (size_t)(ant_global - shard_first);
    const int order = r + 1;
    const float lambda = st->lambda, Q = st->Q;
    const float base = __fdiv_rn(__fmul_rn(__fsub_rn(lambda, (float)order), Q), L_ant);
    const float elite = __fdiv_rn(__fmul_rn(__fmul_rn(1.0f, lambda), Q), st->best_L);
    const float with_elite = __fadd_rn(base, elite), without = __fadd_rn(base, 0.0f);
    const uint32_t off = rec_off[r];
    const uint32_t* pid = path_ids + ant * cap;
    const uint8_t* pdir = path_dirs + ant * cap;
    for (int i = threadIdx.x; i < steps; i += blockDim.x) {
        const uint32_t node = pid[i];
        const uint32_t next = (i + 1 < steps) ? pid[i + 1] : (uint32_t)goal;
        const bool onb = ((onbest[node >> 5] >> (node & 31)) & 1u) && ((onbest[next >> 5] >> (next & 31)) & 1u);
        const float val = onb ? with_elite : without;
        const uint32_t slot = node * (uint32_t)K + pdir[i];
        if (ATOMIC) atomicAdd(&tau[slot], val);
        else { rec_keys[off + i] = slot; rec_vals[off + i] = __float_as_uint(val); }
    }
}

// ------------------------------------------------------------------------------------------
// Rank-ordered deposit application.  Records [lo, hi) are sorted by slot and, inside a slot, by
// rank (stable sort of records emitted in rank order); slot s lives at buf[s - base].  The float
// additions of one slot form a dependent chain in the reference's order (tau*rho + d_1) + d_2 ...
// Short runs are summed by the thread that owns the run head.  When the colony converges every
// top-w ant deposits on the same few hundred slots (runs of ~0.2*colony records): those runs are
// handed to the whole warp, which loads 32 records per request and lets the chain run on values
// exchanged by shuffle, so the chain costs ~1 FADD per record instead of one L2 round trip.
// Must be called by all threads of the CTA (NT = threads taking part, a multiple of 32).
// ------------------------------------------------------------------------------------------
// EMIT (sharded colonies, owner-computes): every finished run also appends (slot, final value) to `fin` — the list the
// other ranks pull over NVLink instead of redoing this rank's chains (fin[0] = count, records from word 4).
// sent_val: what a slot that still holds the clean-field sentinel is worth after this iteration's evaporation (base * rho).
// lines (clean-tile field, base = 0): the line flags.  The head of the first run in each line marks it (one byte store per
// line, not per slot); the caller marks the tile.
template <bool EMIT = false>
__device__ __forceinline__ void apply_runs(float* buf, uint32_t base, const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                           uint32_t lo, uint32_t hi, uint32_t first, uint32_t stride, uint32_t* fin = nullptr, float sent_val = 0.0f,
                                           uint8_t* lines = nullptr)
{
    const int lane = threadIdx.x & 31;
    for (uint32_t r0 = lo + first; r0 < hi; r0 += stride) {   // r0 is warp-uniform: all 32 lanes run the same trips
        const uint32_t r = r0 + lane;
        bool head = r < hi;
        uint32_t key = 0;
        if (head) {
            key = keys[r];
            const uint32_t prev = r == lo ? ~0u : keys[r - 1];
            head = (r == lo) || prev != key;
            if (lines && (r == lo || prev / (uint32_t)kLineSlots != key / (uint32_t)kLineSlots)) lines[key / (uint32_t)kLineSlots] = 1;
        }
        float x = 0.0f;
        uint32_t j = r;
        bool more = false;
        if (head) {
            x = tau_or_base(buf[key - base], sent_val);
            do { x = __fadd_rn(x, __uint_as_float(vals[j])); j++; } while (j < hi && j < r + 8 && keys[j] == key);
            more = j < hi && keys[j] == key;
            if (!more) buf[key - base] = x;
        }
        if (EMIT) {   // warp-aggregated append: one atomic per warp trip
            const bool done = head && !more;
            const unsigned fm = __ballot_sync(0xffffffffu, done);
            if (fm) {
                uint32_t at = 0;
                if (lane == 0) at = atomicAdd(fin, (uint32_t)__popc(fm));
                at = __shfl_sync(0xffffffffu, at, 0);
                if (done) reinterpret_cast<uint2*>(fin + 4)[at + __popc(fm & ((1u << lane) - 1u))] = make_uint2(key, __float_as_uint(x));
            }
        }
        unsigned m = __ballot_sync(0xffffffffu, more);
        while (m) {
            const int src = __ffs(m) - 1;
            m &= m - 1;
            const uint32_t key0 = __shfl_sync(0xffffffffu, key, src);
            uint32_t j0 = __shfl_sync(0xffffffffu, j, src);
            float x0 = __shfl_sync(0xffffffffu, x, src);
            // The chain only needs the values in order; their loads do not depend on it.  A round fetches
            // kRound*32 records (kRound independent coalesced requests per array) and the next round is in
            // flight while the chain consumes the current one: one memory round trip per 256 records even
            // when the streaming part of the kernel keeps HBM saturated (loaded latency of microseconds).
            constexpr int kRound = 8;
            float v[kRound];
            unsigned ok = 0;   // bit b: this lane's record of batch b belongs to the run
#pragma unroll
            for (int q = 0; q < kRound; q++) {
                const uint32_t idx = j0 + q * 32 + lane;
                const bool valid = idx < hi && keys[idx] == key0;
                v[q] = valid ? __uint_as_float(vals[idx]) : 0.0f;
                ok |= (valid ? 1u : 0u) << q;
            }
            while (true) {
                int cnt = 0;
                bool open = true;
#pragma unroll
                for (int q = 0; q < kRound; q++) {
                    const unsigned bm = __ballot_sync(0xffffffffu, (ok >> q) & 1u);
                    const int c = bm == 0xffffffffu ? 32 : (__ffs(~bm) - 1);
                    if (open) cnt += c;
                    open = open && c == 32;
                }
                float vc[kRound];
#pragma unroll
                for (int q = 0; q < kRound; q++) vc[q] = v[q];
                if (open) {   // warp-uniform: the run continues past this round
                    j0 += kRound * 32;
                    ok = 0;
#pragma unroll
                    for (int q = 0; q < kRound; q++) {
                        const uint32_t idx = j0 + q * 32 + lane;
                        const bool valid = idx < hi && keys[idx] == key0;
                        v[q] = valid ? __uint_as_float(vals[idx]) : 0.0f;
                        ok |= (valid ? 1u : 0u) << q;
                    }
                }
#pragma unroll
                for (int q = 0; q < kRound; q++) {
                    if (q * 32 < cnt) {   // warp-uniform
#pragma unroll
                        for (int i = 0; i < 32; i++) {
                            const float t = __shfl_sync(0xffffffffu, vc[q], i);
                            if (q * 32 + i < cnt) x0 = __fadd_rn(x0, t);
                        }
                    }
                }
                if (!open) break;
            }
            if (lane == src) {
                buf[key0 - base] = x0;
                if (EMIT) reinterpret_cast<uint2*>(fin + 4)[atomicAdd(fin, 1u)] = make_uint2(key0, __float_as_uint(x0));
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// K3 split variants
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_evaporate(float4* __restrict__ tau4, size_t n4, float rho, int cs = 0)
{   // :268-272, 16 B per thread per trip, grid-stride; cs: streaming (evict-first) accesses, see stream_tile
    if (cs) {
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
            float4 v = __ldcs(tau4 + i);
            v.x = __fmul_rn(v.x, rho); v.y = __fmul_rn(v.y, rho); v.z = __fmul_rn(v.z, rho); v.w = __fmul_rn(v.w, rho);
            __stcs(tau4 + i, v);
        }
        return;
    }
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        float4 v = tau4[i];
        v.x = __fmul_rn(v.x, rho); v.y = __fmul_rn(v.y, rho); v.z = __fmul_rn(v.z, rho); v.w = __fmul_rn(v.w, rho);
        tau4[i] = v;
    }
}

// The same pass over the dirty LINES of a clean-tile field only.  One warp per 16 KB tile: each lane reads 4 of the tile's
// 128 line flags (one coalesced 128-byte load, the next tile's already in flight), the warp compacts the dirty lines into a
// shared list and streams them 16 lines per round — 8 lanes x float4 per line, 4 independent loads per lane before the first
// store.  A tile without dirty lines costs its flag load and nothing else.
constexpr int kEvapLinesPerRound = 16;
constexpr int kEvapCtasPerSm = 6;   // 40 registers; the grid is one wave of them
__global__ void __launch_bounds__(256, kEvapCtasPerSm) k_evaporate_lines(float4* __restrict__ tau4, unsigned ntiles, float rho, const uint8_t* __restrict__ lines, int cs)
{
    constexpr unsigned FULL = 0xffffffffu;
    __shared__ uint8_t s_list[8][kTileLines];
    const int lane = threadIdx.x & 31;
    uint8_t* list = s_list[threadIdx.x >> 5];
    const uint32_t* flags = reinterpret_cast<const uint32_t*>(lines) + lane;   // lines 4*lane .. 4*lane+3 of a tile
    const unsigned stride = gridDim.x * 8u;
    unsigned t = blockIdx.x * 8u + (threadIdx.x >> 5);
    uint32_t f = t < ntiles ? flags[(size_t)t * 32] : 0u;
    for (; t < ntiles; t += stride) {   // warp-uniform
        const uint32_t fn = t + stride < ntiles ? flags[(size_t)(t + stride) * 32] : 0u;
        int n = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const bool d = (f >> (8 * k)) & 0xFFu;
            const unsigned m = __ballot_sync(FULL, d);
            if (d) list[n + __popc(m & ((1u << lane) - 1u))] = (uint8_t)(4 * lane + k);
            n += __popc(m);
        }
        f = fn;
        if (n == 0) continue;
        __syncwarp();
        float4* tile = tau4 + ((size_t)t << 10) + (lane & 7);
        for (int b = 0; b < n; b += kEvapLinesPerRound) {
            float4 v[4];
            int o[4];   // float4 offset of this lane's part of line j of the round in the tile, -1: none
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int i = b + 4 * j + (lane >> 3);
                o[j] = i < n ? 8 * list[i] : -1;
                if (o[j] >= 0) v[j] = cs ? __ldcs(tile + o[j]) : tile[o[j]];
            }
#pragma unroll
            for (int j = 0; j < 4; j++) {
                if (o[j] < 0) continue;
                v[j].x = __fmul_rn(v[j].x, rho); v[j].y = __fmul_rn(v[j].y, rho); v[j].z = __fmul_rn(v[j].z, rho); v[j].w = __fmul_rn(v[j].w, rho);
                if (cs) __stcs(tile + o[j], v[j]); else tile[o[j]] = v[j];
            }
        }
        __syncwarp();   // the list is rewritten for the next tile
    }
}

__global__ void __launch_bounds__(256) k_deposit_apply(const IterState* st, const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, float* tau)
{
    const uint32_t n = (uint32_t)st->n_records;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    apply_runs(tau, 0u, keys, vals, 0u, n, warp * 32u, nwarps * 32u);
}

// ------------------------------------------------------------------------------------------
// K3 fused: evaporation + rank-ordered deposits in a single HBM pass over the pheromone field, in
// 16 KB tiles.  tile_off[t] .. tile_off[t+1] delimit tile t's (slot-sorted) records
// (k_tile_offsets, binary search).  (A variant that staged every tile through a 4-stage TMA ring in shared memory was
// measured in round 1 — 90 % of the copy bandwidth without records, 61-70 % with, it pays a load round trip per deposit
// tile — and dropped; profiles/r1*_update_fused_ncu.md keep the numbers.)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int lower_bound_key(const uint32_t* __restrict__ keys, int n, unsigned long long target)
{
    int lo = 0, hi = n;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if ((unsigned long long)keys[mid] < target) lo = mid + 1; else hi = mid;
    }
    return lo;
}
// tile_off[t] = first record of tile t (t = 0 .. ntiles); optionally the list of tiles that receive deposits
__global__ void k_tile_offsets(const int* __restrict__ d_n, const uint32_t* __restrict__ keys, uint32_t* __restrict__ tile_off, unsigned ntiles,
                               uint32_t* __restrict__ dep_list, uint32_t* dep_n)
{
    unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > ntiles) return;
    const int n = *d_n;
    const int lo = lower_bound_key(keys, n, (unsigned long long)t * kUpdTile);
    tile_off[t] = (uint32_t)lo;
    if (dep_list && t < ntiles && lo < n && (unsigned long long)keys[lo] < (unsigned long long)(t + 1) * kUpdTile) dep_list[atomicAdd(dep_n, 1u)] = t;
}

// The shipped fused update.  A CTA owns a contiguous run of 16 KB tiles.  Every tile is streamed
// register-to-register: 4 independent LDG.128 per thread, scale, STG.128 (the instruction mix that
// reaches 95 % of the copy bandwidth in k_evaporate).  If the tile receives deposits (< 5 % of the
// tiles), the CTA synchronises and applies the tile's rank-ordered deposit runs straight away with
// read-modify-writes that hit the lines it has just written (still dirty in L2), so every slot still
// costs one HBM read and one HBM write.  Tiles with deposits are processed first: their dependent
// add chains are the long pole and the plain streaming of the rest of the grid hides them.
// Measured against the all-TMA ring above in profiles/ (the ring pays a load round trip per
// deposit tile; this variant does not stage anything).
constexpr int kFusedCtasPerSm = 5;   // 48 registers per thread (the warp-cooperative chain) -> 5 x 256 threads per SM
constexpr int kFusedChunk = 8;       // plain tiles per queue grab (128 KB)

// CS: streaming (evict-first) loads and stores for tiles nobody touches again this iteration, so that the pass does not
// leave L2 full of dirty pheromone lines when the next walk starts gathering rows.
// lf: the tile's 128 line flags (shared memory); only dirty lines are moved.  nullptr: the whole tile.
template <bool CS = false>
__device__ __forceinline__ void stream_tile(float* tau, unsigned t, float rho, int tid, const uint8_t* lf = nullptr)
{
    constexpr int kVec = kUpdTile / 4 / kUpdThreads;   // float4 per thread per tile
    float4* g4 = reinterpret_cast<float4*>(tau + (size_t)t * kUpdTile);
    float4 v[kVec];
    bool on[kVec];
#pragma unroll
    for (int j = 0; j < kVec; j++) {   // float4 j * kUpdThreads + tid lies in line j * (kUpdThreads / 8) + tid / 8
        on[j] = !lf || lf[j * (kUpdThreads / 8) + (tid >> 3)];
        if (on[j]) v[j] = CS ? __ldcs(g4 + j * kUpdThreads + tid) : g4[j * kUpdThreads + tid];
    }
#pragma unroll
    for (int j = 0; j < kVec; j++) {
        if (!on[j]) continue;
        v[j].x = __fmul_rn(v[j].x, rho); v[j].y = __fmul_rn(v[j].y, rho); v[j].z = __fmul_rn(v[j].z, rho); v[j].w = __fmul_rn(v[j].w, rho);
        if (CS) __stcs(g4 + j * kUpdThreads + tid, v[j]); else g4[j * kUpdThreads + tid] = v[j];
    }
}

// q[0]: queue of deposit tiles, q[1]: queue of plain-tile chunks, q[2]: number of deposit tiles (all zeroed
// before k_tile_offsets).  Work is handed out dynamically: a CTA that sits on a long deposit chain simply
// takes fewer tiles, so the chain is hidden behind the other CTAs' streaming instead of extending the kernel.
template <bool EMIT>
__global__ void __launch_bounds__(kUpdThreads, kFusedCtasPerSm) k_update_fused(float* tau, unsigned ntiles, float rho,
                                                                                const uint32_t* __restrict__ rec_keys,
                                                                                const uint32_t* __restrict__ rec_vals,
                                                                                const uint32_t* __restrict__ tile_off,
                                                                                const uint32_t* __restrict__ dep_list, uint32_t* q, uint32_t* fin,
                                                                                int cs, const IterState* st, DirtyFlags dirty)
{   // a clean tile or line (sentinels and exact zeros only) is neither read nor written; see "Clean-tile pheromone field"
    static_assert(kFusedChunk * kTileLines == 4 * kUpdThreads, "one word of line flags per thread and chunk");
    const float base_new = __fmul_rn(st->base, rho);
    __shared__ unsigned s_next;
    __shared__ uint32_t s_off[kFusedChunk + 1];
    __shared__ uint32_t s_lines[kFusedChunk * kTileLines / 4];
    const int tid = threadIdx.x;
    const unsigned dep_n = q[2];
    if (EMIT && blockIdx.x == 0 && tid == 0) fin[1] = dep_n;   // sharded: this rank's share of the "tiles that received deposits" statistic
    while (true) {   // ---- tiles that receive deposits, first ----
        if (tid == 0) s_next = atomicAdd(&q[0], 1u);
        __syncthreads();
        const unsigned i = s_next;
        __syncthreads();
        if (i >= dep_n) break;
        const unsigned t = dep_list[i];
        const uint32_t lo = tile_off[t], hi = tile_off[t + 1];
        if (dirty.tile[t]) stream_tile(tau, t, rho, tid);   // CTA-uniform; the clean lines of the tile are streamed too (harmless: rho keeps them)
        __syncthreads();   // the scaled tile is visible to the whole CTA
        apply_runs<EMIT>(tau, 0u, rec_keys, rec_vals, lo, hi, (uint32_t)(tid & ~31), (uint32_t)kUpdThreads, fin, base_new, dirty.line);
        if (tid == 0) dirty.tile[t] = 1;
    }
    while (true) {   // ---- everything else: pure streaming ----
        if (tid == 0) s_next = atomicAdd(&q[1], (unsigned)kFusedChunk);
        __syncthreads();
        const unsigned c0 = s_next;
        if (c0 < ntiles && tid <= kFusedChunk) s_off[tid] = tile_off[min(c0 + tid, ntiles)];
        if (c0 < ntiles) s_lines[tid] = c0 + tid / 32u < ntiles ? reinterpret_cast<const uint32_t*>(dirty.line)[(size_t)c0 * 32 + tid] : 0u;
        __syncthreads();
        if (c0 >= ntiles) break;
        const unsigned c1 = min(c0 + kFusedChunk, ntiles);
        const uint8_t* lf = reinterpret_cast<const uint8_t*>(s_lines);
        for (unsigned t = c0; t < c1; t++)
            if (s_off[t - c0] == s_off[t - c0 + 1] && dirty.tile[t]) {
                if (cs) stream_tile<true>(tau, t, rho, tid, lf + (t - c0) * kTileLines); else stream_tile<false>(tau, t, rho, tid, lf + (t - c0) * kTileLines);
            }
        __syncthreads();   // s_off / s_next are reused by the next grab
    }
}

// ------------------------------------------------------------------------------------------
// setPoints (:537-565) on the device.  The reference scans every node and keeps the LAST one (z,y,x
// order = largest id) that is free and within 1.2*precision of the point on every axis.  The per-axis
// test is separable, so the match set is a product of three tiny index lists; one CTA per point
// collects them and takes the largest free id.  ids[p] = -1 when nothing matches.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_snap_points(const float* __restrict__ pts, int npts, const float* __restrict__ coords, int rx, int ry, int rz,
                                                      float t, const uint32_t* __restrict__ occ_bits, long long* __restrict__ ids)
{
    constexpr int kMax = 16;   // matches per axis: spacing = precision, window 2.4*precision -> 2-3 (a few more on duplicate planes)
    __shared__ int list[3][kMax];
    __shared__ int cnt[3];
    __shared__ long long best;
    const int p = blockIdx.x;
    if (p >= npts) return;
    if (threadIdx.x < 3) cnt[threadIdx.x] = 0;
    if (threadIdx.x == 0) best = -1;
    __syncthreads();
    const int n[3] = {rx, ry, rz};
    const float* axis[3] = {coords, coords + rx, coords + rx + ry};
    for (int a = 0; a < 3; a++) {
        const float q = pts[3 * p + a];
        for (int i = threadIdx.x; i < n[a]; i += blockDim.x) {
            const float d = __fsub_rn(q, axis[a][i]);
            const float ad = d > 0.0f ? d : -d;   // my_abs
            if (ad < t) { const int k = atomicAdd(&cnt[a], 1); if (k < kMax) list[a][k] = i; }
        }
    }
    __syncthreads();
    const int cx = min(cnt[0], kMax), cy = min(cnt[1], kMax), cz = min(cnt[2], kMax);
    const int total = cx * cy * cz;
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        const int x = list[0][i % cx], y = list[1][(i / cx) % cy], z = list[2][i / (cx * cy)];
        const long long id = ((long long)z * ry + y) * rx + x;
        if (!((occ_bits[id >> 5] >> (id & 31)) & 1u)) atomicMax(&best, id);
    }
    __syncthreads();
    if (threadIdx.x == 0) ids[p] = best;
}

// all-pairs driver: keep the finished search's best (getSolution :506-509) in slot `pair` of the result arrays
__global__ void k_save_result(const IterState* st, const int* __restrict__ best_n, const uint32_t* __restrict__ best_ids,
                              const uint8_t* __restrict__ best_dirs, int pair, int path_cap, float* __restrict__ res_L, int* __restrict__ res_n,
                              uint32_t* __restrict__ res_ids, uint8_t* __restrict__ res_dirs)
{
    const bool found = st->best_steps != INT_MAX;
    const int n = found ? *best_n : 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) { res_L[pair] = st->best_L; res_n[pair] = n; }
    uint32_t* oi = res_ids + (size_t)pair * path_cap;
    uint8_t* od = res_dirs + (size_t)pair * path_cap;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n && i < path_cap; i += gridDim.x * blockDim.x) {
        oi[i] = best_ids[i];
        if (i + 1 < n) od[i] = best_dirs[i];
    }
}

// Sharded colonies, owner-computes: rank r applied the deposits of its slot slice and listed the final values
// (k_update_fused<true>); every other rank pulls that list straight out of r's HBM over NVLink (peer pointers) and
// overwrites its own, so far only evaporated, copy.  bufs[p]: word 0 = count, records (slot, value bits) from word 4.
// The same pass is the next walk's L2 warm-up: the slots that just received deposits are where the colony walks next, so
// the tau lines are left in L2 — the other ranks' by the writes, this rank's own slice by a touch.
__global__ void __launch_bounds__(256) k_pull_finals(PeerBarrier pb, const IterState* st, float* tau, const uint32_t* const* __restrict__ bufs, int npeers,
                                                      int me, DirtyFlags dirty, uint32_t* upd_q)
{
    peer_barrier(pb, st, 2u);   // every rank's list of final values is complete
    uint32_t acc = 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) {   // tiles that received deposits on ANY rank (the slices are disjoint): the statistic k_iter_begin publishes
        uint32_t tiles = 0;
        for (int p = 0; p < npeers; p++) tiles += __ldcg(bufs[p] + 1);
        upd_q[2] = tiles;
    }
    for (int p = 0; p < npeers; p++) {
        const uint32_t* buf = bufs[p];
        const uint32_t cnt = __ldcg(buf);
        const uint2* rec = reinterpret_cast<const uint2*>(buf + 4);
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += gridDim.x * blockDim.x) {
            const uint2 r = __ldcg(rec + i);
            if (p != me) { tau[r.x] = __uint_as_float(r.y); dirty.mark(r.x); }
            else acc ^= __ldcg(reinterpret_cast<const uint32_t*>(tau) + r.x);
        }
    }
    if (acc == 0x9E3779B9u && npeers < 0) tau[0] = 0.0f;   // keeps the warm-up loads alive; never true
}

// barrier 1 (every rank's walk is complete), then every rank's step counts -> the global colony array the ranking reads
__global__ void __launch_bounds__(256) k_gather_steps(PeerBarrier pb, const IterState* st, const int* const* __restrict__ steps_tab, int nranks, int chunk,
                                                      int* __restrict__ all_steps)
{
    peer_barrier(pb, st, 1u);
    const int total = nranks * chunk;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int r = i / chunk;
        all_steps[i] = __ldcg(steps_tab[r] + (i - r * chunk));
    }
}

// reset() :307-315 and the initial field of initFromGridMap :391-401
__global__ void k_tau_fill(float* tau, size_t n, float v)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) tau[i] = v;
}
// reset() on a clean-tile field: every slot back to "tau0" = the sentinel with base = tau0, every flag back to 0.  all = 0:
// only the dirty lines of the dirty tiles need rewriting (after the first reset() the out-of-bounds slots hold the sentinel
// too, like the reference's, :307-315); all = 1: every line.
__global__ void __launch_bounds__(256) k_tau_reset_lines(float4* __restrict__ tau4, unsigned ntiles, DirtyFlags dirty, int all)
{
    const float s = __uint_as_float(kSentinelBits);
    const float4 v = make_float4(s, s, s, s);
    for (unsigned t = blockIdx.x; t < ntiles; t += gridDim.x) {
        if (!all && !dirty.tile[t]) continue;
        float4* p = tau4 + ((size_t)t << 10) + threadIdx.x;
        const uint8_t* lf = dirty.line + (size_t)t * kTileLines + threadIdx.x / 8;
#pragma unroll
        for (int j = 0; j < 4; j++) if (all || lf[32 * j]) p[256 * j] = v;
        __syncthreads();   // every flag of the tile has been read
        if (threadIdx.x < kTileLines / 4) reinterpret_cast<uint32_t*>(dirty.line)[(size_t)t * (kTileLines / 4) + threadIdx.x] = 0u;
        if (threadIdx.x == 0) dirty.tile[t] = 0;
    }
}
// clean-tile form: the host passes the sentinel as tau0 (the in-bounds slots' value is then IterState::base)
__global__ void k_tau_init(float* tau, int rx, int ry, int rz, unsigned long long N, float tau0)
{   // out-of-bounds slots start at 0 (:396), in-bounds at tau0 (:401)
    unsigned long long id = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= N) return;
    const unsigned long long rxy = (unsigned long long)rx * ry;
    int z = (int)(id / rxy);
    unsigned r = (unsigned)(id % rxy);
    int y = r / rx, x = r % rx;
    float* t = tau + id * 6;
    t[0] = z > 0 ? tau0 : 0.f; t[1] = y > 0 ? tau0 : 0.f; t[2] = x > 0 ? tau0 : 0.f;
    t[3] = x + 1 < rx ? tau0 : 0.f; t[4] = y + 1 < ry ? tau0 : 0.f; t[5] = z + 1 < rz ? tau0 : 0.f;
}

}  // namespace wr
