// K2, pass 2 — and the pieces every walk kernel shares (selectNext ACSRank_3D.hpp:134-193 + the ant loop :252-265).
//
// The ant-construction step as every K = 6 kernel runs it: one ant per 8-lane group (6 neighbour lanes + 2 idle), 4 ants per
// warp stepping in LOCKSTEP so that every warp collective runs with the full mask.  Lane k < 6 owns neighbour slot k: it loads
// tau[cur][k] and the tabulated geometric factor heur[cur][k] (the six lanes of a group read 24 contiguous bytes per array),
// probes the visited set for its neighbour and evaluates tau^alpha * (1 + beta*cos).  The roulette needs the reference's exact
// summation order (ascending for `total`, descending for `prob_sum`), so the six scores are exchanged with width-8 shuffles and
// every lane re-adds them sequentially — two chains of 6 dependent FADDs.  Non-candidates carry info = +0, the identity.
//   * node coordinates live in ONE packed register  P = z<<20 | y<<10 | x  (a move is one add; needs dims <= 1024,
//     wr_acs_create rejects larger grids);
//   * the visited set ("tabu", std::set at :70) is an open-addressed table of 64-bit entries
//     (1<<31 | tile key) << 32 | 32-bit mask  over 4x4x2-node tiles: one 64-bit load per probe, one store per insert;
//   * the move comes from a 64-entry table indexed by the pick ballot.
// Pass 1 of every iteration is k_walk3 (walk3.cuh; k_walk_batch3 for concurrent searches) with the tables in shared memory.  An
// ant whose shared-memory table reaches 3/4 moves its visited set to a table in HBM sized for the step cap, parks {node, steps}
// and is RESUMED by the kernel below, k_walk2, from the very step it stopped at — exact, because its draws are a pure function
// of (search, iteration, ant, step).  Two launches keep shared-memory addressing on the common path (a run-time switch cost
// 8-13 % per step); pass 2 usually finds nothing to do and exits at once.  One k_walk2 serves both: its input type says where
// tau, the factor, the open mask and the ant's identity come from — Dense6 (below) for one search, Batch6 (batch.cuh) for
// concurrent searches.
// (Round 1-2 history: k_walk2 also was pass 1 until k_walk3 replaced it — 164 -> 127 instructions per warp-step, see
// profiles/r2_walk3_*; that generic form, its L1/L2 prefetch modes and the register look-ahead experiment are gone.)
#pragma once
#include "acs_kernels.cuh"

namespace wr {

constexpr uint32_t kPackLow = 0x00100C03u;                    // x bits 0-1, y bits 10-11, z bit 20: position inside a 4x4x2 tile
constexpr uint32_t kPackKey = 0x3FFFFFFFu & ~kPackLow;        // the tile
constexpr uint32_t kPackMul = 0x00101010u;                    // gathers the five position bits at 20..24 (no carries: partial products are disjoint)
constexpr int kWalk2Lut = 1024;                                // bytes of the move table at the start of k_walk2's shared memory
constexpr uint32_t kKeyTag = 0x80000000u;                     // a stored key is never 0 (0 = empty entry)

__device__ __forceinline__ uint32_t pack_xyz(int x, int y, int z) { return (uint32_t)x | ((uint32_t)y << 10) | ((uint32_t)z << 20); }
// table sizes need not be powers of two (768 entries per ant = two CTAs per SM): Fibonacci hash, then multiply-high range reduction
__device__ __forceinline__ uint32_t tile_hash(uint32_t key, uint32_t entries) { return __umulhi(key * 2654435761u, entries); }

// visited-table access: 32-bit shared-window addresses for the on-chip tables (a generic pointer makes the compiler
// re-derive the shared window base inside the step loop), plain global pointers for the HBM tables of pass 2
template <bool GLOBAL> struct TabRef {
    unsigned long long* gp;
    uint32_t sa;
    __device__ __forceinline__ unsigned long long load(unsigned slot) const
    {
        if (GLOBAL) return gp[slot];
        unsigned long long v;
        asm volatile("ld.shared.b64 %0, [%1];" : "=l"(v) : "r"(sa + slot * 8u) : "memory");
        return v;
    }
    __device__ __forceinline__ void store(unsigned slot, unsigned long long v) const
    {
        if (GLOBAL) { gp[slot] = v; return; }
        asm volatile("st.shared.b64 [%0], %1;" ::"r"(sa + slot * 8u), "l"(v) : "memory");
    }
};

// What a lane of the resume pass needs about its neighbour slot at the current node
struct Slot6 {
    float tau;    // as stored: the sentinel stands for the clean-field scalar
    float heur;   // 1 + beta*cos
    bool open;    // in bounds, free, and one of the six neighbour lanes
};

// Inputs of k_walk2 for one search (WalkArgs): tau and the tabulated factor from the dense [N][6] rows
struct Dense6 {
    using Args = WalkArgs;
    const float* tau_k;    // this lane's column of the tau rows; idle lanes (k = 6, 7) re-read slot 5 (same sector)
    const float* heur_k;   // ... of the factor rows; idle lanes read a constant "closed" marker with a zero row stride, so
    int heur_row;          //     `open` is one compare for every lane
    int start, goal;
    uint32_t ant, stream_word, block_hi;   // Philox counter words of the bound ant
    size_t row;            // its row of path_ids / path_dirs / ant_steps
    float tau_v, heur_v;   // this lane's slot of the current row

    __device__ __forceinline__ Dense6(const WalkArgs& a, int k)
        : tau_k(a.tau + (k < 6 ? k : 5)), heur_k(k < 6 ? a.heur + k : a.closed_marker), heur_row(k < 6 ? 6 : 0), start(a.start), goal(a.goal),
          stream_word(a.stream_word), block_hi(a.block_hi)
    {
    }
    // parked ants to resume: the search has an HBM table for every ant of its colony
    __device__ __forceinline__ unsigned items(const WalkArgs&, const IterState* st) const { return st->overflow_n; }
    // entry q of the parked-ant list (has = false: no ant, the group idles)
    __device__ __forceinline__ void bind(const WalkArgs& a, unsigned q, bool has)
    {
        const int ant_local = has ? (int)a.overflow_list[q] : 0;
        ant = (uint32_t)(a.shard_first + ant_local);
        row = (size_t)ant_local;
    }
    // reloaded as soon as the next node is known, ahead of the move's side effects
    __device__ __forceinline__ void issue(int cur, uint32_t)
    {
        tau_v = __ldg(tau_k + (size_t)cur * 6);
        heur_v = __ldg(heur_k + (size_t)cur * heur_row);
    }
    // NaN (duplicate plane) stays open, as in the reference
    __device__ __forceinline__ Slot6 resolve() const { return {tau_v, heur_v, heur_v != kClosedSlot}; }
};

// Pass 2: resume the ants pass 1 parked, with their visited sets in HBM tables.  In = Dense6 (one search) or Batch6
// (concurrent searches, batch.cuh) says where tau, the factor, the open mask and the ant's identity come from.
template <class In, bool ALPHA1>
__global__ void __launch_bounds__(kWalkThreads) k_walk2(typename In::Args a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // [0, 1024): move table indexed by the 6-bit pick ballot: the winner is its highest set bit c (the roulette scans
    //            5 -> 0) -> {node-id stride, packed-coordinate delta, c, -}; one LDS.128 replaces find-leading-one + index math
    int4* move_lut = reinterpret_cast<int4*>(smem_raw);
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
    const int E = 1 << a.gtable_log2;   // entries of an HBM table
    uint32_t lut_sa = (uint32_t)__cvta_generic_to_shared(move_lut);
    TabRef<true> tab;
    tab.gp = a.gtab;
    tab.sa = 0;
    // opaque to the optimiser: otherwise it re-derives the shared-window base (S2UR + ULEA) inside the step loop
    asm volatile("" : "+r"(lut_sa));

    const int rx = a.rx, rxy = a.rx * a.ry;
    const int dxk = (k == 3) - (k == 2), dyk = (k == 4) - (k == 1), dzk = (k == 5) - (k == 0);
    const uint32_t dPk = (uint32_t)(dxk + dyk * 1024 + dzk * 1048576);
    In in(a, k);
    // lane masks of the descending prefix chain: lane k adds v_j only for j >= k
    uint32_t m4 = k <= 4 ? ~0u : 0u, m3 = k <= 3 ? ~0u : 0u, m2 = k <= 2 ? ~0u : 0u, m1 = k <= 1 ? ~0u : 0u, m0 = k <= 0 ? ~0u : 0u;
    asm volatile("" : "+r"(m4), "+r"(m3), "+r"(m2), "+r"(m1), "+r"(m0));   // keep them as register masks (one LOP3 each) instead of re-derived predicates

    IterState* st = a.st;
    const uint32_t iter = (uint32_t)st->iter;
    const float base_now = st->base;   // clean-tile field: what a slot that never received a deposit is worth this iteration
    const unsigned n_items = in.items(a, st);   // the ants pass 1 parked (and found a table for)
    const int cap = a.cap;

    unsigned long long c_steps = 0, c_ants = 0, c_arrived = 0, c_nocand = 0, c_fall = 0, c_cap = 0;

    while (true) {
        unsigned q0 = 0;
        if (lane == 0) q0 = atomicAdd(&st->queue2, 4u);
        q0 = __shfl_sync(FULL, q0, 0);
        if (q0 >= n_items) break;                                              // warp-uniform
        const unsigned q = q0 + (unsigned)(lane >> 3);
        const bool has = q < n_items;
        in.bind(a, q, has);

        int cur = in.start, steps = 0;
        uint32_t P = pack_xyz(cur % rx, (cur % rxy) / rx, cur / rxy);
        float u0 = 0.f, u1 = 0.f, u2 = 0.f, u3 = 0.f;
        auto draw4 = [&](uint32_t block) {
            uint32_t w0, w1, w2, w3;
            philox4(iter, in.ant, block | in.block_hi, in.stream_word, a.seed_lo, a.seed_hi, w0, w1, w2, w3);
            // (float)rand()/(float)RAND_MAX (:169): (float)RAND_MAX is 2^31, so the division is an exact scaling
            u0 = __fmul_rn(__int2float_rn((int)(w0 >> 1)), 4.656612873077392578125e-10f);
            u1 = __fmul_rn(__int2float_rn((int)(w1 >> 1)), 4.656612873077392578125e-10f);
            u2 = __fmul_rn(__int2float_rn((int)(w2 >> 1)), 4.656612873077392578125e-10f);
            u3 = __fmul_rn(__int2float_rn((int)(w3 >> 1)), 4.656612873077392578125e-10f);
        };
        // resume a parked ant: its visited set already lives in HBM table q
        tab.gp = a.gtab + (size_t)(has ? q : 0) * E;
        if (has) {
            const int4 r = a.resume[q];
            cur = r.x; steps = r.y;
            P = pack_xyz(cur % rx, (cur % rxy) / rx, cur / rxy);
            draw4((uint32_t)steps >> 2);
        }
        __syncwarp();

        bool live = has;
        int result = -1;   // >= 0: steps of an ant that arrived, -1: dead, -2: parked (table 3/4 full -> pass 2)
        int reason = 0;    // why a dead ant died: 1 no candidate, 2 roulette fall-through, 3 step cap
        if (live && steps >= cap) { live = false; reason = 3; }
        uint32_t* pid = a.path_ids + in.row * cap;
        uint8_t* pdir = a.path_dirs + in.row * cap;
        in.issue(cur, P);

        auto step = [&]() {
            // ---- Philox: one call yields the draws of 4 consecutive steps (live ants of a warp are in lockstep) ----
            if (live && (steps & 3) == 0) draw4((uint32_t)steps >> 2);
            const float u = (steps & 2) ? ((steps & 1) ? u3 : u2) : ((steps & 1) ? u1 : u0);
            // ---- neighbour k: open, tau, factor, tabu probe -----------------------------------------------------------
            const Slot6 sl = in.resolve();
            const bool open_k = sl.open;
            const uint32_t Pk = P + dPk;
            const uint32_t key = (Pk & kPackKey) | kKeyTag;
            const uint32_t bitm = 1u << ((((Pk & kPackLow) * kPackMul) >> 20) & 31u);
            unsigned slot = tile_hash(key, (uint32_t)E);
            unsigned long long e = tab.load(slot);
            while (open_k && (uint32_t)(e >> 32) != key && (uint32_t)(e >> 32) != 0u) {   // collisions are rare at load <= 3/4
                slot = slot + 1 < (unsigned)E ? slot + 1 : 0u;
                e = tab.load(slot);
            }
            const bool found = (uint32_t)(e >> 32) == key;
            const uint32_t emask = found ? (uint32_t)e : 0u;
            const bool cand = live && open_k && !(emask & bitm);
            // ---- info = tau^alpha * (1 + beta*cos)  (:151-154) -------------------------------------------------------
            const float tau_now = tau_or_base(sl.tau, base_now);
            const float tpow = ALPHA1 ? tau_now : pow_int(tau_now, a.alpha);
            const float info = cand ? __fmul_rn(tpow, sl.heur) : 0.0f;
            // ---- roulette in the reference's order (:155, :172-181) ------------------------------
            const unsigned cb = (__ballot_sync(FULL, cand) >> gbase) & 0x3Fu;
            const float v0 = __shfl_sync(FULL, info, 0, 8), v1 = __shfl_sync(FULL, info, 1, 8), v2 = __shfl_sync(FULL, info, 2, 8);
            const float v3 = __shfl_sync(FULL, info, 3, 8), v4 = __shfl_sync(FULL, info, 4, 8), v5 = __shfl_sync(FULL, info, 5, 8);
            const float total = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(0.0f, v0), v1), v2), v3), v4), v5);
            const float rnd = __fmul_rn(u, total);
            // this lane's prob_sum: v5 + v4 + ... + v_k, then +0 (the identity of the chain), so one chain serves all lanes
            float mine = __fadd_rn(0.0f, v5);
            mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v4) & m4));
            mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v3) & m3));
            mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v2) & m2));
            mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v1) & m1));
            mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v0) & m0));
            const bool pick = cand && (mine >= rnd);
            const unsigned pb = (__ballot_sync(FULL, pick) >> gbase) & 0x3Fu;   // the first hit scanning 5 -> 0 is its highest set bit
            // ---- the move: one table look-up on the ballot, then the next row's loads go out at once ---------------
            int4 mv;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(mv.x), "=r"(mv.y), "=r"(mv.z), "=r"(mv.w) : "r"(lut_sa + pb * 16u) : "memory");
            const int c = mv.z;
            const bool stepok = live && pb != 0;
            const int prev = cur, at = steps;
            if (stepok) { cur += mv.x; P += (uint32_t)mv.y; steps++; }
            in.issue(cur, P);
            // ---- outcome -------------------------------------------------------------------------
            if (live && !stepok) reason = cb == 0 ? 1 : 2;              // :162-166 / fall-through :191-192
            if (stepok && k == c) {   // the winning lane performs the move's side effects: tabu insert + addNextNode (:73-79)
                tab.store(slot, ((unsigned long long)key << 32) | (unsigned long long)(emask | bitm));
                pid[at] = (uint32_t)prev;
                pdir[at] = (uint8_t)c;
            }
            const bool arrived = stepok && cur == in.goal;           // :182-186
            const bool capped = stepok && !arrived && steps >= cap;   // a deviation the oracle mirrors; the reference is unbounded
            result = arrived ? steps : result;
            reason = capped ? 3 : reason;
            live = stepok && !arrived && !capped;
            __syncwarp();
        };
        while (__any_sync(FULL, live)) {   // two steps per trip: halves the cost of the loop's vote + branch; a finished ant just idles
            step();
            step();
        }
        if (has) {
            c_arrived += result >= 0 ? 1 : 0;
            c_nocand += (result < 0 && reason == 1) ? 1 : 0;
            c_fall += (result < 0 && reason == 2) ? 1 : 0;
            c_cap += (result < 0 && reason == 3) ? 1 : 0;
            c_steps += (unsigned long long)steps; c_ants++;
            if (k == 0) a.ant_steps[in.row] = result;
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
    }
}

}  // namespace wr
