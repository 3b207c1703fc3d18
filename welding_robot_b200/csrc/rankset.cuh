// Rank-set deposits (WR_UPDATE_RANKSET): update_pheromone (core/ACSRank_3D.hpp:198-215) without sorting records.
//
// The reference adds, per directed slot, the deposits of the ants that crossed it in RANK order (the sorted colony is
// walked front to back, :275-280, and a self-avoiding ant crosses a slot at most once):
//     tau[s] = ((tau[s]*rho + d(r1, s)) + d(r2, s)) + ...      r1 < r2 < ... the ranks of the ants that crossed s
//     d(r, s) = (lambda - order_r)*Q/L_r + float(s's edge lies on the best path)*lambda*Q/L_best            (:209-211)
// so the value depends on the rank and on ONE bit of the slot.  What has to be known per slot is therefore the SET of
// ranks that crossed it — a bitmask over the <= 0.2*colony eligible ranks — and a set is built with atomicOr in any
// order: no (slot, rank) sort, no record list.  OR is also what makes the set shardable: every rank of a multi-GPU
// colony builds the sets of ITS ants (bits = global ranks) and the partial sets are OR-merged (k_rankset_merge).
//
// Table: open-addressed, keyed by (slot, group) where group = rank >> 10; an entry owns one ROW BLOCK of 32 words =
// 1024 rank bits (128 B, one cache line).  Key (64 bit, claimed by atomicCAS): slot+1 | group << 32 | on-best << 63 —
// every ant that crosses a slot computes the same on-best bit, so the bit is part of the key.  Colonies of any size
// use the same code: 4096 ants -> 820 eligible ranks -> one group; 65 536 ants -> 13 groups.  The table has a FIXED
// capacity (the path is only chosen while the colony's deposits are concentrated; acs.cu): a build that would exceed
// half of it raises the overflow flag, the blocks claimed so far are wiped and the iteration's deposits are applied by
// k_deposit_serial — the reference's own loop order, exact for any input, slow, and in practice never taken.
//
//   k_rankset_gen     one CTA per eligible rank: value pair of the rank -> vtab; every step of its (local) trail:
//                     find or claim the block of (slot, rank >> 10), set bit (rank & 1023); claimed blocks -> `list`.
//                     Group deposits (converged iterations): the ranks whose local ant k_path_verify saw follow the whole
//                     best path cross the same slots with the same on-best bits, so k_rank_small lists them in one mask per
//                     rank group and kRsGroupCtas CTAs of the same launch walk ONE such trail, OR-ing the masks into each
//                     step's blocks; their own CTAs only write the vtab pair.  Same (key, bits) in the table, same field.
//   k_rankset_publish / k_rankset_merge   sharded colonies: the claimed blocks (key + 32 words) are copied to the peer
//                     slab, and every rank ORs every peer's blocks into its own table
//   k_evaporate_lines (acs_kernels.cuh) tau *= rho over the dirty lines, :268-272 — the one HBM stream of the update
//   k_rankset_apply   per slot, the block of its lowest group leads: it adds the ranks' values of group 0, 1, 2 ... to
//                     tau[slot] in ascending rank order (the higher groups' blocks are looked up) = the reference's
//                     additions in the reference's order; then the blocks and keys are wiped for the next iteration
//                     (in the same kernel for one group, by k_rankset_clear otherwise)
#pragma once
#include "acs_kernels.cuh"

namespace wr {

constexpr int kRsRowWords = 32;                       // words per row block
constexpr int kRsGroupRanks = kRsRowWords * 32;       // 1024 ranks per group
constexpr int kRsPubWords = 2 + kRsRowWords;          // a published block: key (2 words) + row

struct RankSet {
    unsigned long long* key;   // [R]  slot+1 | group << 32 | onbest << 63; 0 = free
    uint32_t* rows;            // [R][32]
    uint32_t* list;            // [limit+1] blocks claimed (or merged in) this iteration
    uint32_t* count;           // [0] blocks in `list` [1] blocks of the previous rank-set iteration (0xFFFFFFFF: it overflowed) [2] always 0
                               // [3] overflow flag
    float* vtab;               // [w_max][2]  d(r, s) without / with the elitist term
    uint32_t rmask;            // R - 1
    int shift;                 // 32 - log2(R)
    uint32_t limit;            // claims allowed per iteration (<= R/2; sharded: also the capacity of the publish area)
};

__device__ __forceinline__ uint32_t rankset_hash(uint32_t slot, uint32_t group) { return (slot * 2654435761u) ^ (group * 0x9E3779B1u + (group << 15)); }

// find or claim the block of `want`; returns its index, sets `claimed`.  Returns 0xFFFFFFFF once the table has overflowed.
__device__ __forceinline__ uint32_t rankset_find_or_claim(const RankSet& rs, unsigned long long want, uint32_t h, bool& claimed)
{
    claimed = false;
    for (uint32_t probes = 0; probes <= rs.rmask; probes++) {
        unsigned long long k = __ldcg(rs.key + h);
        if (k == 0ull) {
            k = atomicCAS(rs.key + h, 0ull, want);
            if (k == 0ull) { claimed = true; return h; }
        }
        if (k == want) return h;
        h = (h + 1) & rs.rmask;
    }
    return 0xFFFFFFFFu;   // table completely full: cannot happen below the claim limit
}

constexpr int kRsGenThreads = 256;                 // k_rankset_gen: threads per CTA = steps per trip of one rank's trail
constexpr int kRsGroupCtas = 1024 / kRsGenThreads;  // CTAs behind the per-rank ones that set the group's bits (1024 steps per trip)

// The group's bits (k_rank_small: the eligible ranks whose local ant followed the whole best path): every such ant crossed the
// same slots with the same on-best bits, so the representative's trail is walked ONCE and each group's 32 mask words are
// OR-ed into the block of every step, one lane per word — instead of one find-or-claim + atomicOr per step and rank.  The
// trail rows are the representative's own: k_best_copy may already have replaced the best path of this iteration.
__device__ __forceinline__ void rankset_gen_group(const IterState* st, const uint32_t* __restrict__ path_ids, const uint8_t* __restrict__ path_dirs, int cap,
                                                  int goal, const uint32_t* __restrict__ onbest, const RankSet& rs, int K, const uint32_t* __restrict__ gmask, int gc)
{
    constexpr unsigned FULL = 0xffffffffu;
    const int steps = st->grp_steps;
    const size_t ant = (size_t)st->grp_rep;
    const uint32_t* pid = path_ids + ant * cap;
    const uint8_t* pdir = path_dirs + ant * cap;
    const uint32_t groups = ((uint32_t)st->n_eligible + kRsGroupRanks - 1) / kRsGroupRanks;
    const int lane = threadIdx.x & 31;
    volatile uint32_t* over = rs.count + 3;
    for (int i0 = gc * blockDim.x; i0 < steps; i0 += kRsGroupCtas * blockDim.x) {   // CTA-uniform trips
        const int i = i0 + threadIdx.x;
        uint32_t slot = 0;
        bool onb = false;
        if (i < steps) {   // the same expressions as the per-rank loop below
            const uint32_t node = pid[i];
            slot = node * (uint32_t)K + pdir[i];
            const uint32_t next = (i + 1 < steps) ? pid[i + 1] : (uint32_t)goal;
            onb = ((onbest[node >> 5] >> (node & 31)) & 1u) && ((onbest[next >> 5] >> (next & 31)) & 1u);
        }
        for (uint32_t g = 0; g < groups; g++) {
            const uint32_t mw = gmask[g * kRsRowWords + lane];   // lane j holds word j of the group's mask
            if (!__any_sync(FULL, mw != 0u)) continue;         // warp-uniform: no rank of this group is in the group path
            const bool valid = i < steps && *over == 0u;
            uint32_t h = 0xFFFFFFFFu;
            bool claimed = false;
            if (valid) {
                const unsigned long long want = (unsigned long long)(slot + 1u) | ((unsigned long long)g << 32) | (onb ? (1ull << 63) : 0ull);
                h = rankset_find_or_claim(rs, want, rankset_hash(slot, g) >> rs.shift, claimed);
            }
            const unsigned cm = __ballot_sync(FULL, claimed);
            if (cm) {   // one counter update per warp, as in the per-rank loop
                uint32_t at = 0;
                if (lane == __ffs(cm) - 1) at = atomicAdd(rs.count, (uint32_t)__popc(cm));
                at = __shfl_sync(FULL, at, __ffs(cm) - 1);
                const uint32_t mine = at + __popc(cm & ((1u << lane) - 1u));
                if (claimed) {
                    if (mine < rs.limit) rs.list[mine] = h;
                    else *over = 1u;
                }
            }
            unsigned hm = __ballot_sync(FULL, h != 0xFFFFFFFFu);
            while (hm) {   // the warp's steps one after the other, the 32 words of each block at once
                const int src = __ffs(hm) - 1;
                hm &= hm - 1;
                const uint32_t hs = __shfl_sync(FULL, h, src);
                if (mw) atomicOr(rs.rows + (size_t)hs * kRsRowWords + lane, mw);
            }
        }
    }
}

// path_ids/path_dirs: THIS rank's trails (local ant index = global - shard_first); eligible ranks whose ant lives on
// another rank only contribute their vtab pair here (their owner sets their bits and the merge brings them over).
// Grid: w_max CTAs, one per rank, then kRsGroupCtas for the group (gmask, st->grp_rep).  A rank in the group only writes its
// vtab pair: the group CTAs set its bits.
__global__ void __launch_bounds__(kRsGenThreads) k_rankset_gen(const IterState* st, const uint32_t* __restrict__ rank_keys, const uint32_t* __restrict__ rank_vals,
                                                      const uint32_t* __restrict__ path_ids, const uint8_t* __restrict__ path_dirs, int cap, int goal,
                                                      const float* __restrict__ Ltab, const uint32_t* __restrict__ onbest, RankSet rs, int K,
                                                      const int* __restrict__ steps26, int shard_first, int shard_chunk, const uint32_t* __restrict__ gmask)
{
    constexpr unsigned FULL = 0xffffffffu;
    const int gc = (int)blockIdx.x - (int)(gridDim.x - kRsGroupCtas);
    if (gc >= 0) {
        if (st->use_rankset && st->grp_rep >= 0) rankset_gen_group(st, path_ids, path_dirs, cap, goal, onbest, rs, K, gmask, gc);
        return;
    }
    const int r = blockIdx.x;
    if (r >= st->n_eligible || !st->use_rankset) return;
    const int ant_global = (int)rank_vals[r];
    const int steps = steps26 ? steps26[ant_global] : (int)rank_keys[r];
    if (threadIdx.x == 0) {   // the same expressions, in the same order, as k_deposit_gen
        const float L_ant = steps26 ? __uint_as_float(rank_keys[r]) : Ltab[steps];
        const float lambda = st->lambda, Q = st->Q;
        const float base = __fdiv_rn(__fmul_rn(__fsub_rn(lambda, (float)(r + 1)), Q), L_ant);
        const float elite = __fdiv_rn(__fmul_rn(__fmul_rn(1.0f, lambda), Q), st->best_L);
        rs.vtab[2 * r] = __fadd_rn(base, 0.0f);
        rs.vtab[2 * r + 1] = __fadd_rn(base, elite);
    }
    if (ant_global < shard_first || ant_global >= shard_first + shard_chunk) return;   // another rank holds this trail
    if (st->grp_rep >= 0 && ((gmask[r >> 5] >> (r & 31)) & 1u)) return;               // set by the group CTAs
    const size_t ant = (size_t)(ant_global - shard_first);
    const uint32_t* pid = path_ids + ant * cap;
    const uint8_t* pdir = path_dirs + ant * cap;
    const uint32_t group = (uint32_t)r >> 10;
    const uint32_t word = ((uint32_t)r >> 5) & 31u, bit = 1u << (r & 31);
    const int lane = threadIdx.x & 31;
    volatile uint32_t* over = rs.count + 3;
    for (int i0 = 0; i0 < steps; i0 += blockDim.x) {         // CTA-uniform trips: the list append below is warp-aggregated
        const int i = i0 + threadIdx.x;
        const bool valid = i < steps && *over == 0u;
        uint32_t h = 0;
        bool claimed = false;
        if (valid) {
            const uint32_t node = pid[i];
            const uint32_t slot = node * (uint32_t)K + pdir[i];
            const uint32_t next = (i + 1 < steps) ? pid[i + 1] : (uint32_t)goal;
            const bool onb = ((onbest[node >> 5] >> (node & 31)) & 1u) && ((onbest[next >> 5] >> (next & 31)) & 1u);
            const unsigned long long want = (unsigned long long)(slot + 1u) | ((unsigned long long)group << 32) | (onb ? (1ull << 63) : 0ull);
            h = rankset_find_or_claim(rs, want, rankset_hash(slot, group) >> rs.shift, claimed);
        }
        const unsigned cm = __ballot_sync(FULL, claimed);
        if (cm) {   // one counter update per warp
            uint32_t at = 0;
            if (lane == __ffs(cm) - 1) at = atomicAdd(rs.count, (uint32_t)__popc(cm));
            at = __shfl_sync(FULL, at, __ffs(cm) - 1);
            const uint32_t mine = at + __popc(cm & ((1u << lane) - 1u));
            if (claimed) {
                if (mine < rs.limit) rs.list[mine] = h;
                else *over = 1u;   // beyond the claim limit: the block stays out of the list and is wiped by the sweep of the last apply launch
            }
        }
        if (valid && h != 0xFFFFFFFFu) atomicOr(rs.rows + (size_t)h * kRsRowWords + word, bit);
    }
}

// Sharded colonies: copy the blocks this rank claimed into its publish area (peer slab): pub[0] = count, pub[1] = overflow,
// blocks of kRsPubWords words from word 4.
__global__ void __launch_bounds__(256) k_rankset_publish(const IterState* st, RankSet rs, uint32_t* __restrict__ pub)
{
    if (!st->use_rankset) return;
    const uint32_t n = min(rs.count[0], rs.limit);
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t e = warp; e < n; e += nwarps) {
        const uint32_t h = rs.list[e];
        uint32_t* o = pub + 4 + (size_t)e * kRsPubWords;
        if (lane == 0) { const unsigned long long k = rs.key[h]; o[0] = (uint32_t)k; o[1] = (uint32_t)(k >> 32); }
        o[2 + lane] = rs.rows[(size_t)h * kRsRowWords + lane];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { pub[0] = n; pub[1] = rs.count[3]; }
}

// ... and OR every peer's published blocks into the local table (warp per block).  After this kernel the table, the
// list and the overflow flag are identical on every rank (up to the order of the list, which nothing depends on).
__global__ void __launch_bounds__(256) k_rankset_merge(PeerBarrier pb, const IterState* st, RankSet rs, const uint32_t* const* __restrict__ pubs, int npeers, int me)
{
    constexpr unsigned FULL = 0xffffffffu;
    if (!st->use_rankset) return;
    peer_barrier(pb, st, 2u);   // every rank has published its blocks
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    volatile uint32_t* over = rs.count + 3;
    for (int p = 0; p < npeers; p++) {
        if (p == me) continue;
        const uint32_t* pub = pubs[p];
        const uint32_t n = __ldcg(pub);
        if (__ldcg(pub + 1) != 0u && warp == 0 && lane == 0) *over = 1u;
        for (uint32_t e = warp; e < n; e += nwarps) {
            const uint32_t* in = pub + 4 + (size_t)e * kRsPubWords;
            const uint32_t w = __ldcg(in + 2 + lane);
            uint32_t h = 0xFFFFFFFFu;
            if (lane == 0 && *over == 0u) {
                const uint32_t k0 = __ldcg(in), k1 = __ldcg(in + 1);
                const unsigned long long want = (unsigned long long)k0 | ((unsigned long long)k1 << 32);
                bool claimed;
                h = rankset_find_or_claim(rs, want, rankset_hash(k0 - 1u, k1 & 0x7FFFFFFFu) >> rs.shift, claimed);
                if (claimed) {
                    const uint32_t at = atomicAdd(rs.count, 1u);
                    if (at < rs.limit) rs.list[at] = h; else *over = 1u;
                }
            }
            h = __shfl_sync(FULL, h, 0);
            if (h != 0xFFFFFFFFu && w) atomicOr(rs.rows + (size_t)h * kRsRowWords + lane, w);
        }
    }
}

// block of `want` (key with its on-best bit), or 0xFFFFFFFF.  Read-only: nothing is wiped while k_rankset_apply looks up.
__device__ __forceinline__ uint32_t rankset_find(const RankSet& rs, unsigned long long want, uint32_t h)
{
    for (uint32_t probes = 0; probes <= rs.rmask; probes++) {
        const unsigned long long k = __ldcg(rs.key + h);
        if (k == want) return h;
        if (k == 0ull) return 0xFFFFFFFFu;
        h = (h + 1) & rs.rmask;
    }
    return 0xFFFFFFFFu;
}

// The ordered chains, ONE launch for all rank groups.  A slot's chain must run group 0, 1, 2 ... (ascending ranks), so the
// block of the slot's LOWEST group is the slot's leader and processes the whole chain, looking the higher groups' blocks up
// in the table; the other blocks of the slot do nothing.  Lane per leader while the chain is one light block (a wandering
// colony: ~10^5 slots with a handful of ranks each); a leader with more than 64 ranks in its block or with further groups
// is handed to the whole warp: the 32 values of a word are fetched by the lanes at once and the dependent FADD chain runs on
// values exchanged by shuffle (a converged colony puts ~0.2*colony ranks on every slot of the best path).  Absent ranks
// contribute +0, the identity of the chain.
// groups_max == 1 (colonies up to 5120 ants): no look-ups happen, so every block is wiped as soon as it is consumed;
// otherwise k_rankset_clear follows (a wipe during the look-ups would cut other slots' probe chains).
__global__ void __launch_bounds__(256) k_rankset_apply(const IterState* st, float* tau, RankSet rs, float rho, DirtyFlags dirty, int groups_max)
{
    if (!st->use_rankset) return;
    const bool overflow = rs.count[3] != 0u;   // the table is incomplete: wipe only, k_deposit_serial applies the deposits
    const float base_new = __fmul_rn(st->base, rho);   // clean-tile field: a slot that still holds the sentinel is worth this after the evaporation
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const uint32_t n = min(rs.count[0], rs.limit);
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t groups = ((uint32_t)max(st->n_eligible, 1) + kRsGroupRanks - 1) / kRsGroupRanks;   // groups that can exist this iteration
    const bool wipe_here = groups_max == 1;
    // Consecutive list entries go to consecutive WARPS (entry = base + lane*nwarps + warp): the first ant to run claims
    // the whole best path in one stretch of the list, and those are exactly the heavy blocks — one per warp, not 32.
    for (uint32_t base = 0; base < n && !(overflow && !wipe_here); base += nwarps * 32u) {   // warp-uniform trips
        const uint32_t e = base + (uint32_t)lane * nwarps + warp;
        const bool has = e < n;
        uint32_t h = 0, slot = 0, flag = 0, group = 0;
        unsigned long long key = 0ull;
        if (has) {
            h = rs.list[e];
            key = rs.key[h];
            slot = (uint32_t)key - 1u;
            flag = (uint32_t)(key >> 63);
            group = ((uint32_t)(key >> 32)) & 0x7FFFFFFFu;
        }
        uint32_t* row = rs.rows + (size_t)h * kRsRowWords;
        bool leader = has && !overflow;
        bool more = false;   // the slot has blocks of higher groups
        if (leader && groups > 1) {
            const unsigned long long kbase = key & ~(0x7FFFFFFFull << 32);   // slot + on-best bit
            for (uint32_t g = group; g-- > 0 && leader;) leader = rankset_find(rs, kbase | ((unsigned long long)g << 32), rankset_hash(slot, g) >> rs.shift) == 0xFFFFFFFFu;
            for (uint32_t g = group + 1; g < groups && leader && !more; g++) more = rankset_find(rs, kbase | ((unsigned long long)g << 32), rankset_hash(slot, g) >> rs.shift) != 0xFFFFFFFFu;
        }
        int pc = 0;
        uint4 q[8];
        if (leader && !more) {
#pragma unroll
            for (int j = 0; j < 8; j++) { q[j] = reinterpret_cast<const uint4*>(row)[j]; pc += __popc(q[j].x) + __popc(q[j].y) + __popc(q[j].z) + __popc(q[j].w); }
        }
        const bool heavy = leader && (more || pc > 64);
        if (leader && !heavy) {
            const float* vt = rs.vtab + 2 * (size_t)group * kRsGroupRanks;
            float x = tau_or_base(tau[slot], base_new);
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const uint32_t wv[4] = {q[j].x, q[j].y, q[j].z, q[j].w};
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    uint32_t m = wv[c];
                    while (m) {
                        const int b = __ffs(m) - 1;
                        m &= m - 1;
                        x = __fadd_rn(x, vt[2 * ((j * 4 + c) * 32 + b) + flag]);
                    }
                }
            }
            tau[slot] = x;
            dirty.mark(slot);
        }
        unsigned hm = __ballot_sync(FULL, heavy);
        while (hm) {
            const int src = __ffs(hm) - 1;
            hm &= hm - 1;
            const uint32_t ss = __shfl_sync(FULL, slot, src);
            const uint32_t fs = __shfl_sync(FULL, flag, src);
            const uint32_t g0 = __shfl_sync(FULL, group, src);
            uint32_t hs = __shfl_sync(FULL, h, src);
            const unsigned long long kbase = (unsigned long long)(ss + 1u) | ((unsigned long long)fs << 63);
            float x = tau_or_base(tau[ss], base_new);
            for (uint32_t g = g0; g < groups; g++) {   // warp-uniform
                if (g != g0) {
                    uint32_t f = 0xFFFFFFFFu;
                    if (lane == 0) f = rankset_find(rs, kbase | ((unsigned long long)g << 32), rankset_hash(ss, g) >> rs.shift);
                    hs = __shfl_sync(FULL, f, 0);
                    if (hs == 0xFFFFFFFFu) continue;
                }
                const float* vt = rs.vtab + 2 * (size_t)g * kRsGroupRanks;
                const uint32_t mine = rs.rows[(size_t)hs * kRsRowWords + lane];   // the row: one coalesced load, lane j holds word j
                // all of the block's values first (32 independent loads per lane, one round trip), then the chain runs on shuffles alone
                float v[kRsRowWords];
#pragma unroll
                for (int w = 0; w < kRsRowWords; w++) {
                    const uint32_t m = __shfl_sync(FULL, mine, w);
                    v[w] = ((m >> lane) & 1u) ? vt[2 * (w * 32 + lane) + fs] : 0.0f;
                }
#pragma unroll
                for (int w = 0; w < kRsRowWords; w++) {
                    if (__shfl_sync(FULL, mine, w) == 0u) continue;   // warp-uniform
#pragma unroll
                    for (int i = 0; i < 32; i++) x = __fadd_rn(x, __shfl_sync(FULL, v[w], i));
                }
            }
            if (lane == 0) { tau[ss] = x; dirty.mark(ss); }
        }
        __syncwarp();
        if (has && wipe_here) {   // leave the table empty for the next iteration
#pragma unroll
            for (int j = 0; j < 8; j++) reinterpret_cast<uint4*>(row)[j] = make_uint4(0u, 0u, 0u, 0u);
            rs.key[h] = 0ull;
        }
    }
    if (!wipe_here) return;
    if (blockIdx.x == 0 && threadIdx.x == 0) rs.count[1] = overflow ? 0xFFFFFFFFu : n;
    if (overflow) {   // blocks claimed beyond the list (their indices were dropped): a sweep of the whole table finds them
        const size_t R = (size_t)rs.rmask + 1;
        for (size_t h = (size_t)blockIdx.x * blockDim.x + threadIdx.x; h < R; h += (size_t)gridDim.x * blockDim.x) {
            if (rs.key[h] == 0ull) continue;
            uint4* r4 = reinterpret_cast<uint4*>(rs.rows + h * kRsRowWords);
#pragma unroll
            for (int j = 0; j < 8; j++) r4[j] = make_uint4(0u, 0u, 0u, 0u);
            rs.key[h] = 0ull;
        }
    }
}

// groups_max > 1: after the chains, every listed block and its key are wiped for the next iteration (and, after an overflow,
// the blocks that did not make it into the list: a sweep of the whole table finds them)
__global__ void __launch_bounds__(256) k_rankset_clear(const IterState* st, RankSet rs)
{
    if (!st->use_rankset) return;
    const uint32_t n = min(rs.count[0], rs.limit);
    const bool overflow = rs.count[3] != 0u;
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t e = warp; e < n; e += nwarps) {   // warp per block: one coalesced 128-byte store
        const uint32_t h = rs.list[e];
        rs.rows[(size_t)h * kRsRowWords + lane] = 0u;
        __syncwarp();
        if (lane == 0) rs.key[h] = 0ull;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) rs.count[1] = overflow ? 0xFFFFFFFFu : n;
    if (overflow) {
        const size_t R = (size_t)rs.rmask + 1;
        for (size_t h = (size_t)blockIdx.x * blockDim.x + threadIdx.x; h < R; h += (size_t)gridDim.x * blockDim.x) {
            if (rs.key[h] == 0ull) continue;
            uint4* r4 = reinterpret_cast<uint4*>(rs.rows + h * kRsRowWords);
#pragma unroll
            for (int j = 0; j < 8; j++) r4[j] = make_uint4(0u, 0u, 0u, 0u);
            rs.key[h] = 0ull;
        }
    }
}

// Overflow only: the deposits of the iteration exactly as the reference orders them (:275-280) — eligible ants front to
// back, one CTA-wide barrier per ant; within an ant every slot occurs once, so its steps run in parallel.  Single CTA.
// ids_tab/dirs_tab: every rank's trail buffers (sharded colonies; a one-entry table on a single GPU).
__global__ void __launch_bounds__(1024) k_deposit_serial(const IterState* st, const uint32_t* __restrict__ rank_keys, const uint32_t* __restrict__ rank_vals,
                                                          const uint32_t* const* __restrict__ ids_tab, const uint8_t* const* __restrict__ dirs_tab, int cap,
                                                          int shard_chunk, int goal, const float* __restrict__ Ltab, const uint32_t* __restrict__ onbest,
                                                          const uint32_t* __restrict__ over, float* tau, float rho, DirtyFlags dirty, int K,
                                                          const int* __restrict__ steps26)
{
    if (!st->use_rankset || *over == 0u) return;
    const float base_new = __fmul_rn(st->base, rho);
    const int n = st->n_eligible;
    const float lambda = st->lambda, Q = st->Q;
    const float elite = __fdiv_rn(__fmul_rn(__fmul_rn(1.0f, lambda), Q), st->best_L);
    for (int r = 0; r < n; r++) {
        const int ant_global = (int)rank_vals[r];
        const int steps = steps26 ? steps26[ant_global] : (int)rank_keys[r];
        const float L_ant = steps26 ? __uint_as_float(rank_keys[r]) : Ltab[steps];
        const float base = __fdiv_rn(__fmul_rn(__fsub_rn(lambda, (float)(r + 1)), Q), L_ant);
        const float with_elite = __fadd_rn(base, elite), without = __fadd_rn(base, 0.0f);
        const int owner = ant_global / shard_chunk;
        const uint32_t* pid = ids_tab[owner] + (size_t)(ant_global - owner * shard_chunk) * cap;
        const uint8_t* pdir = dirs_tab[owner] + (size_t)(ant_global - owner * shard_chunk) * cap;
        for (int i = threadIdx.x; i < steps; i += blockDim.x) {
            const uint32_t node = pid[i];
            const uint32_t next = (i + 1 < steps) ? pid[i + 1] : (uint32_t)goal;
            const bool onb = ((onbest[node >> 5] >> (node & 31)) & 1u) && ((onbest[next >> 5] >> (next & 31)) & 1u);
            const uint32_t slot = node * (uint32_t)K + pdir[i];
            tau[slot] = __fadd_rn(tau_or_base(tau[slot], base_new), onb ? with_elite : without);
            dirty.mark(slot);
        }
        __syncthreads();
    }
}

}  // namespace wr
