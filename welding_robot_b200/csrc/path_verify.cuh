// Converged colony: check the best path against roulette thresholds instead of walking it step by step.
//
// An ant that has followed the best path up to position t stands where every other such ant stands: node best[t], visited
// set best[0..t], the same tau and factor rows.  Its six scores, the roulette total and the suffix sums are therefore the
// same for all of them; only its draw u differs.  It takes the path's next slot d_t iff, with r = u * total_t,
//     hi_t >= r && !(lo_t >= r)
// where hi_t is the suffix sum of slot d_t and lo_t the largest suffix sum of a candidate slot above d_t (-1: none) — the
// comparisons k_walk3's step makes, so the outcome is the same bit for bit.  Draws are a pure function of (search,
// iteration, ant, step), so the steps of one ant can be checked independently, many at a time.
//   k_path_thresholds  once per iteration: {total, hi, lo} of every position and the verifiable prefix D
//   k_path_verify      per ant: the first step that fails (dev), and the trail prefix copied from the best path
//   k_walk3<*, 0>      resumes each warp at min floor8(dev) of its ants (walk3.cuh), or only books ants that followed it all
#pragma once
#include "walk3.cuh"

namespace wr {

constexpr int kPathThreads = 1024;    // k_path_thresholds: one CTA
constexpr int kVerifyThreads = 256;   // k_path_verify: one warp per ant

// node / tile -> first position on the path: open addressing, key 0 = empty, {key, position}
__device__ __forceinline__ void pos_insert(uint2* map, uint32_t mask, uint32_t key, uint32_t p)
{
    uint32_t slot = tile_hash(key, mask + 1);
    while (true) {
        const uint32_t old = atomicCAS(&map[slot].x, 0u, key);
        if (old == 0u || old == key) { atomicMin(&map[slot].y, p); return; }
        slot = (slot + 1) & mask;
    }
}
__device__ __forceinline__ uint32_t pos_lookup(const uint2* map, uint32_t mask, uint32_t key)
{
    uint32_t slot = tile_hash(key, mask + 1);
    while (true) {
        const uint2 e = map[slot];
        if (e.x == key) return e.y;
        if (e.x == 0u) return 0xFFFFFFFFu;
        slot = (slot + 1) & mask;
    }
}

// Thresholds of every best-path position t < best_n - 1 and the verifiable prefix D: the first t whose step k_walk3 might
// not take the way thr[t] describes (any content of best_ids / best_dirs is checked, so a stale or broken path only
// shortens D).  pv[0] = {D, best_n - 1 if D == best_n - 1 else -1}; pv[1].x = 1 tells the ranking that follows that this
// iteration's dev values are fresh (k_rank_small consumes it).  map: 2 * map_entries entries (a power of two >= 2 * (cap + 1)).
__global__ void __launch_bounds__(kPathThreads) k_path_thresholds(const IterState* st, const int* best_n, const uint32_t* __restrict__ best_ids,
                                                                  const uint8_t* __restrict__ best_dirs, const float* __restrict__ tau,
                                                                  const float* __restrict__ heur, int alpha, int rx, int ry, int rz, int start, int goal,
                                                                  int cap, uint32_t limit, uint2* map, uint32_t map_entries, float4* thr, int2* pv)
{
    __shared__ int s_fail;
    __shared__ uint32_t s_warp[kPathThreads / 32];
    const int n = *best_n;
    if (n < 2 || n > cap + 1) {   // no best path yet
        if (threadIdx.x == 0) { pv[0] = make_int2(0, -1); pv[1] = make_int2(1, 0); }
        return;
    }
    const uint32_t N = (uint32_t)rx * (uint32_t)ry * (uint32_t)rz;
    const int rxy = rx * ry;
    const float base = st->base;
    uint32_t M = 2;
    while (M < 2u * (uint32_t)n) M <<= 1;
    M = min(M, map_entries);
    uint2* nmap = map;                 // node + 1 -> first position
    uint2* tmap = map + map_entries;   // tile key -> first position
    for (uint32_t i = threadIdx.x; i < M; i += blockDim.x) { nmap[i] = make_uint2(0u, 0xFFFFFFFFu); tmap[i] = make_uint2(0u, 0xFFFFFFFFu); }
    if (threadIdx.x == 0) s_fail = n - 1;
    __syncthreads();
    auto tile_of = [&](uint32_t node) {
        return (pack_xyz((int)(node % rx), (int)((node % rxy) / rx), (int)(node / rxy)) & kPackKey) | kKeyTag;
    };
    for (int p = threadIdx.x; p < n; p += blockDim.x) {
        const uint32_t node = best_ids[p];
        if (node >= N) continue;       // such a position fails below
        pos_insert(nmap, M - 1, node + 1, (uint32_t)p);
        pos_insert(tmap, M - 1, tile_of(node), (uint32_t)p);
    }
    __syncthreads();

    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t carry = 0;   // distinct tiles of the positions before this chunk
    for (int c0 = 0; c0 < n; c0 += blockDim.x) {
        const int t = c0 + threadIdx.x;
        const uint32_t node = t < n ? best_ids[t] : 0xFFFFFFFFu;
        const bool valid = node < N;
        // tiles of best[0..t] (k_walk3's ntiles at step t): a block-wide inclusive count of the tiles' first positions
        const bool first = valid && pos_lookup(tmap, M - 1, tile_of(node)) == (uint32_t)t;
        const unsigned fb = __ballot_sync(0xffffffffu, first);
        if (lane == 31) s_warp[wid] = __popc(fb);
        __syncthreads();
        uint32_t tiles = carry + __popc(fb & (0xffffffffu >> (31 - lane))), chunk_tiles = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) {
            const uint32_t c = s_warp[w];
            tiles += w < wid ? c : 0u;
            chunk_tiles += c;
        }
        carry += chunk_tiles;
        if (t < n - 1) {
            const uint32_t next = best_ids[t + 1];
            const int d = best_dirs[t];
            // the ant must still be walking when it decides step t: at the start (t = 0), not yet arrived, below the step cap,
            // and its visited table not full (k_walk3's `full` at step t is ntiles > limit; it parks the ant after that step)
            bool ok = valid && (t > 0 || (int)node == start) && t + 1 < cap && tiles <= limit && d < 6 && (((int)next == goal) == (t + 1 == n - 1));
            float total = 0.0f, hi = 0.0f, lo = -1.0f;
            if (ok) {
                float v[6];
                bool cand[6], cand_d = false;
                uint32_t nb_d = 0;
#pragma unroll
                for (int k = 0; k < 6; k++) {
                    const int dxk = (k == 3) - (k == 2), dyk = (k == 4) - (k == 1), dzk = (k == 5) - (k == 0);
                    const float h = heur[(size_t)node * 6 + k];
                    // open: in bounds and free (folded into the factor table); candidate: open and not in best[0..t]
                    const bool open = h != kClosedSlot;
                    const uint32_t nb = node + (uint32_t)(dxk + dyk * rx + dzk * rxy);
                    cand[k] = open && pos_lookup(nmap, M - 1, nb + 1) > (uint32_t)t;
                    if (k == d) { cand_d = cand[k]; nb_d = nb; }
                    v[k] = alpha == 1 ? slot_score<true>(cand[k], tau[(size_t)node * 6 + k], h, base, alpha)
                                      : slot_score<false>(cand[k], tau[(size_t)node * 6 + k], h, base, alpha);
                }
                total = roulette_total(v[0], v[1], v[2], v[3], v[4], v[5]);
                bool finite = isfinite(total);
#pragma unroll
                for (int k = 0; k < 6; k++) {
                    const float s = roulette_suffix(v[0], v[1], v[2], v[3], v[4], v[5], k <= 4 ? ~0u : 0u, k <= 3 ? ~0u : 0u, k <= 2 ? ~0u : 0u,
                                                    k <= 1 ? ~0u : 0u, k <= 0 ? ~0u : 0u);
                    finite = finite && isfinite(s);
                    if (k == d) hi = s;
                    if (k > d && cand[k]) lo = fmaxf(lo, s);
                }
                ok = finite && cand_d && next == nb_d;
            }
            thr[t] = make_float4(total, hi, lo, 0.0f);
            if (!ok) atomicMin(&s_fail, t);
        }
        __syncthreads();   // s_warp is rewritten by the next chunk
    }
    if (threadIdx.x == 0) {
        const int D = s_fail;
        pv[0] = make_int2(D, D == n - 1 ? n - 1 : -1);
        pv[1] = make_int2(1, 0);
    }
}

// One warp per ant of this shard: dev = the first step < D whose draw leaves the best path (D if none; the ant is complete
// when D == best_n - 1 as well).  Lane l checks Philox blocks l, l + 32, ... (steps 4b..4b+3) in k_walk3's draw order.  The
// trail rows k_walk3 will not rewrite are copied from the best path: all best_n - 1 steps of a complete ant, else [0, floor8(dev)).
__global__ void __launch_bounds__(kVerifyThreads) k_path_verify(const IterState* st, const int2* pv, const float4* __restrict__ thr,
                                                                const uint32_t* __restrict__ best_ids, const uint8_t* __restrict__ best_dirs,
                                                                uint32_t seed_lo, uint32_t seed_hi, uint32_t stream_word, uint32_t block_hi,
                                                                int shard_first, int shard_chunk, int cap, int* dev, uint32_t* path_ids, uint8_t* path_dirs)
{
    const int ant = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    const int local_n = min(max(st->colony - shard_first, 0), shard_chunk);
    if (ant >= local_n) return;   // warp-uniform
    const int2 v = *pv;
    const int D = v.x;
    const uint32_t iter = (uint32_t)st->iter, ant_global = (uint32_t)(shard_first + ant);
    int d = D;
    for (int b0 = 0; 4 * b0 < D; b0 += 32) {
        const int b = b0 + lane;
        int fs = INT_MAX;
        if (4 * b < D) {
            uint32_t w[4];
            philox4(iter, ant_global, (uint32_t)b | block_hi, stream_word, seed_lo, seed_hi, w[0], w[1], w[2], w[3]);
#pragma unroll
            for (int j = 3; j >= 0; j--) {
                const int s = 4 * b + j;
                const float u = __fmul_rn(__int2float_rn((int)(w[j] >> 1)), 4.656612873077392578125e-10f);
                if (s < D) {
                    const float4 h = thr[s];
                    const float r = __fmul_rn(u, h.x);
                    if (!(h.y >= r && !(h.z >= r))) fs = s;
                }
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, fs != INT_MAX);
        if (m) { d = __shfl_sync(0xffffffffu, fs, __ffs(m) - 1); break; }
    }
    if (lane == 0) dev[ant] = d;
    const int L = d == v.y ? d : (d & ~7);
    uint32_t* pid = path_ids + (size_t)ant * cap;
    uint8_t* pdir = path_dirs + (size_t)ant * cap;
    for (int s = lane; s < L; s += 32) { pid[s] = best_ids[s]; pdir[s] = best_dirs[s]; }
}

}  // namespace wr
