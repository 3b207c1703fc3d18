// Concurrent searches (batch.cuh) for the K = 26 neighbourhood (walk26.cuh).  Everything but the walk's inputs is shared with
// K = 6: the (query, node) pheromone table with 128-byte entries (key, the node's 26 slots in the slot26 enumeration, 4 unused
// words), k_batch_rank on the bits of each ant's L, k_batch_deposit with the ant's own L and the 0..25 direction of a step.
// The walk is k_walk26<Batch26, GLOBAL>: k_walk26's step with its inputs taken from where a batch keeps them.
#pragma once
#include "batch.cuh"
#include "walk26.cuh"

namespace wr {

// Inputs of k_walk26 over a batch; a work item is (query, ant) = query * colony_max + ant.
//   * tau: word 2 + s of the (query, node) entry, or the scalar if the node has none;
//   * open: neighbour in bounds and free in the grid's occupancy bits;
//   * factor: heur26, the function k_heuristic26 tabulates, per step for the query's goal, so no dense N x 26 table is
//     built per goal;
//   * draws: Philox with the query's search index and the ant's index within its query;
//   * parking: the HBM tables come from a pool; when it is exhausted the batch is marked failed and the ant dies here.
struct Batch26 {
    using Args = BatchArgs;
    int kk, stride_k;
    bool active;                      // one of the 26 slot lanes
    int rx, ry, rz, rxy;
    const float *xs, *ys, *zs;
    const uint32_t* ent;
    const uint32_t* occ;
    int shift;
    uint32_t tmask;
    float beta;
    // the bound ant
    uint32_t qi, qhash;
    float gxv, gyv, gzv;
    int start, sx, sy, sz, goal;
    uint32_t ant, stream_word, block_hi;
    uint32_t row;

    __device__ __forceinline__ Batch26(const BatchArgs& a, int kk_, bool active_, int stride)
        : kk(kk_), stride_k(stride), active(active_), rx(a.rx), ry(a.ry), rz(a.rz), rxy(a.rx * a.ry), xs(a.coords), ys(a.coords + a.rx), zs(a.coords + a.rx + a.ry),
          ent(a.tab.ent), occ(a.occ), shift(a.tab.shift), tmask(a.tab.tmask), beta(a.beta)
    {
    }
    __device__ __forceinline__ unsigned items(const BatchArgs& a, const IterState* st, bool resumed) const
    {
        return resumed ? min(st->overflow_n, a.pool) : (unsigned)(a.nq * a.colony_max);
    }
    // false: the ant is beyond this iteration's colony of its query
    __device__ __forceinline__ bool bind(const BatchArgs& a, uint32_t item, bool resumed)
    {
        qi = item / (uint32_t)a.colony_max;
        ant = item - qi * (uint32_t)a.colony_max;
        const BatchQuery& bq = a.qs[qi];
        if (!resumed && (int)ant >= bq.colony) return false;
        start = bq.start; goal = bq.goal;
        sx = start % rx; sy = (start % rxy) / rx; sz = start / rxy;
        stream_word = bq.stream_word; block_hi = bq.block_hi;
        qhash = qi * 0x85EBCA6Bu + (qi << 13);
        gxv = __ldg(xs + goal % rx); gyv = __ldg(ys + (goal % rxy) / rx); gzv = __ldg(zs + goal / rxy);
        row = item;
        return true;
    }
    __device__ __forceinline__ float tau(int cur) const
    {
        const uint32_t want0 = (uint32_t)cur + 1u;
        uint32_t eh = (((uint32_t)cur * 2654435761u) ^ qhash) >> shift;
        const uint32_t* e = ent + (size_t)eh * kBatchEntryWords26;
        uint2 ekey = __ldg(reinterpret_cast<const uint2*>(e));
        uint32_t etau = __ldg(e + 2 + kk);
        uint32_t probes = 0;
        while ((ekey.x != want0 || (ekey.y & 0x7FFFFFFFu) != qi) && (ekey.x | ekey.y) != 0u) {   // rare: linear probing at load <= 1/2
            if (++probes > tmask) { ekey = make_uint2(0u, 0u); break; }   // a full table: only in a batch that has already failed and will be re-run
            eh = (eh + 1) & tmask;
            e = ent + (size_t)eh * kBatchEntryWords26;
            ekey = __ldg(reinterpret_cast<const uint2*>(e));
            etau = __ldg(e + 2 + kk);
        }
        return (ekey.x | ekey.y) != 0u ? __uint_as_float(etau) : __uint_as_float(kSentinelBits);
    }
    __device__ __forceinline__ bool open(int cur, int x, int y, int z, int nx, int ny, int nz, float& heur) const
    {
        const bool inb = active && nx >= 0 && nx < rx && ny >= 0 && ny < ry && nz >= 0 && nz < rz;
        bool open_k = false;
        heur = 0.0f;
        if (inb) {
            const uint32_t nid = (uint32_t)(cur + stride_k);
            if (!((__ldg(occ + (nid >> 5)) >> (nid & 31)) & 1u)) {
                heur = heur26(__ldg(xs + x), __ldg(ys + y), __ldg(zs + z), gxv, gyv, gzv, __ldg(xs + nx), __ldg(ys + ny), __ldg(zs + nz), beta);
                open_k = heur != kClosedSlot;   // Dense26's test on the tabulated factor; NaN (duplicate plane) stays open, as in the reference
            }
        }
        return open_k;
    }
    __device__ __forceinline__ bool park(const BatchArgs& a, int o, int lane) const
    {
        if ((uint32_t)o < a.pool) return true;
        if (lane == 0) a.tab.count[1] = 1u;   // pool exhausted: the chunk fails and runs as the sequential loop
        return false;
    }
};

}  // namespace wr
