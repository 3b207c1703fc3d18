// Concurrent searches (batch.cuh) for the K = 26 neighbourhood (walk26.cuh).  Everything but the walk is shared with K = 6:
// the (query, node) pheromone table with 128-byte entries (key, the node's 26 slots in the slot26 enumeration, 4 unused
// words), k_batch_rank on the bits of each ant's L, k_batch_deposit with the ant's own L and the 0..25 direction of a step.
//
//   k_walk_batch26   the step of k_walk26 — one ant per warp, lane s < 26 owns slot s, unpacked coordinates (no axis limit),
//                    the same 4x4x4-tile visited tables — with its inputs taken from where a batch keeps them:
//                      * tau: word 2 + s of the (query, node) entry, or the scalar if the node has none;
//                      * open: neighbour in bounds and free in the grid's occupancy bits;
//                      * heuristic: heur26 (walk26.cuh), the function k_heuristic26 tabulates, per step for the query's goal,
//                        so no dense N x 26 table is built per goal;
//                      * draws: Philox with the query's search index and the ant's index within its query.
//                    GLOBAL = false is pass 1 (shared-memory tables); an ant that fills its table to 3/4 parks {node, steps,
//                    tiles, L} with its visited set in an HBM table from a pool, and GLOBAL = true resumes it from there.
#pragma once
#include "batch.cuh"
#include "walk26.cuh"

namespace wr {

template <bool GLOBAL>
__global__ void __launch_bounds__(kWalk26Threads) k_walk_batch26(BatchArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int w = threadIdx.x >> 5;
    const int tlog2 = GLOBAL ? a.gtable_log2 : a.table_log2;
    const int E = 1 << tlog2;
    const int hshift = 32 - tlog2;

    unsigned long long* masks = nullptr;
    uint32_t* keys = nullptr;
    if (!GLOBAL) {
        unsigned long long* mbase = reinterpret_cast<unsigned long long*>(smem_raw);
        masks = mbase + (size_t)w * E;
        keys = reinterpret_cast<uint32_t*>(mbase + (size_t)kWalk26Ants * E) + (size_t)w * E;
    }

    const int rx = a.rx, ry = a.ry, rz = a.rz;
    const int rxy = rx * ry;
    const int TX = (rx + 3) >> 2, TY = (ry + 3) >> 2;
    const bool active = lane < kK26;
    const int kk = active ? lane : kK26 - 1;             // idle lanes re-read slot 25 (same line)
    int dxk, dyk, dzk;
    slot26(kk, dxk, dyk, dzk);
    const int stride_k = dxk + dyk * rx + dzk * rxy;
    const int type_k = (dxk != 0) + (dyk != 0) + (dzk != 0);
    const float dist_k = type_k == 1 ? a.precision : (type_k == 2 ? __fmul_rn(a.precision, 1.414f) : __fmul_rn(a.precision, 1.732f));
    const float* xs = a.coords;
    const float* ys = xs + rx;
    const float* zs = ys + ry;
    const bool alpha1 = a.alpha == 1;
    const float beta = a.beta;
    const int cap = a.cap;

    IterState* st = a.st;
    const uint32_t iter = (uint32_t)st->iter;
    const float base_now = st->base;
    const unsigned n_items = GLOBAL ? min(st->overflow_n, a.pool) : (unsigned)(a.nq * a.colony_max);
    const int limit = (E >> 2) * 3;
    const uint32_t* ent = a.tab.ent;

    unsigned long long c_steps = 0, c_ants = 0, c_arrived = 0, c_nocand = 0, c_fall = 0, c_cap = 0, c_over = 0;

    while (true) {
        unsigned q = 0;
        if (lane == 0) q = atomicAdd(GLOBAL ? &st->queue2 : &st->queue, 1u);
        q = __shfl_sync(FULL, q, 0);
        if (q >= n_items) break;                                         // warp-uniform
        const uint32_t ga = GLOBAL ? a.overflow_list[q] : q;             // query * colony_max + ant
        const uint32_t qi = ga / (uint32_t)a.colony_max;
        const int ant = (int)(ga - qi * (uint32_t)a.colony_max);
        const BatchQuery& bq = a.qs[qi];
        if (!GLOBAL && ant >= bq.colony) continue;                       // this iteration's colony of the query is smaller
        const int goal = bq.goal;
        const uint32_t stream_word = bq.stream_word, block_hi = bq.block_hi;
        const uint32_t qhash = qi * 0x85EBCA6Bu + (qi << 13);
        const float gxv = __ldg(xs + goal % rx), gyv = __ldg(ys + (goal % rxy) / rx), gzv = __ldg(zs + goal / rxy);

        int cur = bq.start, steps = 0, ntiles = 1;
        int x = cur % rx, y = (cur % rxy) / rx, z = cur / rxy;
        float L = 0.0f;                                   // addStartNode :81-86
        uint32_t rw0 = 0, rw1 = 0, rw2 = 0, rw3 = 0;
        if (GLOBAL) {   // resume a parked ant: its visited set already lives in HBM table q
            keys = a.gkeys + (size_t)q * E;
            masks = a.gtab + (size_t)q * E;
            const int4 r = a.resume[q];
            cur = r.x; steps = r.y; ntiles = r.z; L = __int_as_float(r.w);
            z = cur / rxy; y = (cur % rxy) / rx; x = cur % rx;
            philox4(iter, (uint32_t)ant, ((uint32_t)steps >> 2) | block_hi, stream_word, a.seed_lo, a.seed_hi, rw0, rw1, rw2, rw3);
        } else {
            for (int i = lane; i < E; i += 32) keys[i] = kEmptyKey;
            __syncwarp();
            if (lane == 0) {
                const uint32_t tile = (uint32_t)(((z >> 2) * TY + (y >> 2)) * TX + (x >> 2));
                const unsigned bit = ((z & 3) << 4) | ((y & 3) << 2) | (x & 3);
                const unsigned slot = (tile * 2654435761u) >> hshift;
                keys[slot] = tile; masks[slot] = 1ull << bit;
            }
        }
        __syncwarp();

        int result = -1;   // >= 0: steps of an ant that arrived, -1: dead, -2: parked (pass 2 finishes it)
        int reason = 0;    // 1 no candidate, 2 roulette fall-through, 3 step cap
        uint32_t* pid = a.path_ids + (size_t)ga * cap;
        uint8_t* pdir = a.path_dirs + (size_t)ga * cap;

        while (true) {
            if (steps >= cap) { reason = 3; break; }   // step cap (a deviation the oracle mirrors)
            // ---- pheromone of slot kk: the (query, node) entry, or the scalar if it has none --------------------------
            const uint32_t want0 = (uint32_t)cur + 1u;
            uint32_t eh = (((uint32_t)cur * 2654435761u) ^ qhash) >> a.tab.shift;
            const uint32_t* e = ent + (size_t)eh * kBatchEntryWords26;
            uint2 ekey = __ldg(reinterpret_cast<const uint2*>(e));
            uint32_t etau = __ldg(e + 2 + kk);
            uint32_t probes = 0;
            while ((ekey.x != want0 || (ekey.y & 0x7FFFFFFFu) != qi) && (ekey.x | ekey.y) != 0u) {   // rare: linear probing at load <= 1/2
                if (++probes > a.tab.tmask) { ekey = make_uint2(0u, 0u); break; }   // a full table: only in a batch that has already failed and will be re-run
                eh = (eh + 1) & a.tab.tmask;
                e = ent + (size_t)eh * kBatchEntryWords26;
                ekey = __ldg(reinterpret_cast<const uint2*>(e));
                etau = __ldg(e + 2 + kk);
            }
            const float tau_k = tau_or_base((ekey.x | ekey.y) != 0u ? __uint_as_float(etau) : __uint_as_float(kSentinelBits), base_now);
            if ((steps & 3) == 0) philox4(iter, (uint32_t)ant, ((uint32_t)steps >> 2) | block_hi, stream_word, a.seed_lo, a.seed_hi, rw0, rw1, rw2, rw3);
            const uint32_t rsel = (steps & 2) ? ((steps & 1) ? rw3 : rw2) : ((steps & 1) ? rw1 : rw0);
            const float u = __fmul_rn(__int2float_rn((int)(rsel >> 1)), 4.656612873077392578125e-10f);   // (float)rand()/(float)RAND_MAX :169
            // ---- neighbour of this lane: open (in bounds and free), geometric factor, tabu probe ----
            const int nx = x + dxk, ny = y + dyk, nz = z + dzk;
            const bool inb = active && nx >= 0 && nx < rx && ny >= 0 && ny < ry && nz >= 0 && nz < rz;
            bool open_k = false;
            float heur_k = 0.0f;
            if (inb) {
                const uint32_t nid = (uint32_t)(cur + stride_k);
                if (!((__ldg(a.occ + (nid >> 5)) >> (nid & 31)) & 1u)) {
                    heur_k = heur26(__ldg(xs + x), __ldg(ys + y), __ldg(zs + z), gxv, gyv, gzv, __ldg(xs + nx), __ldg(ys + ny), __ldg(zs + nz), beta);
                    open_k = heur_k != kClosedSlot;   // k_walk26's test on the tabulated factor; NaN (duplicate plane) stays open, as in the reference
                }
            }
            const uint32_t tile = (uint32_t)(((nz >> 2) * TY + (ny >> 2)) * TX + (nx >> 2));
            const unsigned bit = ((nz & 3) << 4) | ((ny & 3) << 2) | (nx & 3);
            unsigned slot = (tile * 2654435761u) >> hshift;
            uint32_t kf = keys[slot];
            unsigned long long mm = masks[slot];
            while (open_k && kf != tile && kf != kEmptyKey) {
                slot = (slot + 1) & (E - 1);
                kf = keys[slot]; mm = masks[slot];
            }
            const bool found = kf == tile;
            const bool cand = open_k && !(found && ((mm >> bit) & 1ull));
            const float tpow = alpha1 ? tau_k : pow_int(tau_k, a.alpha);
            const float info = cand ? __fmul_rn(tpow, heur_k) : 0.0f;   // :154; +0 is the identity of both chains below
            const unsigned cb = __ballot_sync(FULL, cand);
            // ---- roulette in the reference's order (:155 ascending total, :172-181 descending prob_sum) ----
            float v[kK26];
#pragma unroll
            for (int i = 0; i < kK26; i++) v[i] = __shfl_sync(FULL, info, i);
            float total = 0.0f;
#pragma unroll
            for (int i = 0; i < kK26; i++) total = __fadd_rn(total, v[i]);
            const float rnd = __fmul_rn(u, total);
            float run = 0.0f, mine = 0.0f;
#pragma unroll
            for (int i = kK26 - 1; i >= 0; i--) {
                run = __fadd_rn(run, v[i]);
                mine = (i == lane) ? run : mine;
            }
            const bool pick = cand && (mine >= rnd);
            const unsigned pb = __ballot_sync(FULL, pick);
            if (pb == 0) { reason = cb == 0 ? 1 : 2; break; }   // :162-166 / fall-through :191-192 (NaN, rounding)
            const int c = 31 - __clz((int)pb);                  // first hit scanning 25 -> 0
            // ---- addNextNode (:73-79) ----
            if (lane == 0) { pid[steps] = (uint32_t)cur; pdir[steps] = (uint8_t)c; }
            if (lane == c) { keys[slot] = tile; masks[slot] = found ? (mm | (1ull << bit)) : (1ull << bit); }
            const unsigned fb = __ballot_sync(FULL, found);
            const int newtile = (int)(((fb >> c) & 1u) ^ 1u);
            cur += __shfl_sync(FULL, stride_k, c);
            x += __shfl_sync(FULL, dxk, c); y += __shfl_sync(FULL, dyk, c); z += __shfl_sync(FULL, dzk, c);
            L = __fadd_rn(L, __shfl_sync(FULL, dist_k, c));   // :78
            steps++;
            ntiles += newtile;
            __syncwarp();
            if (cur == goal) { result = steps; break; }         // :182-186
            if (!GLOBAL && newtile && ntiles > limit) {          // rare: shared-memory table 3/4 full -> park for pass 2
                int o = 0;
                if (lane == 0) o = (int)atomicAdd(&st->overflow_n, 1u);
                o = __shfl_sync(FULL, o, 0);
                if ((uint32_t)o >= a.pool) {                     // pool exhausted: the chunk fails and runs as the sequential loop
                    if (lane == 0) a.tab.count[1] = 1u;
                    break;
                }
                const int Eg = 1 << a.gtable_log2, gsh = 32 - a.gtable_log2;
                uint32_t* nkeys = a.gkeys + (size_t)o * Eg;
                unsigned long long* nmasks = a.gtab + (size_t)o * Eg;
                for (int i = lane; i < Eg; i += 32) nkeys[i] = kEmptyKey;
                __syncwarp();
                for (int i = lane; i < E; i += 32) {
                    const uint32_t t = keys[i];
                    if (t == kEmptyKey) continue;
                    unsigned sl = (t * 2654435761u) >> gsh;
                    while (atomicCAS(&nkeys[sl], kEmptyKey, t) != kEmptyKey) sl = (sl + 1) & (Eg - 1);
                    nmasks[sl] = masks[i];
                }
                if (lane == 0) {
                    a.resume[o] = make_int4(cur, steps, ntiles, __float_as_int(L));
                    a.overflow_list[o] = ga;
                }
                result = -2;
                break;
            }
        }
        __syncwarp();
        if (result == -2) {
            c_over++;   // its steps are counted by pass 2
        } else {
            if (lane == 0) {
                a.ant_steps[ga] = result;
                a.ant_L[ga] = result >= 0 ? L : INFINITY;   // setDeadEnd :88-91
            }
            c_steps += (unsigned long long)steps; c_ants++;
            c_arrived += result >= 0 ? 1 : 0;
            c_nocand += (result < 0 && reason == 1) ? 1 : 0;
            c_fall += (result < 0 && reason == 2) ? 1 : 0;
            c_cap += (result < 0 && reason == 3) ? 1 : 0;
        }
        __syncwarp();
    }
    if (lane == 0) {
        if (c_steps) atomicAdd(&st->cnt[0], c_steps);
        if (c_ants) atomicAdd(&st->cnt[1], c_ants);
        if (c_arrived) atomicAdd(&st->cnt[2], c_arrived);
        if (c_nocand) atomicAdd(&st->cnt[3], c_nocand);
        if (c_fall) atomicAdd(&st->cnt[4], c_fall);
        if (c_cap) atomicAdd(&st->cnt[5], c_cap);
        if (c_over) atomicAdd(&st->cnt[8], c_over);
    }
}

}  // namespace wr
