// K = 26 neighbourhood — the extension the reference scaffolds and then disables (core/ACSRank_3D.hpp:355-389: edge and
// corner neighbours get `distance = 0` and are skipped; the intended lengths `precision*1.414f` / `precision*1.732f` are
// the commented-out values at :381 and :384).  The CPU oracle (oracle/wr_oracle.cpp, K = 26) is the specification: the
// same enumeration order as :355-359 with the centre left out, every slot evaporated, L accumulated per step.
//
//   slot s in [0,26):  i = s < 13 ? s : s+1;  dz = i/9 - 1, dy = (i/3)%3 - 1, dx = i%3 - 1      (z outer, y, x inner)
//
//   k_tau_init26     initFromGridMap :391-401 for 26 slots per node
//   k_heuristic26    1 + beta*cos(theta) per (node, slot, goal); closed slots carry the sentinel
//   k_walk26         one ant per WARP: lane s < 26 owns slot s — the node's 26 pheromone values (104 contiguous bytes) and
//                    its 26 heuristic factors are one coalesced request each; the roulette re-adds the 26 scores in the
//                    reference's order (ascending total, descending prob_sum) from values exchanged by shuffle
//   ranking          an ant's length is no longer a function of its step count (three step lengths, float sums in path
//                    order), so the colony is ranked by the bits of L (non-negative floats order like their bit patterns;
//                    +inf for a dead ant): rank_small.cuh with ant_L != nullptr
// Algorithmic bytes per ant-step (SURVEY.md section 8d): 4*26 tau + 26/8 occupancy + 4 id + 1 slot = 112 B.
#pragma once
#include "acs_kernels.cuh"
#include "walk3.cuh"

namespace wr {

constexpr int kK26 = 26;
constexpr int kWalk26Threads = 128;                 // 4 warps = 4 ants per CTA
constexpr int kWalk26Ants = kWalk26Threads / 32;

__host__ __device__ __forceinline__ void slot26(int s, int& dx, int& dy, int& dz)
{
    const int i = s < 13 ? s : s + 1;
    dz = i / 9 - 1; dy = (i / 3) % 3 - 1; dx = i % 3 - 1;
}

__global__ void __launch_bounds__(256) k_tau_init26(float* tau, int rx, int ry, int rz, unsigned long long N, float tau0)
{   // out-of-bounds slots start at 0 (:396), in-bounds at tau0 (:401)
    const unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= N * kK26) return;
    const unsigned long long id = idx / kK26;
    const int s = (int)(idx % kK26);
    const unsigned long long rxy = (unsigned long long)rx * ry;
    const int z = (int)(id / rxy), y = (int)((id % rxy) / rx), x = (int)(id % rx);
    int dx, dy, dz;
    slot26(s, dx, dy, dz);
    const int nx = x + dx, ny = y + dy, nz = z + dz;
    const bool inb = nx >= 0 && nx < rx && ny >= 0 && ny < ry && nz >= 0 && nz < rz;
    tau[idx] = inb ? tau0 : 0.0f;
}

// selectNext :137, :151-154 with a general vector_b (up to three non-zero components): the reference's expressions,
// left to right, no contraction: norm = sqrt((x*x + y*y) + z*z) (model_grid_map.hpp:51-54), dot = (ax*bx + ay*by) + az*bz.
// c*: coordinates of the node, g*: of the goal, n*: of the neighbour.  k_heuristic26 tabulates it, k_walk_batch26 (batch26.cuh)
// evaluates it per step: one function, so the two cannot drift apart.
__device__ __forceinline__ float heur26(float cx, float cy, float cz, float gx, float gy, float gz, float nx, float ny, float nz, float beta)
{
    const float ax = __fsub_rn(gx, cx), ay = __fsub_rn(gy, cy), az = __fsub_rn(gz, cz);
    const float bx = __fsub_rn(nx, cx), by = __fsub_rn(ny, cy), bz = __fsub_rn(nz, cz);
    const float na = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(ax, ax), __fmul_rn(ay, ay)), __fmul_rn(az, az)));
    const float nb = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(bx, bx), __fmul_rn(by, by)), __fmul_rn(bz, bz)));
    const float dot = __fadd_rn(__fadd_rn(__fmul_rn(ax, bx), __fmul_rn(ay, by)), __fmul_rn(az, bz));
    const float cosv = __fdiv_rn(dot, __fmul_rn(na, nb));
    return __fadd_rn(1.0f, __fmul_rn(beta, cosv));
}

__global__ void __launch_bounds__(256) k_heuristic26(float* __restrict__ heur, const float* __restrict__ coords, const uint32_t* __restrict__ occ_bits,
                                                      int rx, int ry, int rz, unsigned long long N, int goal, float beta)
{
    const unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= N * kK26) return;
    const unsigned long long id = idx / kK26;
    const int s = (int)(idx % kK26);
    const float* xs = coords;
    const float* ys = xs + rx;
    const float* zs = ys + ry;
    const unsigned long long rxy = (unsigned long long)rx * ry;
    const int z = (int)(id / rxy), y = (int)((id % rxy) / rx), x = (int)(id % rx);
    const int gz = (int)(goal / rxy), gy = (int)((goal % rxy) / rx), gx = (int)(goal % rx);
    int dx, dy, dz;
    slot26(s, dx, dy, dz);
    const int nx = x + dx, ny = y + dy, nz = z + dz;
    const bool inb = nx >= 0 && nx < rx && ny >= 0 && ny < ry && nz >= 0 && nz < rz;
    float v = kClosedSlot;
    if (inb) {
        const unsigned long long nid = ((unsigned long long)nz * ry + ny) * rx + nx;
        if (!((occ_bits[nid >> 5] >> (nid & 31)) & 1u)) v = heur26(xs[x], ys[y], zs[z], xs[gx], ys[gy], zs[gz], xs[nx], ys[ny], zs[nz], beta);
    }
    heur[idx] = v;
}

// ------------------------------------------------------------------------------------------
// K2 for K = 26: one ant per warp, persistent warps pulling ants from the device queue.  Everything in a step is
// warp-uniform (one ant), so there is no predication on liveness: an ant that arrives, dies or parks leaves the loop.
// Visited set: the same open-addressed hash of 4x4x4-node tiles (u32 key + u64 mask per entry) in shared
// memory, one table per warp; an ant that fills it to 3/4 moves the set to its table in HBM, parks {node, steps, tiles,
// L} and is resumed by pass 2 (GLOBAL) — exact, its draws are a pure function of (iteration, ant, step).
// ------------------------------------------------------------------------------------------
template <bool GLOBAL>
__global__ void __launch_bounds__(kWalk26Threads) k_walk26(WalkArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int w = threadIdx.x >> 5;
    const int E = 1 << a.table_log2;
    const int hshift = 32 - a.table_log2;

    unsigned long long* masks;
    uint32_t* keys;
    if (GLOBAL) {
        keys = a.gkeys; masks = a.gmasks;   // re-pointed per ant below
    } else {
        unsigned long long* mbase = reinterpret_cast<unsigned long long*>(smem_raw);
        masks = mbase + (size_t)w * E;
        keys = reinterpret_cast<uint32_t*>(mbase + (size_t)kWalk26Ants * E) + (size_t)w * E;
    }

    const int rx = a.rx, ry = a.ry;
    const int rxy = rx * ry;
    const int TX = (rx + 3) >> 2, TY = (ry + 3) >> 2;
    const bool active = lane < kK26;
    const int kk = active ? lane : kK26 - 1;             // idle lanes re-read slot 25 (same sector)
    int dxk, dyk, dzk;
    slot26(kk, dxk, dyk, dzk);
    const int stride_k = dxk + dyk * rx + dzk * rxy;
    const int type_k = (dxk != 0) + (dyk != 0) + (dzk != 0);
    // per-slot step length, initFromGridMap :375-385 with the commented-out lengths enabled
    const float dist_k = type_k == 1 ? a.precision : (type_k == 2 ? __fmul_rn(a.precision, 1.414f) : __fmul_rn(a.precision, 1.732f));

    const int sz = a.start / rxy, sy = (a.start % rxy) / rx, sx = a.start % rx;
    const bool alpha1 = a.alpha == 1;

    IterState* st = a.st;
    const int colony = st->colony;
    const uint32_t iter = (uint32_t)st->iter;
    const float base_now = st->base;
    int local_n = min(max(colony - a.shard_first, 0), a.shard_chunk);
    if (GLOBAL) local_n = (int)st->overflow_n;
    const int limit = (E >> 2) * 3;

    unsigned long long c_steps = 0, c_ants = 0, c_arrived = 0, c_nocand = 0, c_fall = 0, c_cap = 0, c_over = 0;

    while (true) {
        unsigned q = 0;
        if (lane == 0) q = atomicAdd(GLOBAL ? &st->queue2 : &st->queue, 1u);
        q = __shfl_sync(FULL, q, 0);
        if (q >= (unsigned)local_n) break;
        const int ant_local = GLOBAL ? (int)a.overflow_list[q] : (int)q;
        const uint32_t ant_global = (uint32_t)(a.shard_first + ant_local);

        int cur = a.start, x = sx, y = sy, z = sz, steps = 0, ntiles = 1;
        float L = 0.0f;                                   // addStartNode :81-86
        uint32_t rw0 = 0, rw1 = 0, rw2 = 0, rw3 = 0;
        if (GLOBAL) {   // resume a parked ant: its visited set already lives in HBM table q
            keys = a.gkeys + (size_t)q * E;
            masks = a.gmasks + (size_t)q * E;
            const int4 r = a.resume[q];
            cur = r.x; steps = r.y; ntiles = r.z; L = __int_as_float(r.w);
            z = cur / rxy; y = (cur % rxy) / rx; x = cur % rx;
            philox4(iter, ant_global, ((uint32_t)steps >> 2) | a.block_hi, a.stream_word, a.seed_lo, a.seed_hi, rw0, rw1, rw2, rw3);
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

        int result = -1;   // >= 0: steps of an ant that arrived, -1: dead, -2: parked (table overflow -> pass 2)
        int reason = 0;    // 1 no candidate, 2 roulette fall-through, 3 step cap
        uint32_t* pid = a.path_ids + (size_t)ant_local * a.cap;
        uint8_t* pdir = a.path_dirs + (size_t)ant_local * a.cap;

        while (true) {
            if (steps >= a.cap) { reason = 3; break; }   // step cap (a deviation the oracle mirrors)
            const float tau_k = tau_or_base(__ldg(a.tau + (size_t)cur * kK26 + kk), base_now);
            const float heur_k = __ldg(a.heur + (size_t)cur * kK26 + kk);
            if ((steps & 3) == 0) philox4(iter, ant_global, ((uint32_t)steps >> 2) | a.block_hi, a.stream_word, a.seed_lo, a.seed_hi, rw0, rw1, rw2, rw3);
            const uint32_t rsel = (steps & 2) ? ((steps & 1) ? rw3 : rw2) : ((steps & 1) ? rw1 : rw0);
            const float u = __fmul_rn(__int2float_rn((int)(rsel >> 1)), 4.656612873077392578125e-10f);   // (float)rand()/(float)RAND_MAX :169
            // ---- neighbour of this lane: open (in bounds and free, folded into the table), tabu probe ----
            const int nx = x + dxk, ny = y + dyk, nz = z + dzk;
            const bool open_k = active && heur_k != kClosedSlot;   // NaN (duplicate plane) stays open, as in the reference
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
            if (cur == a.goal) { result = steps; break; }       // :182-186
            if (!GLOBAL && newtile && ntiles > limit) {          // rare: shared-memory table 3/4 full -> park for pass 2
                int o = 0;
                if (lane == 0) o = (int)atomicAdd(&st->overflow_n, 1u);
                o = __shfl_sync(FULL, o, 0);
                const int Eg = 1 << a.gtable_log2, gsh = 32 - a.gtable_log2;
                uint32_t* nkeys = a.gkeys + (size_t)o * Eg;
                unsigned long long* nmasks = a.gmasks + (size_t)o * Eg;
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
                    a.overflow_list[o] = (uint32_t)ant_local;
                    a.ant_steps[ant_local] = -2;
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
                a.ant_steps[ant_local] = result;
                a.ant_L[ant_local] = result >= 0 ? L : INFINITY;   // setDeadEnd :88-91
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


// ------------------------------------------------------------------------------------------
// K2 for K = 26, pass 1, second generation (round 2): the step of k_walk26 with the instruction stream cut from ~340 to ~170
// per step, by the means that worked for K = 6 (walk3.cuh) plus two that are specific to 26 slots:
//   * the 26 scores are exchanged through 128 bytes of shared memory (one store, seven broadcast LDS.128) instead of 26 shuffles;
//   * both roulette chains (ascending `total`, descending `prob_sum`) are computed once, the 26 suffix sums go back through shared
//     memory and every lane reads its own — instead of 26 compare-and-select pairs per lane;
//   * packed coordinates z<<20 | y<<10 | x (one add per move, tile key = one AND, bit index = one multiply);
//   * the move (node stride, packed delta, step length) is one LDS.128 from a 26-entry table instead of five shuffles;
//   * Philox for steps T+4..T+7 in four slices beside steps T..T+3; the trail in registers, 32 steps per coalesced store.
// Grids with an axis above 1024 nodes keep k_walk26<false>; parked ants are resumed by k_walk26<true> either way (the visited set
// is re-keyed to its tile indices when it moves to HBM).
// ------------------------------------------------------------------------------------------
constexpr uint32_t kLow26 = 0x00300C03u;                       // x, y, z bits 0-1: position inside a 4x4x4 tile
constexpr uint32_t kKey26 = 0x3FFFFFFFu & ~kLow26;
constexpr uint32_t kMul26 = 0x00101010u;                       // gathers the six position bits at 20..25
constexpr int kWalk26pExtra = 512 + kWalk26Ants * 256;         // move table + per-warp exchange rows in front of the visited tables

__global__ void __launch_bounds__(kWalk26Threads) k_walk26p(WalkArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int w = threadIdx.x >> 5;
    const int E = 1 << a.table_log2;
    const int hshift = 32 - a.table_log2;
    int4* lut = reinterpret_cast<int4*>(smem_raw);                                     // [26] {node stride, packed delta, bits of the step length, -}
    float* xch = reinterpret_cast<float*>(smem_raw + 512) + w * 64;                     // [0, 32): scores, [32, 64): suffix sums
    unsigned long long* mbase = reinterpret_cast<unsigned long long*>(smem_raw + kWalk26pExtra);
    unsigned long long* masks = mbase + (size_t)w * E;
    uint32_t* keys = reinterpret_cast<uint32_t*>(mbase + (size_t)kWalk26Ants * E) + (size_t)w * E;

    const int rx = a.rx, ry = a.ry;
    const int rxy = rx * ry;
    const int TX = (rx + 3) >> 2, TY = (ry + 3) >> 2;
    if (threadIdx.x < kK26) {
        int dx, dy, dz;
        slot26(threadIdx.x, dx, dy, dz);
        const int type = (dx != 0) + (dy != 0) + (dz != 0);
        // per-slot step length, initFromGridMap :375-385 with the commented-out lengths enabled
        const float dist = type == 1 ? a.precision : (type == 2 ? __fmul_rn(a.precision, 1.414f) : __fmul_rn(a.precision, 1.732f));
        lut[threadIdx.x] = make_int4(dx + dy * rx + dz * rxy, dx + dy * 1024 + dz * 1048576, __float_as_int(dist), 0);
    }
    __syncthreads();

    const bool active = lane < kK26;
    const int kk = active ? lane : kK26 - 1;             // idle lanes re-read slot 25 (same sector)
    int dxk, dyk, dzk;
    slot26(kk, dxk, dyk, dzk);
    const uint32_t dPk = (uint32_t)(dxk + dyk * 1024 + dzk * 1048576);
    const float* tau_k = a.tau + kk;
    const float* heur_k = a.heur + kk;
    const bool alpha1 = a.alpha == 1;

    IterState* st = a.st;
    const int colony = st->colony;
    const uint32_t iter = (uint32_t)st->iter;
    const float base_now = st->base;
    const int local_n = min(max(colony - a.shard_first, 0), a.shard_chunk);
    const int limit = (E >> 2) * 3;
    const int cap = a.cap, goal = a.goal;
    const uint32_t Pstart = pack_xyz(a.start % rx, (a.start % rxy) / rx, a.start / rxy);

    unsigned long long c_steps = 0, c_ants = 0, c_arrived = 0, c_nocand = 0, c_fall = 0, c_cap = 0, c_over = 0;

    while (true) {
        unsigned q = 0;
        if (lane == 0) q = atomicAdd(&st->queue, 1u);
        q = __shfl_sync(FULL, q, 0);
        if (q >= (unsigned)local_n) break;
        const int ant_local = (int)q;
        const uint32_t ant_global = (uint32_t)(a.shard_first + ant_local);

        for (int i = lane; i < E; i += 32) keys[i] = kEmptyKey;
        __syncwarp();
        if (lane == 0) {   // addStartNode :81-86
            const uint32_t key = Pstart & kKey26;
            const unsigned bit = (((Pstart & kLow26) * kMul26) >> 20) & 63u;
            const unsigned slot = (key * 2654435761u) >> hshift;
            keys[slot] = key; masks[slot] = 1ull << bit;
        }
        __syncwarp();

        int cur = a.start, steps = 0, ntiles = 1;
        uint32_t P = Pstart;
        float L = 0.0f;
        int result = -1;   // >= 0: steps of an ant that arrived, -1: dead, -2: parked (table overflow -> pass 2)
        int reason = 0;    // 1 no candidate, 2 roulette fall-through, 3 step cap
        uint32_t rec_id = 0, rec_dir = 0;
        uint32_t* pid = a.path_ids + (size_t)ant_local * cap;
        uint8_t* pdir = a.path_dirs + (size_t)ant_local * cap;

        float u0, u1, u2, u3;
        {
            uint32_t w0, w1, w2, w3;
            philox4(iter, ant_global, a.block_hi, a.stream_word, a.seed_lo, a.seed_hi, w0, w1, w2, w3);
            u0 = __fmul_rn(__int2float_rn((int)(w0 >> 1)), 4.656612873077392578125e-10f);   // (float)rand()/(float)RAND_MAX :169
            u1 = __fmul_rn(__int2float_rn((int)(w1 >> 1)), 4.656612873077392578125e-10f);
            u2 = __fmul_rn(__int2float_rn((int)(w2 >> 1)), 4.656612873077392578125e-10f);
            u3 = __fmul_rn(__int2float_rn((int)(w3 >> 1)), 4.656612873077392578125e-10f);
        }
        uint32_t pc0 = 0, pc1 = 0, pc2 = 0, pc3 = 0;

        float tau_v = __ldg(tau_k + (size_t)cur * kK26);
        float heur_v = __ldg(heur_k + (size_t)cur * kK26);

        // one step with the draw u; returns true when the ant is finished (arrived, dead, capped or parked)
        auto step = [&](const float u) -> bool {
            if (steps >= cap) { reason = 3; return true; }   // step cap (a deviation the oracle mirrors)
            // ---- neighbour of this lane: open (in bounds and free, folded into the table), tabu probe ----
            const uint32_t Pk = P + dPk;
            const uint32_t key = Pk & kKey26;
            const unsigned bit = (((Pk & kLow26) * kMul26) >> 20) & 63u;
            const bool open_k = active && heur_v != kClosedSlot;   // NaN (duplicate plane) stays open, as in the reference
            unsigned slot = (key * 2654435761u) >> hshift;
            uint32_t kf = keys[slot];
            unsigned long long mm = masks[slot];
            while (open_k && kf != key && kf != kEmptyKey) {
                slot = (slot + 1) & (E - 1);
                kf = keys[slot]; mm = masks[slot];
            }
            const bool found = kf == key;
            const bool cand = open_k && !(found && ((mm >> bit) & 1ull));
            const float tau_now = tau_or_base(tau_v, base_now);
            const float tpow = alpha1 ? tau_now : pow_int(tau_now, a.alpha);
            const float info = cand ? __fmul_rn(tpow, heur_v) : 0.0f;   // :154; +0 is the identity of both chains below
            const unsigned cb = __ballot_sync(FULL, cand);
            // ---- roulette in the reference's order (:155 ascending total, :172-181 descending prob_sum) ----
            xch[lane] = info;
            __syncwarp();
            float v[28];
#pragma unroll
            for (int i = 0; i < 7; i++) {
                const float4 t = reinterpret_cast<const float4*>(xch)[i];
                v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
            }
            float total = 0.0f;
#pragma unroll
            for (int i = 0; i < kK26; i++) total = __fadd_rn(total, v[i]);
            const float rnd = __fmul_rn(u, total);
            float run[28];
            run[27] = 0.0f; run[26] = 0.0f;
            float acc = 0.0f;
#pragma unroll
            for (int i = kK26 - 1; i >= 0; i--) { acc = __fadd_rn(acc, v[i]); run[i] = acc; }
#pragma unroll
            for (int i = 0; i < 7; i++) reinterpret_cast<float4*>(xch + 32)[i] = make_float4(run[4 * i], run[4 * i + 1], run[4 * i + 2], run[4 * i + 3]);   // every lane holds the same 26 sums
            __syncwarp();
            const float mine = xch[32 + kk];
            const bool pick = cand && (mine >= rnd);
            const unsigned pb = __ballot_sync(FULL, pick);
            if (pb == 0) { reason = cb == 0 ? 1 : 2; return true; }   // :162-166 / fall-through :191-192 (NaN, rounding)
            const int c = 31 - __clz((int)pb);                        // first hit scanning 25 -> 0
            const int4 mv = lut[c];
            // ---- addNextNode (:73-79): lane (steps & 31) keeps the trail entry; 32 of them go out as one coalesced store ----
            if (lane == (steps & 31)) { rec_id = (uint32_t)cur; rec_dir = (uint32_t)c; }
            if (lane == c) { keys[slot] = key; masks[slot] = found ? (mm | (1ull << bit)) : (1ull << bit); }
            const unsigned fb = __ballot_sync(FULL, found);
            const int newtile = (int)(((fb >> c) & 1u) ^ 1u);
            cur += mv.x;
            P += (uint32_t)mv.y;
            tau_v = __ldg(tau_k + (size_t)cur * kK26);
            heur_v = __ldg(heur_k + (size_t)cur * kK26);
            L = __fadd_rn(L, __int_as_float(mv.z));   // :78
            steps++;
            ntiles += newtile;
            if ((steps & 31) == 0) { pid[steps - 32 + lane] = rec_id; pdir[steps - 32 + lane] = (uint8_t)rec_dir; }
            __syncwarp();
            if (cur == goal) { result = steps; return true; }       // :182-186
            if (newtile && ntiles > limit) { result = -2; return true; }   // shared-memory table 3/4 full -> park for pass 2
            return false;
        };

        for (uint32_t T = 0;; T += 4u) {
            pc0 = iter; pc1 = ant_global; pc2 = ((T >> 2) + 1u) | a.block_hi; pc3 = a.stream_word;
            if (step(u0)) break;
            philox_rounds<0, 3>(pc0, pc1, pc2, pc3, a.seed_lo, a.seed_hi);
            if (step(u1)) break;
            philox_rounds<3, 6>(pc0, pc1, pc2, pc3, a.seed_lo, a.seed_hi);
            if (step(u2)) break;
            philox_rounds<6, 9>(pc0, pc1, pc2, pc3, a.seed_lo, a.seed_hi);
            if (step(u3)) break;
            philox_rounds<9, 10>(pc0, pc1, pc2, pc3, a.seed_lo, a.seed_hi);
            u0 = __fmul_rn(__int2float_rn((int)(pc0 >> 1)), 4.656612873077392578125e-10f);
            u1 = __fmul_rn(__int2float_rn((int)(pc1 >> 1)), 4.656612873077392578125e-10f);
            u2 = __fmul_rn(__int2float_rn((int)(pc2 >> 1)), 4.656612873077392578125e-10f);
            u3 = __fmul_rn(__int2float_rn((int)(pc3 >> 1)), 4.656612873077392578125e-10f);
        }
        if (lane < (steps & 31)) { pid[(steps & ~31) + lane] = rec_id; pdir[(steps & ~31) + lane] = (uint8_t)rec_dir; }   // the last, partial block of the trail
        __syncwarp();
        if (result == -2) {   // rare: move the visited set to the ant's HBM table, re-keyed to tile indices (what pass 2 probes with)
            int o = 0;
            if (lane == 0) o = (int)atomicAdd(&st->overflow_n, 1u);
            o = __shfl_sync(FULL, o, 0);
            const int Eg = 1 << a.gtable_log2, gsh = 32 - a.gtable_log2;
            uint32_t* nkeys = a.gkeys + (size_t)o * Eg;
            unsigned long long* nmasks = a.gmasks + (size_t)o * Eg;
            for (int i = lane; i < Eg; i += 32) nkeys[i] = kEmptyKey;
            __syncwarp();
            for (int i = lane; i < E; i += 32) {
                const uint32_t pk = keys[i];
                if (pk == kEmptyKey) continue;
                const uint32_t t = (uint32_t)((((pk >> 22) & 255u) * TY + ((pk >> 12) & 255u)) * TX + ((pk >> 2) & 255u));
                unsigned sl = (t * 2654435761u) >> gsh;
                while (atomicCAS(&nkeys[sl], kEmptyKey, t) != kEmptyKey) sl = (sl + 1) & (Eg - 1);
                nmasks[sl] = masks[i];
            }
            if (lane == 0) {
                a.resume[o] = make_int4(cur, steps, ntiles, __float_as_int(L));
                a.overflow_list[o] = (uint32_t)ant_local;
                a.ant_steps[ant_local] = -2;
            }
            c_over++;   // its steps are counted by pass 2
        } else {
            if (lane == 0) {
                a.ant_steps[ant_local] = result;
                a.ant_L[ant_local] = result >= 0 ? L : INFINITY;   // setDeadEnd :88-91
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
