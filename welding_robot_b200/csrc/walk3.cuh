// K2, pass 1: the ant-construction step described in walk2.cuh (selectNext ACSRank_3D.hpp:134-193 + the ant loop :252-265) with
// everything that is not the roulette itself taken off the warp's dependent instruction chain.
//
// What the mid-round-2 capture of the previous pass-1 kernel showed (profiles/r2_walk2_ncu.md): 1.7 warps per scheduler, 27 % of the issue slots, 6.3
// cycles per issued instruction — the kernel's time is (longest ant's steps) x (latency of ONE warp's instruction chain), every
// instruction of a step costs its full dependent latency, and nothing else on the scheduler hides it.  So this kernel removes
// instructions and branches from the step, and moves work that has no consumer inside the step to where a stall would be:
//   * in pass 1 every live ant of the warp is at the SAME step index T (they all start at 0 and a finished ant idles), so the
//     step counter, the step-cap test and the choice of the uniform draw are warp-uniform / compile-time (four steps per trip);
//   * Philox is software-pipelined: the block of draws for steps T+4..T+7 is computed in four slices spread over steps T..T+3
//     (straight-line code next to the gather latency) instead of a 72-instruction burst in front of every fourth step;
//   * the trail (addNextNode :73-79) is not stored by the winning lane per step (two scattered stores + 64-bit address
//     arithmetic inside a divergent branch): every lane of the group knows the node left and the slot taken, lane (T & 7) keeps
//     them in two registers and the group writes eight steps at once, coalesced, every second trip;
//   * the visited insert is a predicated store by the lane whose pick is the highest (known from the ballot, before the
//     move table answers); the tile count lives in a register fed by one vote — no winner branch, no shared-memory counter,
//     no flag word to poll;
//   * outcome bookkeeping (arrived / died why / capped) is reconstructed after the loop from (cur, steps, last candidate mask).
//   * PREFETCH = 0 (the colony has converged: chosen by the same device feedback that selects the rank-set deposits): the
//     gathers are PREDICTED.  The ncu capture of the first k_walk3 showed 46 % of the stall samples on the four instructions
//     that wait for tau[cur] / heur[cur]: the ~28 ants of an SM advance in lockstep along the same path, whose rows (735 x 2
//     lines of 128 B) do not fit L1, so every step somebody pays an L2 round trip.  But where a converged ant will stand at
//     step t is known: node t of the best path so far.  Every trip loads the next four best-path node ids (one broadcast
//     LDG.128) and this lane's tau / heur values of those nodes, a whole trip before they are needed; after a move the lane
//     compares the node it reached with the predicted one and takes the values from registers, or — a deviating ant —
//     issues the ordinary loads.  The values come from the same addresses either way, so every ant is bit-identical.
//   * PREFETCH = 1 (the colony still wanders): the six neighbours' rows are prefetched a step ahead, and a visited-table look-up
//     fetches four entries at once (no probe loop: most look-ups there are of tiles that are not present yet).
// Ants whose table fills up move their visited set to a table in HBM, park {node, steps} and are resumed by k_walk2 (pass 2).
#pragma once
#include "walk2.cuh"

namespace wr {

template <int V> struct IC { static constexpr int value = V; };

// rounds [R0, R1) of Philox4x32-10 on a block in flight (wr_common.cuh philox4, cut into slices)
template <int R0, int R1>
__device__ __forceinline__ void philox_rounds(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3, uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = R0; r < R1; r++) {
        const uint32_t hi0 = __umulhi(kPhiloxM0, c0), lo0 = kPhiloxM0 * c0;
        const uint32_t hi1 = __umulhi(kPhiloxM1, c2), lo1 = kPhiloxM1 * c2;
        const uint32_t n0 = hi1 ^ c1 ^ (k0 + (uint32_t)r * kPhiloxW0), n2 = hi0 ^ c3 ^ (k1 + (uint32_t)r * kPhiloxW1);
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    }
}

// The roulette arithmetic of one step, shared with k_path_thresholds (path_verify.cuh), which must reproduce it bit for bit.
// Score of a slot (:151-154): tau^alpha * (1 + beta*cos), 0 for a slot that is no candidate.
template <bool ALPHA1>
__device__ __forceinline__ float slot_score(bool cand, float tau_v, float heur_v, float base, int alpha)
{
    const float tau_now = tau_or_base(tau_v, base);
    const float tpow = ALPHA1 ? tau_now : pow_int(tau_now, alpha);
    return cand ? __fmul_rn(tpow, heur_v) : 0.0f;
}
// the roulette total (:155) and the suffix sum v5 + ... + v_k that slot k compares with the draw (:172-181); m_j = k <= j ? ~0 : 0
__device__ __forceinline__ float roulette_total(float v0, float v1, float v2, float v3, float v4, float v5)
{
    return __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(0.0f, v0), v1), v2), v3), v4), v5);
}
__device__ __forceinline__ float roulette_suffix(float v0, float v1, float v2, float v3, float v4, float v5, uint32_t m4, uint32_t m3, uint32_t m2,
                                                 uint32_t m1, uint32_t m0)
{
    float mine = __fadd_rn(0.0f, v5);
    mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v4) & m4));
    mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v3) & m3));
    mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v2) & m2));
    mine = __fadd_rn(mine, __uint_as_float(__float_as_uint(v1) & m1));
    return __fadd_rn(mine, __uint_as_float(__float_as_uint(v0) & m0));
}

template <bool ALPHA1, int PREFETCH>
__global__ void __launch_bounds__(kWalkThreads, 2) k_walk3(WalkArgs a)   // two CTAs per SM (shared memory); no register squeeze
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // [0, 1024): move table indexed by the 6-bit pick ballot (see k_walk2); [1024, 1152): unused here; [1152, ...): tables [16][E]
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
    constexpr bool PREDICT = PREFETCH == 0;   // 0: converged colony, predicted gathers; 1: wandering colony, neighbour rows prefetched
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
    asm volatile("" : "+r"(lut_sa), "+r"(tab.sa), "+r"(gmask));   // opaque: no re-derivation of the shared window base inside the loop

    const int rx = a.rx, rxy = a.rx * a.ry;
    const int dxk = (k == 3) - (k == 2), dyk = (k == 4) - (k == 1), dzk = (k == 5) - (k == 0);
    const uint32_t dPk = (uint32_t)(dxk + dyk * 1024 + dzk * 1048576);
    // the two idle lanes of a group re-read slot 5 (same sector) and are never alive (cap_k = 0), so their values are never candidates
    const int kk6 = k < 6 ? k : 5;
    const float* tau_k = a.tau + kk6;
    const float* heur_k = a.heur + kk6;
    const long long stride_k = (long long)(dxk + dyk * rx + dzk * rxy);
    const long long last_node = (long long)rxy * a.rz - 1;
    uint32_t m4 = k <= 4 ? ~0u : 0u, m3 = k <= 3 ? ~0u : 0u, m2 = k <= 2 ? ~0u : 0u, m1 = k <= 1 ? ~0u : 0u, m0 = k <= 0 ? ~0u : 0u;
    asm volatile("" : "+r"(m4), "+r"(m3), "+r"(m2), "+r"(m1), "+r"(m0));

    // the packed position carries the key tag in bit 31 (in-bounds moves never borrow out of the z field), so a tile key is one AND
    const uint32_t Pstart = pack_xyz(a.start % rx, (a.start % rxy) / rx, a.start / rxy) | kKeyTag;
    constexpr uint32_t kKeyMask = kPackKey | kKeyTag;

    IterState* st = a.st;
    const int colony = st->colony;
    const uint32_t iter = (uint32_t)st->iter;
    const float base_now = st->base;
    const int local_n = min(max(colony - a.shard_first, 0), a.shard_chunk);
    const uint32_t limit = (uint32_t)((E >> 2) * 3);
    const int cap = a.cap, goal = a.goal;
    int cap_k = k < 6 ? cap : 0;
    uint32_t lut_rot = (uint32_t)(gbase - 4) & 31u;   // rotating the ballot right by this puts the group's six bits at 4..9: the byte offset into the move table
    asm volatile("" : "+r"(cap_k), "+r"(lut_rot));

    unsigned long long c_steps = 0, c_ants = 0, c_arrived = 0, c_nocand = 0, c_fall = 0, c_cap = 0, c_over = 0;
    uint32_t c_vants = 0, c_vsteps = 0;    // ants completed by verification, steps not walked here because they were verified
    const int vfull = (PREDICT && a.verify_dev) ? a.verify_n->y : -1;   // best_n - 1 when the whole best path verified, else -1

    while (true) {
        unsigned q0 = 0;
        if (lane == 0) q0 = atomicAdd(&st->queue, 4u);
        q0 = __shfl_sync(FULL, q0, 0);
        if (q0 >= (unsigned)local_n) break;                                    // warp-uniform
        const unsigned q = q0 + (unsigned)(lane >> 3);
        const bool has = q < (unsigned)local_n;
        const int ant_local = has ? (int)q : 0;
        const uint32_t ant_global = (uint32_t)(a.shard_first + ant_local);

        // Converged colony with the path verified (k_path_verify): every ant of the warp has followed the best path for at least
        // T steps, a multiple of 8, so it stands on best[T] with visited set best[0..T], like any other such ant.  The warp
        // resumes there; if all its ants followed the whole path, it only does their bookkeeping.
        uint32_t T = 0;                    // step index of every live ant of the warp
        bool done = false;
        if (PREDICT && a.verify_dev) {
            const int dv = has ? a.verify_dev[ant_local] : INT_MAX;
            const bool complete = has && dv == vfull;
            T = __reduce_min_sync(FULL, (uint32_t)(complete ? vfull : dv) & ~7u);
            done = __all_sync(FULL, !has || complete);
            if (done) { c_vants += has ? 1u : 0u; c_vsteps += has ? (uint32_t)vfull : 0u; }
            else c_vsteps += has ? T : 0u;
        }
        uint32_t ntiles = 1u;
        if (!done) {
            for (int i = k; i < E; i += kGroup) tab.store(i, 0ull);
            __syncwarp();
            if (T == 0) {
                if (k == 0) {   // addStartNode :81-86
                    const uint32_t key = Pstart & kKeyMask;
                    const uint32_t bit = (((Pstart & kPackLow) * kPackMul) >> 20) & 31u;
                    tab.store(tile_hash(key, (uint32_t)E - 3u), ((unsigned long long)key << 32) | (unsigned long long)(1u << bit));
                }
            } else {   // the tiles of best[0..T], the group's lanes in parallel; linear probing gives the same look-ups in any insertion order
                unsigned* tw = reinterpret_cast<unsigned*>(tab_s + (size_t)g * E);   // entry i: mask word 2i, key word 2i + 1
                uint32_t claims = 0;
                for (uint32_t p = (uint32_t)k; p <= T; p += kGroup) {
                    const int node = (int)a.best_ids[p];
                    const uint32_t Pn = pack_xyz(node % rx, (node % rxy) / rx, node / rxy) | kKeyTag;
                    const uint32_t key = Pn & kKeyMask;
                    const uint32_t bit = (((Pn & kPackLow) * kPackMul) >> 20) & 31u;
                    unsigned slot = tile_hash(key, (uint32_t)E - 3u);
                    while (true) {
                        const unsigned old = atomicCAS(tw + 2 * slot + 1, 0u, key);
                        if (old == 0u || old == key) { atomicOr(tw + 2 * slot, 1u << bit); claims += old == 0u ? 1u : 0u; break; }
                        slot = slot + 1 < (unsigned)E ? slot + 1 : 0u;
                    }
                }
                __syncwarp();
                claims += __shfl_xor_sync(FULL, claims, 4);
                claims += __shfl_xor_sync(FULL, claims, 2);
                claims += __shfl_xor_sync(FULL, claims, 1);
                ntiles = claims;
            }
            __syncwarp();
        }

        int cur = done ? goal : (T ? (int)a.best_ids[T] : a.start), steps = done ? vfull : (int)T;
        uint32_t P = T ? pack_xyz(cur % rx, (cur % rxy) / rx, cur / rxy) | kKeyTag : Pstart;
        uint32_t lastcb = 1u;              // candidate mask of the last step the ant was alive in (why a dead ant died)
        bool parked = false;
        bool live = has && cap_k > 0 && !done;
        uint32_t kt = (uint32_t)k;         // (k - T) & 7: the lane that keeps step T + j of the trail is the one with kt == j (T % 8 == 0)
        uint32_t rec_id = 0, rec_dir = 0;
        uint32_t* pid = a.path_ids + (size_t)ant_local * cap;
        uint8_t* pdir = a.path_dirs + (size_t)ant_local * cap;

        // draws of steps T..T+3; the next block is produced inside the loop, one slice per step
        float u0, u1, u2, u3;
        {
            uint32_t w0, w1, w2, w3;
            philox4(iter, ant_global, (T >> 2) | a.block_hi, a.stream_word, a.seed_lo, a.seed_hi, w0, w1, w2, w3);
            // (float)rand()/(float)RAND_MAX (:169): (float)RAND_MAX is 2^31, so the division is an exact scaling
            u0 = __fmul_rn(__int2float_rn((int)(w0 >> 1)), 4.656612873077392578125e-10f);
            u1 = __fmul_rn(__int2float_rn((int)(w1 >> 1)), 4.656612873077392578125e-10f);
            u2 = __fmul_rn(__int2float_rn((int)(w2 >> 1)), 4.656612873077392578125e-10f);
            u3 = __fmul_rn(__int2float_rn((int)(w3 >> 1)), 4.656612873077392578125e-10f);
        }
        uint32_t pc0 = 0, pc1 = 0, pc2 = 0, pc3 = 0;
        auto rounds = [&](auto r0, auto r1) { philox_rounds<decltype(r0)::value, decltype(r1)::value>(pc0, pc1, pc2, pc3, a.seed_lo, a.seed_hi); };

        float tau_v = __ldg(tau_k + (size_t)cur * 6);
        float heur_v = __ldg(heur_k + (size_t)cur * 6);

        // predicted rows (PREDICT): best-path positions T+1..T+3 (c*) and T+4..T+7 (n*), this lane's slot of each
        uint32_t c1 = 0, c2 = 0, c3 = 0, n0 = 0, n1 = 0, n2 = 0, n3 = 0;
        float ct1 = 0.f, ct2 = 0.f, ct3 = 0.f, ch1 = 0.f, ch2 = 0.f, ch3 = 0.f;
        float nt0 = 0.f, nt1 = 0.f, nt2 = 0.f, nt3 = 0.f, nh0 = 0.f, nh1 = 0.f, nh2 = 0.f, nh3 = 0.f;
        if (PREDICT) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(a.best_ids + T));
            c1 = q.y; c2 = q.z; c3 = q.w;
            ct1 = __ldg(tau_k + (size_t)c1 * 6); ch1 = __ldg(heur_k + (size_t)c1 * 6);
            ct2 = __ldg(tau_k + (size_t)c2 * 6); ch2 = __ldg(heur_k + (size_t)c2 * 6);
            ct3 = __ldg(tau_k + (size_t)c3 * 6); ch3 = __ldg(heur_k + (size_t)c3 * 6);
        }

        // one step at index T + J with the draw u; (pn, pt, ph) = predicted next node and this lane's values of its row
        auto step = [&](const uint32_t J, const float u, const uint32_t pn, const float pt_v, const float ph_v) {
            if (PREFETCH & 1) {
                // (Also measured and rejected, for both modes: one Philox evaluation per 32 steps by letting lane k of a group compute
                // block 8 w + k and shuffling the four draws of a trip out of lane (trip & 7) — 16 instructions per step fewer, yet the
                // walk got 3 % slower and C5 10 %: four more shuffles at the head of every trip, three uniform branches, +8 registers.)
                // Measured and rejected instead of this prefetch: (a) prediction AND prefetch together (slower than either alone in
                // its regime); (b) staging the six neighbours' rows in shared memory with cp.async and letting only the winning lane
                // wait for its own copies — the wait (DEPBAR on the warp's scoreboard) is per WARP, so every step waited for the
                // slowest of 144 copies: iteration 1 1.64 -> 1.94 ms.
                long long nb = (long long)cur + stride_k;
                nb = nb < 0 ? 0 : (nb > last_node ? last_node : nb);
                const float* pt = a.tau + nb * 6;
                const float* ph = a.heur + nb * 6;
                asm volatile("prefetch.global.L1 [%0];" ::"l"(pt));
                asm volatile("prefetch.global.L1 [%0];" ::"l"(ph));
            }
            // ---- neighbour k: open (folded into the heuristic table), tabu probe ---------------------------------------
            const uint32_t Pk = P + dPk;
            const uint32_t key = Pk & kKeyMask;
            const uint32_t bitm = 1u << ((((Pk & kPackLow) * kPackMul) >> 20) & 31u);
            const bool open_k = heur_v != kClosedSlot;
            // scans start in [0, E-4]: the first four entries of a scan need no wrap-around
            unsigned slot = tile_hash(key, (uint32_t)E - 3u);
            bool found;
            uint32_t emask;
            if (PREFETCH & 1) {
                // wandering colony: tables are half full and a step's lookups are mostly of tiles that are NOT there (scan to the first
                // empty entry), so the probe loop ran ~3 extra trips per warp-step (the longest of 24 scans), each a dependent
                // LDS + branch.  Here the first four entries of the scan are fetched at once and resolved with selects.
                unsigned long long e0, e1, e2, e3;
                const uint32_t sa = tab.sa + slot * 8u;
                asm volatile("ld.shared.b64 %0, [%4];\n\tld.shared.b64 %1, [%4+8];\n\tld.shared.b64 %2, [%4+16];\n\tld.shared.b64 %3, [%4+24];"
                             : "=l"(e0), "=l"(e1), "=l"(e2), "=l"(e3) : "r"(sa) : "memory");
                const uint32_t k0 = (uint32_t)(e0 >> 32), k1 = (uint32_t)(e1 >> 32), k2 = (uint32_t)(e2 >> 32), k3 = (uint32_t)(e3 >> 32);
                const bool h0 = k0 == key, h1 = k1 == key, h2 = k2 == key, h3 = k3 == key;   // an entry is never behind an empty one of its own scan
                const bool s0 = h0 || k0 == 0u, s1 = h1 || k1 == 0u, s2 = h2 || k2 == 0u, s3 = h3 || k3 == 0u;
                found = h0 || h1 || h2 || h3;
                emask = (h0 ? (uint32_t)e0 : 0u) | (h1 ? (uint32_t)e1 : 0u) | (h2 ? (uint32_t)e2 : 0u) | (h3 ? (uint32_t)e3 : 0u);
                slot += s0 ? 0u : (s1 ? 1u : (s2 ? 2u : 3u));
                if (open_k && !(s0 || s1 || s2 || s3)) {   // rare: keep scanning
                    unsigned long long e;
                    do {
                        slot = slot + 1 < (unsigned)E ? slot + 1 : 0u;
                        e = tab.load(slot);
                    } while ((uint32_t)(e >> 32) != key && (uint32_t)(e >> 32) != 0u);
                    found = (uint32_t)(e >> 32) == key;
                    emask = found ? (uint32_t)e : 0u;
                }
            } else {
                unsigned long long e = tab.load(slot);
                while (open_k && (uint32_t)(e >> 32) != key && (uint32_t)(e >> 32) != 0u) {   // collisions are rare once the colony has converged
                    slot = slot + 1 < (unsigned)E ? slot + 1 : 0u;
                    e = tab.load(slot);
                }
                found = (uint32_t)(e >> 32) == key;
                emask = found ? (uint32_t)e : 0u;
            }
            const bool cand = live && open_k && !(emask & bitm);
            // ---- info = tau^alpha * (1 + beta*cos)  (:151-154) ------------------------------------------------------
            const float info = slot_score<ALPHA1>(cand, tau_v, heur_v, base_now, a.alpha);
            // ---- roulette in the reference's order (:155, :172-181) ------------------------------------------------
            const unsigned cb = __ballot_sync(FULL, cand) & gmask;
            const float v0 = __shfl_sync(FULL, info, 0, 8), v1 = __shfl_sync(FULL, info, 1, 8), v2 = __shfl_sync(FULL, info, 2, 8);
            const float v3 = __shfl_sync(FULL, info, 3, 8), v4 = __shfl_sync(FULL, info, 4, 8), v5 = __shfl_sync(FULL, info, 5, 8);
            const float total = roulette_total(v0, v1, v2, v3, v4, v5);
            const float rnd = __fmul_rn(u, total);
            const float mine = roulette_suffix(v0, v1, v2, v3, v4, v5, m4, m3, m2, m1, m0);
            const bool pick = cand && (mine >= rnd);
            const unsigned pball = __ballot_sync(FULL, pick);
            // ---- the move: a dead or finished ant has no pick and the table's entry 0 moves nowhere --------------------
            int4 mv;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(mv.x), "=r"(mv.y), "=r"(mv.z), "=r"(mv.w) : "r"(lut_sa + (__funnelshift_r(pball, pball, lut_rot) & 0x3F0u)) : "memory");
            const unsigned pb = (pball >> gbase) & 0x3Fu;                        // the first hit scanning 5 -> 0 is its highest set bit
            const uint32_t prev = (uint32_t)cur;
            cur += mv.x;
            P += (uint32_t)mv.y;
            if (PREDICT) {
                tau_v = pt_v; heur_v = ph_v;
                if ((uint32_t)cur != pn) {   // off the best path (or a finished ant idling): the ordinary gathers
                    tau_v = __ldg(tau_k + (size_t)cur * 6);
                    heur_v = __ldg(heur_k + (size_t)cur * 6);
                }
            } else {
                tau_v = __ldg(tau_k + (size_t)cur * 6);
                heur_v = __ldg(heur_k + (size_t)cur * 6);
            }
            // ---- side effects, all predicated -------------------------------------------------------------------------
            const bool stepok = pb != 0u;                      // implies live (a candidate needs a live ant)
            const bool win = pick && (pb >> k) == 1u;          // this lane's pick is the highest one
            if (win) tab.store(slot, ((unsigned long long)key << 32) | (unsigned long long)(emask | bitm));   // tabu insert
            if (stepok && kt == J) { rec_id = prev; rec_dir = (uint32_t)mv.z; }                                   // addNextNode :73-79
            const bool full = ntiles > limit;                  // as of the previous step, like k_walk2's flag word
            const unsigned nt = __ballot_sync(FULL, win && !found) & gmask;
            ntiles += nt ? 1u : 0u;
            lastcb = live ? cb : lastcb;
            steps = stepok ? (int)(T + J + 1u) : steps;
            const bool go = stepok && cur != goal;             // not arrived (:182-186)
            parked = parked || (go && full);
            live = go && !full && (int)(T + J + 1u) < cap_k;
            __syncwarp();
        };

        while (__any_sync(FULL, live)) {
            pc0 = iter; pc1 = ant_global; pc2 = ((T >> 2) + 1u) | a.block_hi; pc3 = a.stream_word;
            if (PREDICT) {   // ids of best-path positions T+4..T+7 (the same 16 bytes for every lane); consumed after step 0
                const uint4 q = __ldg(reinterpret_cast<const uint4*>(a.best_ids + T + 4u));
                n0 = q.x; n1 = q.y; n2 = q.z; n3 = q.w;
            }
            step(0u, u0, c1, ct1, ch1); rounds(IC<0>{}, IC<3>{});
            if (PREDICT) {   // their rows: first needed by the last step of this trip
                nt0 = __ldg(tau_k + (size_t)n0 * 6); nh0 = __ldg(heur_k + (size_t)n0 * 6);
                nt1 = __ldg(tau_k + (size_t)n1 * 6); nh1 = __ldg(heur_k + (size_t)n1 * 6);
                nt2 = __ldg(tau_k + (size_t)n2 * 6); nh2 = __ldg(heur_k + (size_t)n2 * 6);
                nt3 = __ldg(tau_k + (size_t)n3 * 6); nh3 = __ldg(heur_k + (size_t)n3 * 6);
            }
            step(1u, u1, c2, ct2, ch2); rounds(IC<3>{}, IC<6>{});
            step(2u, u2, c3, ct3, ch3); rounds(IC<6>{}, IC<9>{});
            step(3u, u3, n0, nt0, nh0); rounds(IC<9>{}, IC<10>{});
            if (PREDICT) { c1 = n1; c2 = n2; c3 = n3; ct1 = nt1; ct2 = nt2; ct3 = nt3; ch1 = nh1; ch2 = nh2; ch3 = nh3; }
            u0 = __fmul_rn(__int2float_rn((int)(pc0 >> 1)), 4.656612873077392578125e-10f);
            u1 = __fmul_rn(__int2float_rn((int)(pc1 >> 1)), 4.656612873077392578125e-10f);
            u2 = __fmul_rn(__int2float_rn((int)(pc2 >> 1)), 4.656612873077392578125e-10f);
            u3 = __fmul_rn(__int2float_rn((int)(pc3 >> 1)), 4.656612873077392578125e-10f);
            if (T & 4u) {   // steps T-4 .. T+3 are complete: eight trail entries per ant, one coalesced store each
                const int base8 = (int)T - 4;
                if (k < steps - base8) { pid[base8 + k] = rec_id; pdir[base8 + k] = (uint8_t)rec_dir; }
            }
            T += 4u;
            kt ^= 4u;
        }
        if (T & 4u) {   // the last trip filled the lower half of a block of eight
            const int base8 = (int)T - 4;
            if (k < steps - base8) { pid[base8 + k] = rec_id; pdir[base8 + k] = (uint8_t)rec_dir; }
        }
        const bool arrived = has && steps > 0 && cur == goal;
        const int result = arrived ? steps : (parked ? -2 : -1);   // >= 0: steps of an ant that arrived, -1: dead, -2: parked -> pass 2
        int reason = 0;                                             // why a dead ant died: 1 no candidate, 2 roulette fall-through, 3 step cap
        if (result == -1) reason = steps >= cap ? 3 : (lastcb == 0u ? 1 : 2);

        // ---- park the ants whose table filled up (as k_walk2) ----------------------------------------------------------------
        {
            const bool pk = has && parked && !arrived;
            const unsigned pm = __ballot_sync(FULL, pk && k == 0);
            if (pm) {   // warp-uniform, rare
                int o = 0;
                if (pk && k == 0) o = (int)atomicAdd(&st->overflow_n, 1u);
                o = __shfl_sync(FULL, o, 0, 8);
                const int Eg = 1 << a.gtable_log2;
                for (unsigned rest = pm; rest; rest &= rest - 1) {
                    const int src = __ffs(rest) - 1;
                    const int oo = __shfl_sync(FULL, o, src);
                    uint4* z = reinterpret_cast<uint4*>(a.gtab + (size_t)oo * Eg);
                    for (int i = lane; i < Eg / 2; i += 32) z[i] = make_uint4(0u, 0u, 0u, 0u);
                }
                __syncwarp();
                if (pk) {
                    unsigned long long* ntab = a.gtab + (size_t)o * Eg;
                    for (int i = k; i < E; i += kGroup) {
                        const unsigned long long t = tab.load(i);
                        if (t == 0ull) continue;
                        unsigned sl = tile_hash((uint32_t)(t >> 32), (uint32_t)Eg);
                        while (atomicCAS(&ntab[sl], 0ull, t) != 0ull) sl = (sl + 1) & (Eg - 1);
                    }
                    if (k == 0) {
                        a.resume[o] = make_int4(cur, steps, 0, 0);
                        a.overflow_list[o] = (uint32_t)ant_local;
                    }
                }
                __syncwarp();
            }
        }
        if (has) {
            if (result == -2) {
                c_over++;   // its steps are counted by pass 2
            } else {
                c_arrived += result >= 0 ? 1 : 0;
                c_nocand += reason == 1 ? 1 : 0;
                c_fall += reason == 2 ? 1 : 0;
                c_cap += reason == 3 ? 1 : 0;
                c_steps += (unsigned long long)steps; c_ants++;
            }
            if (k == 0) a.ant_steps[ant_local] = result;
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
        if (c_vants) atomicAdd(&st->verified[0], (unsigned long long)c_vants);
        if (c_vsteps) atomicAdd(&st->verified[1], (unsigned long long)c_vsteps);
    }
}

}  // namespace wr
