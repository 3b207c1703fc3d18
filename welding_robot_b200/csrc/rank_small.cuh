// Colony ranking in ONE kernel for colonies of up to kRankSmallMax ants (the reference's adaptive colonies are tens of
// ants, BASELINE's C2 colony is 4096, four ranks of it 16384): keys, stable LSD radix sort, best decision, eligibility, record offsets and the
// old best path's membership bits — what launch_rank otherwise spreads over k_rank_keys + 3 kernels per sort pass +
// k_rank_finish + k_best_clear (10 dependent launches whose cost is launch latency, not work).
//
// Sort: a single CTA of 1024 threads, keys and values ping-pong in shared memory, 8-bit digits.  Warp w owns the
// contiguous index block [w*chunk, (w+1)*chunk) and walks it 32 keys at a time, so "earlier index" = (earlier warp) or
// (same warp, earlier round) or (same round, lower lane): a key's position inside its digit is
//     prefix over (digit, warp) of the per-warp counts  +  count of this warp's earlier rounds  +  match-any rank
// which makes every pass stable, hence the result the oracle's total order (key, ant index).
#pragma once
#include "acs_kernels.cuh"

namespace wr {

constexpr int kRankSmallMax = 16384;
constexpr int kRankSmallThreads = 1024;
constexpr int kRankSmallRounds = kRankSmallMax / kRankSmallThreads;   // 32-key rounds per warp
// dynamic shared memory: keys[2][max] (u32) + vals[2][max] (u16: ant indices < 65536) + whist[32][256] (u32) = 224 KB
constexpr size_t kRankSmallSmem = (size_t)2 * kRankSmallMax * sizeof(uint32_t) + (size_t)2 * kRankSmallMax * sizeof(uint16_t) + (size_t)32 * 256 * sizeof(uint32_t);

// Keys + stable sort of ants [first, first + n) in shared memory; returns which ping-pong buffer holds the result
// (kbuf[src] keys, vbuf[src] ant indices relative to `first`).  All 1024 threads of the CTA take part.
__device__ __forceinline__ int rank_sort_chunk(uint32_t* const kbuf[2], uint16_t* const vbuf[2], uint32_t* whist, uint32_t* warp_sum, const int* __restrict__ ant_steps,
                                               const float* __restrict__ ant_L, int first, int n, int cap, int key_bits)
{
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const bool k26 = ant_L != nullptr;
    const int rounds = (n + kRankSmallThreads - 1) / kRankSmallThreads;   // per warp
    const int chunk = rounds * 32;

    // ---- keys (k_rank_keys / k_rank_keys26) ----
    for (int i = threadIdx.x; i < n; i += kRankSmallThreads) {
        const int s = ant_steps[first + i];
        kbuf[0][i] = k26 ? (s < 0 ? 0x7F800000u : __float_as_uint(ant_L[first + i])) : (s < 0 ? (uint32_t)(cap + 1) : (uint32_t)s);
        vbuf[0][i] = (uint16_t)i;
    }
    __syncthreads();

    // ---- stable LSD radix sort, 8 bits per pass ----
    int src = 0;
    for (int shift = 0; shift < key_bits; shift += 8, src ^= 1) {
        const uint32_t* ki = kbuf[src];
        const uint16_t* vi = vbuf[src];
        for (int d = lane; d < 256; d += 32) whist[w * 256 + d] = 0;
        __syncwarp();
        uint32_t local[kRankSmallRounds];   // position of this thread's key of round r among its warp's keys of the same digit
#pragma unroll
        for (int r = 0; r < kRankSmallRounds; r++) {
            if (r < rounds) {   // warp-uniform
                const int idx = w * chunk + r * 32 + lane;
                const bool ok = idx < n;
                const uint32_t d = ok ? ((ki[idx] >> shift) & 255u) : 256u;
                const unsigned peers = __match_any_sync(FULL, d);
                const uint32_t base = ok ? whist[w * 256 + d] : 0u;
                local[r] = base + (uint32_t)__popc(peers & ((1u << lane) - 1u));
                __syncwarp();
                if (ok && lane == __ffs(peers) - 1) whist[w * 256 + d] = base + (uint32_t)__popc(peers);
                __syncwarp();
            }
        }
        __syncthreads();
        // exclusive scan of the 8192 counters in (digit, warp) order: thread t owns digit t/4, warps (t%4)*8 .. +7
        {
            const int d = threadIdx.x >> 2, w0 = (threadIdx.x & 3) * 8;
            uint32_t c[8], sum = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) { c[j] = whist[(w0 + j) * 256 + d]; sum += c[j]; }
            uint32_t incl = sum;
            for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += u; }
            if (lane == 31) warp_sum[w] = incl;
            __syncthreads();
            if (w == 0) {
                const uint32_t s = warp_sum[lane];
                uint32_t si = s;
                for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(FULL, si, o); if (lane >= o) si += u; }
                warp_sum[lane] = si - s;
            }
            __syncthreads();
            uint32_t run = warp_sum[w] + (incl - sum);
#pragma unroll
            for (int j = 0; j < 8; j++) { whist[(w0 + j) * 256 + d] = run; run += c[j]; }
        }
        __syncthreads();
        uint32_t* ko = kbuf[src ^ 1];
        uint16_t* vo = vbuf[src ^ 1];
#pragma unroll
        for (int r = 0; r < kRankSmallRounds; r++) {
            if (r < rounds) {
                const int idx = w * chunk + r * 32 + lane;
                if (idx < n) {
                    const uint32_t key = ki[idx];
                    const uint32_t pos = whist[w * 256 + ((key >> shift) & 255u)] + local[r];
                    ko[pos] = key; vo[pos] = vi[idx];
                }
            }
        }
        __syncthreads();
    }
    return src;
}

// steps26 / ant_L: K = 26 (key = bits of L); else key = steps (cap+1 for a dead ant), as k_rank_keys / k_rank_keys26.
__global__ void __launch_bounds__(kRankSmallThreads) k_rank_small(IterState* st, const int* __restrict__ ant_steps, const float* __restrict__ ant_L, int cap,
                                                                   int key_bits, const float* __restrict__ Ltab, uint32_t* __restrict__ out_keys,
                                                                   uint32_t* __restrict__ out_vals, uint32_t* __restrict__ rec_off,
                                                                   int* __restrict__ order_of_ant, const int* __restrict__ best_n,
                                                                   const uint32_t* __restrict__ best_ids, uint32_t* onbest)
{
    extern __shared__ __align__(16) uint32_t rs_smem[];
    uint32_t* kbuf[2] = {rs_smem, rs_smem + kRankSmallMax};
    uint16_t* vbase = reinterpret_cast<uint16_t*>(rs_smem + 2 * kRankSmallMax);
    uint16_t* vbuf[2] = {vbase, vbase + kRankSmallMax};
    uint32_t* whist = rs_smem + 3 * kRankSmallMax;   // [warp][digit]
    __shared__ uint32_t warp_sum[32];
    __shared__ uint32_t carry, elig_total;

    constexpr unsigned FULL = 0xffffffffu;
    const int n = st->colony;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const bool k26 = ant_L != nullptr;
    const int src = rank_sort_chunk(kbuf, vbuf, whist, warp_sum, ant_steps, ant_L, 0, n, cap, key_bits);
    const uint32_t* keys = kbuf[src];
    const uint16_t* vals = vbuf[src];

    // ---- k_rank_finish: best decision (:263-264), eligibility (:200), record offsets ----
    const float lambda = st->lambda;
    if (threadIdx.x == 0) {
        carry = 0; elig_total = 0;
        if (n > 0 && k26) {
            const float L0 = __uint_as_float(keys[0]);
            if (L0 < st->best_L) { st->best_steps = ant_steps[vals[0]]; st->best_L = L0; st->best_changed = 1; st->best_ant = (int)vals[0]; }
        } else if (n > 0) {
            const int s = (int)keys[0];
            if (s <= cap && s < st->best_steps) { st->best_steps = s; st->best_L = Ltab[s]; st->best_changed = 1; st->best_ant = (int)vals[0]; }
        }
    }
    __syncthreads();
    for (int base = 0; base < n; base += kRankSmallThreads) {
        const int r = base + threadIdx.x;
        uint32_t len = 0; bool el = false;
        if (r < n) {
            const uint32_t key = keys[r], ant = vals[r];
            out_keys[r] = key; out_vals[r] = ant;
            const int s = k26 ? ant_steps[ant] : (int)key;
            const bool arrived = k26 ? key != 0x7F800000u : s <= cap;
            const int order = r + 1;
            order_of_ant[ant] = order;
            el = arrived && !((float)order > __fsub_rn(lambda, 1.0f));   // :200
            len = el ? (uint32_t)s : 0u;
        }
        uint32_t incl = len;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += u; }
        if (lane == 31) warp_sum[w] = incl;
        const unsigned em = __ballot_sync(FULL, el);
        if (lane == 0 && em) atomicAdd(&elig_total, (uint32_t)__popc(em));
        __syncthreads();
        if (w == 0) {
            const uint32_t s = warp_sum[lane];
            uint32_t si = s;
            for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(FULL, si, o); if (lane >= o) si += u; }
            warp_sum[lane] = si - s;
        }
        __syncthreads();
        const uint32_t excl = carry + warp_sum[w] + (incl - len);
        if (r < n) rec_off[r] = excl;
        __syncthreads();
        if (threadIdx.x == kRankSmallThreads - 1) carry = excl + len;
        __syncthreads();
    }
    if (threadIdx.x == 0) { st->n_eligible = (int)elig_total; st->n_records = (int)carry; st->n_records_sort = st->use_rankset ? 0 : (int)carry; st->cnt[7] += carry; }

    // ---- k_best_clear: best = agentK (:264) drops the old best path's membership bits ----
    if (st->best_changed) {   // written by thread 0 before the barrier above
        const int nb = *best_n;
        for (int i = threadIdx.x; i < nb; i += kRankSmallThreads) {
            const uint32_t id = best_ids[i];
            atomicAnd(&onbest[id >> 5], ~(1u << (id & 31)));
        }
    }
}

// ---- colonies beyond one CTA (C2 on eight GPUs: 32 768 ants; C3: 65 536) -----------------------------------------------------
// k_rank_chunks: one CTA per chunk of kRankChunk ants sorts its chunk as above (chunks in parallel) -> chunk-sorted
// (key, ant) lists in global memory.  k_rank_merge: an element's final position is its position in its own chunk plus, for
// every other chunk, the number of elements that precede it there — keys <= its key in chunks of LOWER ant indices (ties go
// to the lower index), keys < its key in the others: binary searches in L2-resident lists, one thread per element.
// k_rank_finish_prefix: best decision, eligibility and record offsets; eligible ranks are a prefix of the sorted colony
// (arrived ants first) no longer than w_max, so one CTA scans min(n, w_max + 1) elements instead of the colony.
constexpr int kRankChunk = 4096;   // ants per chunk of the chunked path: short sorts, many CTAs in parallel
constexpr size_t kRankChunkSmem = (size_t)12 * kRankChunk + (size_t)32 * 256 * sizeof(uint32_t);
__global__ void __launch_bounds__(kRankSmallThreads) k_rank_chunks(const IterState* st, const int* __restrict__ ant_steps, const float* __restrict__ ant_L, int cap,
                                                                    int key_bits, uint32_t* __restrict__ ck, uint32_t* __restrict__ cv)
{
    extern __shared__ __align__(16) uint32_t rs_smem[];
    uint32_t* kbuf[2] = {rs_smem, rs_smem + kRankChunk};
    uint16_t* vbase = reinterpret_cast<uint16_t*>(rs_smem + 2 * kRankChunk);
    uint16_t* vbuf[2] = {vbase, vbase + kRankChunk};
    uint32_t* whist = rs_smem + 3 * kRankChunk;
    __shared__ uint32_t warp_sum[32];
    const int n = st->colony;
    const int first = blockIdx.x * kRankChunk;
    if (first >= n) return;
    const int nc = min(kRankChunk, n - first);
    const int src = rank_sort_chunk(kbuf, vbuf, whist, warp_sum, ant_steps, ant_L, first, nc, cap, key_bits);
    for (int i = threadIdx.x; i < nc; i += kRankSmallThreads) { ck[first + i] = kbuf[src][i]; cv[first + i] = (uint32_t)first + vbuf[src][i]; }
}

// One CTA per 1024 consecutive elements of one chunk.  With keys16 the other chunks' keys are staged in shared memory 16 bits
// wide (launch_rank sets it only for K = 6 step-count keys with cap + 1 <= 0xFFFF; K = 26 keys and larger caps are compared
// through global memory), so the 12-step binary searches run at shared-memory latency instead of one L2 round trip per step.
constexpr int kRankMergeThreads = 1024;
__global__ void __launch_bounds__(kRankMergeThreads) k_rank_merge(const IterState* st, const uint32_t* __restrict__ ck, const uint32_t* __restrict__ cv,
                                                                   uint32_t* __restrict__ out_keys, uint32_t* __restrict__ out_vals, int* __restrict__ order_of_ant,
                                                                   int keys16)
{
    extern __shared__ __align__(16) uint16_t mk_smem[];   // [chunks that fit][kRankChunk]
    const int n = st->colony;
    const int nchunks = (n + kRankChunk - 1) / kRankChunk;
    const int i = blockIdx.x * kRankMergeThreads + threadIdx.x;
    const int mine = (blockIdx.x * kRankMergeThreads) / kRankChunk;   // CTA-uniform: kRankChunk is a multiple of the CTA size
    constexpr int kStage = 24;                                         // chunks staged per round (192 KB)
    uint32_t key = 0, ant = 0;
    int pos = 0;
    if (i < n) { key = ck[i]; ant = cv[i]; pos = i - mine * kRankChunk; }
    for (int c0 = 0; c0 < nchunks; c0 += kStage) {
        const int c1 = min(c0 + kStage, nchunks);
        if (keys16) {
            __syncthreads();
            for (int j = threadIdx.x; j < (c1 - c0) * kRankChunk; j += kRankMergeThreads) {
                const int g = c0 * kRankChunk + j;
                mk_smem[j] = g < n ? (uint16_t)ck[g] : (uint16_t)0xFFFF;
            }
            __syncthreads();
        }
        if (i < n) {
            for (int c = c0; c < c1; c++) {
                if (c == mine) continue;
                int lo = 0, hi = min(kRankChunk, n - c * kRankChunk);
                if (keys16) {
                    const uint16_t* k = mk_smem + (size_t)(c - c0) * kRankChunk;
                    if (c < mine) { while (lo < hi) { const int mid = (lo + hi) >> 1; if (k[mid] <= key) lo = mid + 1; else hi = mid; } }   // upper bound
                    else { while (lo < hi) { const int mid = (lo + hi) >> 1; if (k[mid] < key) lo = mid + 1; else hi = mid; } }           // lower bound
                } else {
                    const uint32_t* k = ck + (size_t)c * kRankChunk;
                    if (c < mine) { while (lo < hi) { const int mid = (lo + hi) >> 1; if (k[mid] <= key) lo = mid + 1; else hi = mid; } }
                    else { while (lo < hi) { const int mid = (lo + hi) >> 1; if (k[mid] < key) lo = mid + 1; else hi = mid; } }
                }
                pos += lo;
            }
        }
    }
    if (i < n) {
        out_keys[pos] = key; out_vals[pos] = ant;
        order_of_ant[ant] = pos + 1;
    }
}

__global__ void __launch_bounds__(1024) k_rank_finish_prefix(IterState* st, const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, int cap,
                                                              const float* __restrict__ Ltab, uint32_t* __restrict__ rec_off, int w_max,
                                                              const int* __restrict__ steps26, const int* __restrict__ best_n,
                                                              const uint32_t* __restrict__ best_ids, uint32_t* onbest)
{   // steps26 != nullptr (K = 26): keys are the bits of L and an ant's step count comes from steps26[ant]
    __shared__ uint32_t warp_sum[32];
    __shared__ uint32_t carry, elig_total;
    constexpr unsigned FULL = 0xffffffffu;
    const int n = st->colony;
    const float lambda = st->lambda;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        carry = 0; elig_total = 0;
        if (n > 0 && steps26) {
            const float L0 = __uint_as_float(keys[0]);
            if (L0 < st->best_L) { st->best_steps = steps26[vals[0]]; st->best_L = L0; st->best_changed = 1; st->best_ant = (int)vals[0]; }
        } else if (n > 0) {
            const int s = (int)keys[0];
            if (s <= cap && s < st->best_steps) { st->best_steps = s; st->best_L = Ltab[s]; st->best_changed = 1; st->best_ant = (int)vals[0]; }
        }
    }
    __syncthreads();
    const int lim = min(n, w_max + 1);
    for (int base = 0; base < lim; base += 1024) {
        const int r = base + threadIdx.x;
        uint32_t len = 0; bool el = false;
        if (r < lim) {
            const int s = steps26 ? steps26[vals[r]] : (int)keys[r];
            const bool arrived = steps26 ? keys[r] != 0x7F800000u : s <= cap;
            el = arrived && !((float)(r + 1) > __fsub_rn(lambda, 1.0f));   // :200
            len = el ? (uint32_t)s : 0u;
        }
        uint32_t incl = len;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += u; }
        if (lane == 31) warp_sum[w] = incl;
        const unsigned em = __ballot_sync(FULL, el);
        if (lane == 0 && em) atomicAdd(&elig_total, (uint32_t)__popc(em));
        __syncthreads();
        if (w == 0) {
            const uint32_t s = warp_sum[lane];
            uint32_t si = s;
            for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(FULL, si, o); if (lane >= o) si += u; }
            warp_sum[lane] = si - s;
        }
        __syncthreads();
        const uint32_t excl = carry + warp_sum[w] + (incl - len);
        if (r < lim) rec_off[r] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) carry = excl + len;
        __syncthreads();
    }
    if (threadIdx.x == 0) { st->n_eligible = (int)elig_total; st->n_records = (int)carry; st->n_records_sort = st->use_rankset ? 0 : (int)carry; st->cnt[7] += carry; }
    if (st->best_changed) {   // k_best_clear: written by thread 0 before the first barrier above
        const int nb = *best_n;
        for (int i = threadIdx.x; i < nb; i += 1024) {
            const uint32_t id = best_ids[i];
            atomicAnd(&onbest[id >> 5], ~(1u << (id & 31)));
        }
    }
}

}  // namespace wr
