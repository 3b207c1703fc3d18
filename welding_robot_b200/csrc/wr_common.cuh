// Shared helpers for libwrgpu.so (sm_100a only).  Compiled with -fmad=false: every float
// operation that feeds a comparison must round exactly like the reference's x86-64 SSE2
// scalar code (no FMA contraction, IEEE div/sqrt, denormals kept).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <string>

#include "../../include/wr_gpu.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libwrgpu is written for sm_100a (B200) only"
#endif

namespace wr {

void set_error(const char* fmt, ...);

#define WR_CUDA(expr)                                                                          \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            wr::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return WR_ERR_CUDA;                                                                \
        }                                                                                      \
    } while (0)

#define WR_REQUIRE(cond, status, msg)          \
    do {                                       \
        if (!(cond)) {                         \
            wr::set_error("%s", msg);          \
            return status;                     \
        }                                      \
    } while (0)

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

// Stream-ordered device memory from the device's default pool with the release threshold lifted, so
// that creating and destroying handles in a loop (one search per request) re-uses HBM instead of
// going back to the driver: a 403 MB pheromone field costs microseconds to obtain, not milliseconds.
cudaError_t pool_malloc(void** p, size_t bytes, cudaStream_t s);
void pool_free(void* p, cudaStream_t s);
template <class T> inline cudaError_t dmalloc(T** p, size_t bytes, cudaStream_t s) { return pool_malloc(reinterpret_cast<void**>(p), bytes, s); }

// ---- Philox4x32-10 (Salmon et al. SC'11), same stream layout as the CPU oracle ------------
constexpr uint32_t kPhiloxM0 = 0xD2511F53u, kPhiloxM1 = 0xCD9E8D57u;
constexpr uint32_t kPhiloxW0 = 0x9E3779B9u, kPhiloxW1 = 0xBB67AE85u;
constexpr uint32_t kStreamAcs3D = 0x3D3D0000u;
constexpr uint32_t kStreamGtsp = 0x65700000u;

__host__ __device__ __forceinline__ uint32_t philox_first(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < 10; r++) {
#ifdef __CUDA_ARCH__
        uint32_t hi0 = __umulhi(kPhiloxM0, c0), lo0 = kPhiloxM0 * c0;
        uint32_t hi1 = __umulhi(kPhiloxM1, c2), lo1 = kPhiloxM1 * c2;
#else
        uint64_t p0 = (uint64_t)kPhiloxM0 * c0, p1 = (uint64_t)kPhiloxM1 * c2;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
#endif
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += kPhiloxW0; k1 += kPhiloxW1;
    }
    return c0;
}

// all four output words (the 3-D search uses word (step & 3) of the block keyed by step >> 2)
__host__ __device__ __forceinline__ void philox4(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                                 uint32_t& o0, uint32_t& o1, uint32_t& o2, uint32_t& o3)
{
#pragma unroll
    for (int r = 0; r < 10; r++) {
#ifdef __CUDA_ARCH__
        uint32_t hi0 = __umulhi(kPhiloxM0, c0), lo0 = kPhiloxM0 * c0;
        uint32_t hi1 = __umulhi(kPhiloxM1, c2), lo1 = kPhiloxM1 * c2;
#else
        uint64_t p0 = (uint64_t)kPhiloxM0 * c0, p1 = (uint64_t)kPhiloxM1 * c2;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
#endif
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += kPhiloxW0; k1 += kPhiloxW1;
    }
    o0 = c0; o1 = c1; o2 = c2; o3 = c3;
}

// rand() stand-in: 31-bit draw (RAND_MAX = 2^31-1), see oracle/philox.h.
__host__ __device__ __forceinline__ uint32_t rand31(uint32_t seed_lo, uint32_t seed_hi, uint32_t a, uint32_t b, uint32_t c,
                                                    uint32_t stream)
{
    return philox_first(a, b, c, stream, seed_lo, seed_hi) >> 1;
}

// ---- device-side state of one search, updated by kernels so an iteration needs no host sync
struct IterState {
    int iter;            // iterations since begin()
    int colony;          // ants this iteration (global, all ranks)
    float lambda, Q;     // ACSRank_3D.hpp:248-249
    float predict;
    int best_steps;      // INT_MAX: none yet
    float best_L;        // +inf: none yet
    int best_changed;    // set by the ranking kernel when this iteration improved the best
    int best_ant;        // global ant index that produced it (this iteration)
    int n_eligible;      // ants that deposit this iteration (order <= lambda-1, arrived)
    float base;          // value of every in-bounds slot that never received a deposit since init/reset(): tau0 * rho^iterations, multiplied
                         // once per iteration exactly like the slots themselves would be (clean-tile field, see acs_kernels.cuh)
    int n_records;       // deposit records this iteration
    int n_records_sort;  // = n_records, or 0 on iterations whose deposits go through rank sets (the record path's kernels then run empty)
    int use_rankset;     // adaptive handles (WR_UPDATE_RANKSET): this iteration's deposit path, decided by k_iter_begin
    unsigned spread_tiles;   // pheromone tiles that received deposits in the last record-path iteration
    unsigned spread_slots;   // distinct slots that received deposits in the last rank-set iteration
    unsigned rankset_iters;  // iterations that took the rank-set path since begin
    unsigned queue;      // walk work queue (pass 1)
    unsigned queue2;     // pass 2 (resumed ants): its own counter, so no reset launch sits between the two passes
    unsigned overflow_n; // ants whose shared-memory visited table overflowed (pass 2)
    unsigned long long cnt[9];
    unsigned long long verified[2];   // k_walk3: ants completed by path verification, ant-steps it decided (wr_acs_walk_stats)
    // group deposits of a converged rank-set iteration (k_rank_small -> k_rankset_gen): eligible ranks whose local ant walked
    // exactly the best path set their bits once per best-path slot, from the trail of one of them (the representative)
    int grp_rep;         // local index of the representative ant, -1: no group this iteration
    int grp_steps;       // its step count (best_n - 1 of the path it verified against)
    unsigned grp_ranks;  // eligible ranks in the group this iteration (0 on iterations without rank sets; wr_acs_group_stats)
    unsigned long long grp_ranks_total;   // the same, summed over the earlier iterations since begin (k_iter_begin adds grp_ranks)
};

}  // namespace wr
