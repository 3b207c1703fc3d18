// Host-side handle layouts shared between the translation units of libwrgpu.so.
#pragma once
#include <vector>

#include "wr_common.cuh"

struct wr_grid {
    int device = 0;
    int rx = 0, ry = 0, rz = 0, wall = 0;
    size_t N = 0;
    float precision = 0;
    float gmin[3] = {0, 0, 0}, gmax[3] = {0, 0, 0};
    std::vector<float> h_xs, h_ys, h_zs;  // node coordinates are separable (model_grid_map.hpp:204-211)
    float* d_coords = nullptr;            // [xs | ys | zs] in HBM
    uint32_t* d_bits = nullptr;           // occupancy, 1 bit per node, 1 = occupied
    size_t nwords = 0;
    uint8_t* d_open6 = nullptr;           // per node: bit k set <=> neighbour k in bounds and free (built on demand)
    std::vector<uint32_t> h_bits;         // host mirror for endpoint snapping (filled on demand)
    uint32_t* d_clear = nullptr;          // per node: squared index distance to the nearest occupied node (built on demand)
    uint64_t occupied = 0, tests = 0;
    float vox_ms = 0;
    float clear_ms = 0;                   // device ms of the passes that built d_clear
};

namespace wr {
// grid.cu
int grid_alloc_common(wr_grid* g);
int grid_ensure_open6(wr_grid* g, cudaStream_t s);
int grid_ensure_host_bits(wr_grid* g);
// clearance.cu
int grid_ensure_clearance(wr_grid* g);
inline bool grid_is_free_host(const wr_grid* g, size_t id) { return !((g->h_bits[id >> 5] >> (id & 31)) & 1u); }

// radix_sort.cu — stable LSD radix sort of (u32 key, u32 value) pairs, count on the device.
struct SortPlan {
    uint32_t *keys_a = nullptr, *keys_b = nullptr, *vals_a = nullptr, *vals_b = nullptr;  // ping-pong
    uint32_t* hist = nullptr;  // 256 * max_tiles
    size_t max_n = 0;
    int max_tiles = 0;
};
int sort_plan_create(SortPlan* p, size_t max_n, cudaStream_t s);
void sort_plan_destroy(SortPlan* p, cudaStream_t s);
// Sorts keys_a/vals_a (first *d_n entries) by the low `key_bits` bits; result lands in
// keys_a/vals_a again when the pass count is even, else in keys_b/vals_b: returns which.
int sort_pairs(SortPlan* p, const int* d_n, int key_bits, cudaStream_t s, bool* result_in_b, bool input_in_b = false);
// stable partition: pairs with key in [lo, lo+span) to the front (their count -> *d_count_out); input keys_a/vals_a, result in keys_b/vals_b
int sort_partition(SortPlan* p, const int* d_n, uint32_t lo, uint32_t span, cudaStream_t s, int* d_count_out);
int sort_preload();

// comm.cu — NCCL (opened at run time) for the rendezvous of a sharded colony
int comm_get(const void* unique_id, int rank, int nranks, void** comm_out);
int comm_all_gather(void* comm, const void* d_send, void* d_recv, size_t bytes, cudaStream_t s);
void comm_release();
}  // namespace wr
