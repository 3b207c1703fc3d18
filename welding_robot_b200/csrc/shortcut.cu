// Line-of-sight shortcutting of node rows (searched paths, ant trails, caller polylines) with a clearance floor.  An
// addition with no reference counterpart.
//
// In index space a node (x, y, z) owns the closed cube [x-1/2, x+1/2] x [y-1/2, y+1/2] x [z-1/2, z+1/2].  The cover of
// the segment between two nodes is every cube that meets the closed segment (a conservative supercover: a segment
// through a cube edge or corner takes every cube that shares it).  A cube blocks iff d2 <= r2 (at r2 = 0: iff it is
// occupied, read from the occupancy bits, no field); a segment is clear iff no cube of its cover blocks.  Greedy
// waypoints: from anchor w the next waypoint is the largest j in (w, min(n-1, w+span)] whose segment is clear, else
// w+1 (the fallback: the row's own segment is kept and counted in `blocked`).
//
// One launch for all rows, one CTA per row.  The CTA decodes its node ids to (x, y, z) once, then loops over anchors:
// the candidates of the window are taken from the top down, kShortcutThreads at a time, each thread walking its
// candidate's cover with an exact integer DDA and stopping at the first blocking cube; the first chunk with a clear
// candidate ends the anchor and the smallest clear thread index (the largest j) wins.  No atomics: the result is a
// pure function of (grid, row, r2, max_span).
//
// The DDA: endpoints are integers and cube faces half-integers, so axis k (|d_k| > 0) crosses its c-th face (c = 0 ..
// |d_k|-1) at t = (2c+1) / (2|d_k|).  Scaled by 2 |dx||dy||dz| (zero factors dropped) that is T_k = (2c+1) P_k with P_k
// the product of the other non-zero |d|, an exact int64 (T_k <= 2 |dx||dy||dz| <= 2N).  The next event is the least
// T_k; a 2- or 3-way tie is an edge or corner touch, where the segment meets every cube v + e(U) for the non-empty
// subsets U of the tied axes.  Between events the point lies inside one cube.  Cover size = 1 + sum over events of
// (2^ties - 1): a lattice edge covers 2 cubes, a (1,1,0) step 4, a (1,1,1) step 8.
#include <limits.h>

#include <algorithm>

#include "wr_internal.cuh"

namespace wr {

constexpr int kShortcutThreads = 128;
constexpr int kShortcutWarps = kShortcutThreads / 32;
constexpr int kCoverBatch = 8;   // cubes generated before their loads are issued together

struct Seg {
    long long v;                  // current cube (node id)
    long long st[3];              // signed id stride of a step along each axis
    long long T[3], inc[3];       // next face crossing per axis (LLONG_MAX: none left), its increment 2 P_k
    int left[3];                  // face crossings left per axis
    int sub, S;                   // pending subsets of the tied axes S (enumerated S, (S-1)&S, ...; 0: none)
    bool first;                   // the start cube is still to be emitted
};

__device__ __forceinline__ long long subset_offset(const Seg& s, int u)
{
    return ((u & 1) ? s.st[0] : 0) + ((u & 2) ? s.st[1] : 0) + ((u & 4) ? s.st[2] : 0);
}

// next cube of the cover, -1 when the cover is exhausted
__device__ __forceinline__ long long next_cube(Seg& s)
{
    if (s.first) { s.first = false; return s.v; }
    if (!s.sub) {
        const long long m = min(s.T[0], min(s.T[1], s.T[2]));
        if (m == LLONG_MAX) return -1;
        s.S = 0;
#pragma unroll
        for (int k = 0; k < 3; k++)
            if (s.T[k] == m) {
                s.S |= 1 << k;
                s.T[k] = --s.left[k] ? s.T[k] + s.inc[k] : LLONG_MAX;
            }
        s.sub = s.S;
    }
    const long long c = s.v + subset_offset(s, s.sub);
    s.sub = (s.sub - 1) & s.S;
    if (!s.sub) s.v += subset_offset(s, s.S);   // all cubes of the event visited: move past it
    return c;
}

template <bool kBits>
__device__ __forceinline__ bool cube_blocks(const uint32_t* __restrict__ src, long long c, uint32_t r2)
{
    if (kBits) return (__ldg(src + (c >> 5)) >> (c & 31)) & 1u;
    return __ldg(src + c) <= r2;
}

// is the segment between node `id` at index point a and the node at b clear?
template <bool kBits>
__device__ bool segment_clear(long long id, int4 a, int4 b, long long rx, long long rxy, const uint32_t* __restrict__ src, uint32_t r2)
{
    const int d[3] = {b.x - a.x, b.y - a.y, b.z - a.z};
    const long long stride[3] = {1, rx, rxy};
    long long ad[3], f[3];
    Seg s;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        ad[k] = d[k] < 0 ? -(long long)d[k] : d[k];
        f[k] = ad[k] ? ad[k] : 1;
        s.st[k] = d[k] < 0 ? -stride[k] : stride[k];
        s.left[k] = (int)ad[k];
    }
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const long long p = f[(k + 1) % 3] * f[(k + 2) % 3];
        s.T[k] = ad[k] ? p : LLONG_MAX;
        s.inc[k] = 2 * p;
    }
    s.v = id; s.sub = 0; s.S = 0; s.first = true;
    for (;;) {
        long long c[kCoverBatch];
#pragma unroll
        for (int k = 0; k < kCoverBatch; k++) c[k] = next_cube(s);
        bool blocked = false;
#pragma unroll
        for (int k = 0; k < kCoverBatch; k++)
            if (c[k] >= 0) blocked |= cube_blocks<kBits>(src, c[k], r2);
        if (blocked) return false;
        if (c[kCoverBatch - 1] < 0) return true;
    }
}

// Rows: row p = ids[off[p] .. off[p+1]).  xyz: scratch of the same length (decoded index points).
template <bool kBits>
__global__ void __launch_bounds__(kShortcutThreads) k_shortcut(const long long* __restrict__ ids, const long long* __restrict__ off,
                                                               int4* __restrict__ xyz, int rx, int ry, const uint32_t* __restrict__ src,
                                                               uint32_t r2, int max_span, const float* __restrict__ coords,
                                                               int* __restrict__ keep, int* __restrict__ nkeep, int* __restrict__ blocked,
                                                               double* __restrict__ length)
{
    __shared__ unsigned s_clear[kShortcutWarps];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long base = off[blockIdx.x];
    const int n = (int)(off[blockIdx.x + 1] - base);
    const long long rxy = (long long)rx * ry;
    const long long* row = ids + base;
    int4* p = xyz + base;
    for (int i = tid; i < n; i += kShortcutThreads) {
        const long long id = row[i];
        const long long z = id / rxy, r = id - z * rxy, y = r / rx;
        p[i] = make_int4((int)(r - y * rx), (int)y, (int)z, 0);
    }
    __syncthreads();   // p is read by every thread of the CTA below
    if (n == 0) {
        if (tid == 0) { nkeep[blockIdx.x] = 0; blocked[blockIdx.x] = 0; length[blockIdx.x] = 0.0; }
        return;
    }
    const long long span = max_span > 0 ? max_span : n;
    const float* cx = coords;
    const float* cy = coords + rx;
    const float* cz = coords + rx + ry;
    int w = 0, k = 0, nb = 0;
    double L = 0.0;
    if (tid == 0) keep[base] = 0;
    while (w < n - 1) {
        const int top = (int)min((long long)n - 1, w + span);
        const int4 a = p[w];
        const long long aid = row[w];
        int nw = -1;
        for (int hi = top; hi > w && nw < 0; hi -= kShortcutThreads) {
            const int j = hi - tid;
            const bool ok = j > w && segment_clear<kBits>(aid, a, p[j], rx, rxy, src, r2);
            const unsigned m = __ballot_sync(0xffffffffu, ok);
            if (lane == 0) s_clear[warp] = m;
            __syncthreads();
#pragma unroll
            for (int q = 0; q < kShortcutWarps; q++) {
                const unsigned mq = s_clear[q];
                if (mq) { nw = hi - (32 * q + __ffs(mq) - 1); break; }
            }
            __syncthreads();   // s_clear is rewritten by the next chunk
        }
        if (nw < 0) { nw = w + 1; nb++; }
        if (tid == 0) {
            keep[base + ++k] = nw;
            const int4 b = p[nw];
            const double dx = (double)cx[a.x] - (double)cx[b.x];
            const double dy = (double)cy[a.y] - (double)cy[b.y];
            const double dz = (double)cz[a.z] - (double)cz[b.z];
            L += sqrt(dx * dx + dy * dy + dz * dz);
        }
        w = nw;
    }
    if (tid == 0) { nkeep[blockIdx.x] = k + 1; blocked[blockIdx.x] = nb; length[blockIdx.x] = L; }
}

}  // namespace wr

using namespace wr;

extern "C" int wr_grid_shortcut_paths(wr_grid* g, const int64_t* ids, const int64_t* offsets, int nrows, uint32_t r2, int max_span,
                                      int32_t* keep, int32_t* nkeep, int32_t* blocked, double* length)
{
    WR_REQUIRE(g && nrows >= 0 && max_span >= 0, WR_ERR_INVALID, "wr_grid_shortcut_paths: bad argument");
    if (nrows == 0) return WR_OK;
    WR_REQUIRE(offsets && nkeep, WR_ERR_INVALID, "wr_grid_shortcut_paths: null");
    WR_REQUIRE(offsets[0] == 0, WR_ERR_INVALID, "wr_grid_shortcut_paths: offsets[0] must be 0");
    for (int r = 0; r < nrows; r++) {
        WR_REQUIRE(offsets[r + 1] >= offsets[r], WR_ERR_INVALID, "wr_grid_shortcut_paths: offsets must be non-decreasing");
        WR_REQUIRE(offsets[r + 1] - offsets[r] <= INT32_MAX, WR_ERR_INVALID, "wr_grid_shortcut_paths: a row is longer than INT32_MAX");
    }
    const int64_t total = offsets[nrows];
    WR_REQUIRE(total == 0 || (ids && keep), WR_ERR_INVALID, "wr_grid_shortcut_paths: null");
    for (int64_t i = 0; i < total; i++)
        WR_REQUIRE(ids[i] >= 0 && (uint64_t)ids[i] < g->N, WR_ERR_INVALID, "wr_grid_shortcut_paths: node id out of range");
    if (r2 > 0) {
        const int rc = grid_ensure_clearance(g);
        if (rc != WR_OK) return rc;
    }
    WR_CUDA(cudaSetDevice(g->device));
    cudaStream_t s = 0;
    const size_t nt = (size_t)std::max<int64_t>(total, 1);
    long long *d_ids = nullptr, *d_off = nullptr;
    int4* d_xyz = nullptr;
    int *d_keep = nullptr, *d_nkeep = nullptr, *d_blocked = nullptr;
    double* d_len = nullptr;
    cudaError_t e = dmalloc(&d_ids, nt * sizeof(long long), s);
    if (e == cudaSuccess) e = dmalloc(&d_off, (size_t)(nrows + 1) * sizeof(long long), s);
    if (e == cudaSuccess) e = dmalloc(&d_xyz, nt * sizeof(int4), s);
    if (e == cudaSuccess) e = dmalloc(&d_keep, nt * sizeof(int), s);
    if (e == cudaSuccess) e = dmalloc(&d_nkeep, (size_t)nrows * sizeof(int), s);
    if (e == cudaSuccess) e = dmalloc(&d_blocked, (size_t)nrows * sizeof(int), s);
    if (e == cudaSuccess) e = dmalloc(&d_len, (size_t)nrows * sizeof(double), s);
    static_assert(sizeof(long long) == sizeof(int64_t) && sizeof(int) == sizeof(int32_t), "host and device element sizes");
    if (e == cudaSuccess && total) e = cudaMemcpyAsync(d_ids, ids, (size_t)total * sizeof(int64_t), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_off, offsets, (size_t)(nrows + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
        if (r2 == 0)
            k_shortcut<true><<<(unsigned)nrows, kShortcutThreads, 0, s>>>(d_ids, d_off, d_xyz, g->rx, g->ry, g->d_bits, r2, max_span,
                                                                         g->d_coords, d_keep, d_nkeep, d_blocked, d_len);
        else
            k_shortcut<false><<<(unsigned)nrows, kShortcutThreads, 0, s>>>(d_ids, d_off, d_xyz, g->rx, g->ry, g->d_clear, r2, max_span,
                                                                          g->d_coords, d_keep, d_nkeep, d_blocked, d_len);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess && total) e = cudaMemcpyAsync(keep, d_keep, (size_t)total * sizeof(int32_t), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(nkeep, d_nkeep, (size_t)nrows * sizeof(int32_t), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && blocked) e = cudaMemcpyAsync(blocked, d_blocked, (size_t)nrows * sizeof(int32_t), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && length) e = cudaMemcpyAsync(length, d_len, (size_t)nrows * sizeof(double), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    pool_free(d_ids, s); pool_free(d_off, s); pool_free(d_xyz, s); pool_free(d_keep, s);
    pool_free(d_nkeep, s); pool_free(d_blocked, s); pool_free(d_len, s);
    if (e != cudaSuccess) { set_error("wr_grid_shortcut_paths: %s", cudaGetErrorString(e)); return WR_ERR_CUDA; }
    return WR_OK;
}
