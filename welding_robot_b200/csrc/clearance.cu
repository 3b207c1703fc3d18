// Clearance: exact squared Euclidean distance (index units) of every node to the nearest occupied node, and what is
// built on it -- point queries and obstacle inflation.  An addition with no reference counterpart.
//
// d2(x,y,z) = min over occupied (x',y',z') of (x-x')^2 + (y-y')^2 + (z-z')^2, uint32, 0 on occupied nodes, UINT32_MAX
// everywhere when nothing is occupied.  Three separable passes, exact integer arithmetic, no atomics (the result does
// not depend on scheduling):
//   pass 1 (x)  one warp per row reads the bit-packed occupancy and writes the squared distance to the nearest set bit
//               of the row (UINT32_MAX: none) -> field
//   pass 2 (y)  lower envelope of parabolas along every y column (Meijster et al., integer Sep with an int64
//               numerator) field -> tmp
//   pass 3 (z)  the same along z, tmp -> field
// Passes 2 and 3 give the lanes of a CTA consecutive x, so every step reads and writes 128 contiguous bytes; each lane
// keeps its envelope stack (16-bit apex, 16-bit start, packed in one word) in shared memory.  UINT32_MAX entries take
// no part in an envelope; a line without a finite entry stays UINT32_MAX.  Every pass is linear in the line length.
// Bytes moved: 4 (pass 1 write) + 8 + 8 (read + write in passes 2, 3) per node, plus the bits and the stack tops'
// re-reads (L2 hits).
#include <limits.h>

#include <algorithm>

#include "wr_internal.cuh"

namespace wr {

constexpr uint32_t kFar = 0xffffffffu;
constexpr int kMaxClearanceAxis = 32768;        // 3 * 32767^2 < 2^32: every sum of the passes fits a uint32
constexpr int kRowWarps = 8;                    // pass 1: rows per 256-thread CTA
constexpr int kColPrefetch = 8;                 // passes 2/3: independent loads in flight per lane
constexpr size_t kColSmemMax = 227 * 1024;

// bits of nodes row*rx + x .. x+31 (bit j = node x+j), zero past the row's end (d_bits has 4 words of zero padding)
__device__ __forceinline__ uint32_t row_window(const uint32_t* __restrict__ bits, size_t row, int rx, int x)
{
    if (x >= rx) return 0u;
    const size_t id = row * (size_t)rx + x;
    const size_t w = id >> 5;
    const unsigned off = (unsigned)(id & 31);
    uint32_t v = bits[w] >> off;
    if (off) v |= bits[w + 1] << (32 - off);
    const int valid = rx - x;
    if (valid < 32) v &= (1u << valid) - 1u;
    return v;
}

// first occupied x >= x0 of the row (INT_MAX: none); the warp looks at 1024 nodes per round
__device__ __forceinline__ int next_occupied(const uint32_t* __restrict__ bits, size_t row, int rx, int x0, int lane)
{
    for (int x = x0; x < rx; x += 1024) {
        const uint32_t v = row_window(bits, row, rx, x + 32 * lane);
        const unsigned m = __ballot_sync(0xffffffffu, v != 0u);
        if (m) {
            const int l = __ffs(m) - 1;
            const uint32_t vl = __shfl_sync(0xffffffffu, v, l);
            return x + 32 * l + __ffs(vl) - 1;
        }
    }
    return INT_MAX;
}

__global__ void __launch_bounds__(32 * kRowWarps) k_edt_rows(const uint32_t* __restrict__ bits, uint32_t* __restrict__ out, int rx, unsigned nrows)
{
    const int lane = threadIdx.x & 31;
    const unsigned row = blockIdx.x * kRowWarps + (threadIdx.x >> 5);
    if (row >= nrows) return;   // whole warps
    uint32_t* o = out + (size_t)row * rx;
    int left = -1;              // last occupied x before the current chunk (-1: none)
    int nxt = -1;               // first occupied x at or after the end of the current chunk (INT_MAX: none)
    for (int x0 = 0; x0 < rx; x0 += 32) {
        if (nxt < x0 + 32) nxt = next_occupied(bits, row, rx, x0 + 32, lane);   // warp-uniform; the searches cover disjoint ranges
        const uint32_t win = row_window(bits, row, rx, x0);
        const int x = x0 + lane;
        const uint32_t le = win & (0xffffffffu >> (31 - lane));
        const uint32_t ge = win & (0xffffffffu << lane);
        const int l = le ? x0 + 31 - __clz(le) : left;
        const int r = ge ? x0 + __ffs(ge) - 1 : nxt;
        unsigned d = 0xffffffffu;
        if (l >= 0) d = (unsigned)(x - l);
        if (r != INT_MAX) d = min(d, (unsigned)(r - x));
        if (x < rx) o[x] = d == 0xffffffffu ? kFar : d * d;
        if (win) left = x0 + 31 - __clz(win);
    }
}

__device__ __forceinline__ long long floor_div(long long a, long long b)   // b > 0
{
    return a >= 0 ? a / b : -((-a + b - 1) / b);
}

// One lane per x column: the lines of block (bx, by) are in[by*outer + u*stride + x], u < L, for x = bx*W + lane.
// stk: [L][W] words, (apex s) | (start t) << 16.
__global__ void k_edt_cols(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int rx, int L, size_t stride, size_t outer)
{
    extern __shared__ uint32_t stk[];
    const int W = blockDim.x, lane = threadIdx.x;
    const int x = blockIdx.x * W + lane;
    if (x >= rx) return;
    const uint32_t* f = in + (size_t)blockIdx.y * outer + x;
    uint32_t* o = out + (size_t)blockIdx.y * outer + x;
    uint32_t* st = stk + lane;

    // forward scan: the lower envelope of the finite parabolas (u - i)^2 + f(i)
    int q = -1;
    int ts = 0, tt = 0;          // top of the stack: apex, start
    long long tf = 0;            // f at the apex
    for (int u0 = 0; u0 < L; u0 += kColPrefetch) {
        uint32_t v[kColPrefetch];
#pragma unroll
        for (int k = 0; k < kColPrefetch; k++) v[k] = u0 + k < L ? __ldg(f + (size_t)(u0 + k) * stride) : kFar;
#pragma unroll
        for (int k = 0; k < kColPrefetch; k++) {
            if (v[k] == kFar) continue;
            const long long u = u0 + k, fu = v[k];
            while (q >= 0 && (long long)(tt - ts) * (tt - ts) + tf > (tt - u) * (tt - u) + fu) {
                if (--q >= 0) {
                    const uint32_t e = st[(size_t)q * W];
                    ts = (int)(e & 0xffffu); tt = (int)(e >> 16);
                    tf = __ldg(f + (size_t)ts * stride);
                }
            }
            if (q < 0) {
                q = 0; ts = (int)u; tt = 0; tf = fu;
                st[0] = (uint32_t)u;
            } else {
                const long long w = 1 + floor_div(u * u - (long long)ts * ts + fu - tf, 2 * (u - ts));
                if (w < L) {
                    q++; ts = (int)u; tt = (int)w; tf = fu;
                    st[(size_t)q * W] = (uint32_t)u | ((uint32_t)w << 16);
                }
            }
        }
    }
    // backward scan: every u takes the parabola whose segment holds it
    if (q < 0) {
        for (int u = 0; u < L; u++) o[(size_t)u * stride] = kFar;
        return;
    }
    for (int u = L - 1; u >= 0; u--) {
        const long long du = u - ts;
        o[(size_t)u * stride] = (uint32_t)(du * du + tf);
        if (u == tt && --q >= 0) {
            const uint32_t e = st[(size_t)q * W];
            ts = (int)(e & 0xffffu); tt = (int)(e >> 16);
            tf = __ldg(f + (size_t)ts * stride);
        }
    }
}

static int cols_pass(const uint32_t* in, uint32_t* out, int rx, int L, size_t stride, size_t outer, unsigned nouter, cudaStream_t s)
{
    const int W = (int)std::min<size_t>(32, kColSmemMax / ((size_t)L * sizeof(uint32_t)));   // >= 1: L <= 32768
    const size_t smem = (size_t)W * L * sizeof(uint32_t);
    WR_CUDA(cudaFuncSetAttribute(k_edt_cols, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kColSmemMax));
    dim3 grid((unsigned)((rx + W - 1) / W), nouter);
    k_edt_cols<<<grid, W, smem, s>>>(in, out, rx, L, stride, outer);
    WR_CUDA(cudaGetLastError());
    return WR_OK;
}

int grid_ensure_clearance(wr_grid* g)
{
    if (g->d_clear) return WR_OK;
    WR_REQUIRE(g->rx <= kMaxClearanceAxis && g->ry <= kMaxClearanceAxis && g->rz <= kMaxClearanceAxis, WR_ERR_INVALID,
               "clearance: grid axes longer than 32768 nodes are not supported");
    WR_CUDA(cudaSetDevice(g->device));
    cudaStream_t s = 0;
    uint32_t *field = nullptr, *tmp = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int rc = WR_OK;
    cudaError_t e = dmalloc(&field, g->N * sizeof(uint32_t), s);
    if (e == cudaSuccess) e = dmalloc(&tmp, g->N * sizeof(uint32_t), s);
    if (e == cudaSuccess) e = cudaEventCreate(&e0);
    if (e == cudaSuccess) e = cudaEventCreate(&e1);
    if (e == cudaSuccess) e = cudaEventRecord(e0, s);
    if (e == cudaSuccess) {
        const unsigned nrows = (unsigned)((size_t)g->ry * g->rz);
        k_edt_rows<<<(nrows + kRowWarps - 1) / kRowWarps, 32 * kRowWarps, 0, s>>>(g->d_bits, field, g->rx, nrows);
        e = cudaGetLastError();
    }
    const size_t rxy = (size_t)g->rx * g->ry;
    if (e == cudaSuccess) rc = cols_pass(field, tmp, g->rx, g->ry, g->rx, rxy, (unsigned)g->rz, s);   // along y, per z plane
    if (e == cudaSuccess && rc == WR_OK) rc = cols_pass(tmp, field, g->rx, g->rz, rxy, g->rx, (unsigned)g->ry, s);   // along z, per y
    if (e == cudaSuccess && rc == WR_OK) e = cudaEventRecord(e1, s);
    if (e == cudaSuccess && rc == WR_OK) e = cudaEventSynchronize(e1);
    if (e == cudaSuccess && rc == WR_OK) e = cudaEventElapsedTime(&g->clear_ms, e0, e1);
    pool_free(tmp, s);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (e != cudaSuccess || rc != WR_OK) {
        pool_free(field, s);
        if (rc != WR_OK) return rc;
        set_error("clearance field: %s", cudaGetErrorString(e));
        return WR_ERR_CUDA;
    }
    g->d_clear = field;
    return WR_OK;
}

// ---- point queries -------------------------------------------------------------------------------------------------
struct AxisTable {
    const float* c;
    int n;
    int sorted;   // host-checked: c is non-decreasing (binary search allowed)
};

// argmin_i |p - c[i]| in double, lowest index on ties (a NaN distance counts as the minimum, as numpy's argmin has it)
__device__ int nearest_on_axis(const AxisTable a, float p)
{
    const double pd = p;
    auto dist = [&](int i) { return fabs(pd - (double)a.c[i]); };
    if (!a.sorted) {
        int best = 0;
        double bd = dist(0);
        for (int i = 1; i < a.n && !isnan(bd); i++) {
            const double d = dist(i);
            if (d < bd || isnan(d)) { best = i; bd = d; }
        }
        return best;
    }
    // non-decreasing table: the distance does not increase up to hi-1 and does not decrease from hi = first c[i] >= p
    int lo = 0, hi = a.n;
    while (lo < hi) {
        const int m = (lo + hi) >> 1;
        if (a.c[m] >= p) hi = m; else lo = m + 1;
    }
    if (hi == 0) return 0;
    // left candidate: the first index whose distance equals that of hi-1 (duplicate planes, ties the double rounding made)
    const double dl = dist(hi - 1);
    int a0 = 0, a1 = hi - 1;
    while (a0 < a1) {
        const int m = (a0 + a1) >> 1;
        if (dist(m) <= dl) a1 = m; else a0 = m + 1;
    }
    if (hi == a.n) return a0;
    return dl <= dist(hi) ? a0 : hi;
}

__global__ void k_clearance_at(const float* __restrict__ pts, int npoints, AxisTable tx, AxisTable ty, AxisTable tz,
                               const uint32_t* __restrict__ field, long long* __restrict__ ids, uint32_t* __restrict__ d2)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npoints) return;
    const float px = pts[3 * i], py = pts[3 * i + 1], pz = pts[3 * i + 2];
    if (!(isfinite(px) && isfinite(py) && isfinite(pz))) {
        ids[i] = -1; d2[i] = kFar;
        return;
    }
    const int x = nearest_on_axis(tx, px), y = nearest_on_axis(ty, py), z = nearest_on_axis(tz, pz);
    const long long id = ((long long)z * ty.n + y) * tx.n + x;
    ids[i] = id;
    d2[i] = field[id];
}

// ---- inflation -----------------------------------------------------------------------------------------------------
__global__ void k_inflate(const uint32_t* __restrict__ field, uint32_t r2, uint32_t* __restrict__ bits, unsigned long long N, unsigned long long* occupied)
{
    __shared__ unsigned cta_occ;
    if (threadIdx.x == 0) cta_occ = 0;
    __syncthreads();
    const unsigned long long id = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool occ = id < N && field[id] <= r2;
    const unsigned m = __ballot_sync(0xffffffffu, occ);
    if ((threadIdx.x & 31) == 0) {
        if (id < N) bits[id >> 5] = m;
        if (m) atomicAdd(&cta_occ, (unsigned)__popc(m));
    }
    __syncthreads();
    if (threadIdx.x == 0 && cta_occ) atomicAdd(occupied, (unsigned long long)cta_occ);
}

static bool non_decreasing(const std::vector<float>& c)
{
    for (size_t i = 1; i < c.size(); i++)
        if (!(c[i - 1] <= c[i])) return false;
    return true;
}

}  // namespace wr

using namespace wr;

extern "C" int wr_grid_clearance(wr_grid* g, uint32_t* d2, size_t n)
{
    WR_REQUIRE(g && d2, WR_ERR_INVALID, "wr_grid_clearance: null");
    WR_REQUIRE(n >= g->N, WR_ERR_CAPACITY, "wr_grid_clearance: buffer too small");
    int rc = grid_ensure_clearance(g);
    if (rc != WR_OK) return rc;
    WR_CUDA(cudaMemcpy(d2, g->d_clear, g->N * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return WR_OK;
}

extern "C" int wr_grid_clearance_at(wr_grid* g, const float* pts_xyz, int npoints, int64_t* ids, uint32_t* d2)
{
    WR_REQUIRE(g && pts_xyz && npoints >= 0, WR_ERR_INVALID, "wr_grid_clearance_at: bad argument");
    if (npoints == 0) return WR_OK;
    int rc = grid_ensure_clearance(g);
    if (rc != WR_OK) return rc;
    cudaStream_t s = 0;
    float* d_pts = nullptr;
    long long* d_ids = nullptr;
    uint32_t* d_d2 = nullptr;
    cudaError_t e = dmalloc(&d_pts, (size_t)npoints * 3 * sizeof(float), s);
    if (e == cudaSuccess) e = dmalloc(&d_ids, (size_t)npoints * sizeof(long long), s);
    if (e == cudaSuccess) e = dmalloc(&d_d2, (size_t)npoints * sizeof(uint32_t), s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_pts, pts_xyz, (size_t)npoints * 3 * sizeof(float), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
        AxisTable tx{g->d_coords, g->rx, non_decreasing(g->h_xs)};
        AxisTable ty{g->d_coords + g->rx, g->ry, non_decreasing(g->h_ys)};
        AxisTable tz{g->d_coords + g->rx + g->ry, g->rz, non_decreasing(g->h_zs)};
        k_clearance_at<<<(unsigned)((npoints + 255) / 256), 256, 0, s>>>(d_pts, npoints, tx, ty, tz, g->d_clear, d_ids, d_d2);
        e = cudaGetLastError();
    }
    static_assert(sizeof(long long) == sizeof(int64_t), "ids are copied as int64");
    if (e == cudaSuccess && ids) e = cudaMemcpyAsync(ids, d_ids, (size_t)npoints * sizeof(int64_t), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && d2) e = cudaMemcpyAsync(d2, d_d2, (size_t)npoints * sizeof(uint32_t), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    pool_free(d_pts, s); pool_free(d_ids, s); pool_free(d_d2, s);
    if (e != cudaSuccess) { set_error("wr_grid_clearance_at: %s", cudaGetErrorString(e)); return WR_ERR_CUDA; }
    return WR_OK;
}

extern "C" int wr_grid_inflate(wr_grid* g, uint32_t r2, wr_grid** out)
{
    WR_REQUIRE(g && out, WR_ERR_INVALID, "wr_grid_inflate: null");
    *out = nullptr;
    int rc = grid_ensure_clearance(g);
    if (rc != WR_OK) return rc;
    wr_grid* n = new wr_grid();
    n->rx = g->rx; n->ry = g->ry; n->rz = g->rz; n->wall = g->wall; n->precision = g->precision;
    std::copy(g->gmin, g->gmin + 3, n->gmin); std::copy(g->gmax, g->gmax + 3, n->gmax);
    n->h_xs = g->h_xs; n->h_ys = g->h_ys; n->h_zs = g->h_zs;
    rc = grid_alloc_common(n);
    if (rc != WR_OK) { wr_grid_destroy(n); return rc; }
    unsigned long long* d_occ = nullptr;
    unsigned long long occ = 0;
    cudaError_t e = dmalloc(&d_occ, sizeof(unsigned long long), 0);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_occ, 0, sizeof(unsigned long long), 0);
    if (e == cudaSuccess) {
        k_inflate<<<(unsigned)((n->N + 255) / 256), 256>>>(g->d_clear, r2, n->d_bits, n->N, d_occ);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(&occ, d_occ, sizeof occ, cudaMemcpyDeviceToHost);
    pool_free(d_occ, 0);
    if (e != cudaSuccess) { set_error("wr_grid_inflate: %s", cudaGetErrorString(e)); wr_grid_destroy(n); return WR_ERR_CUDA; }
    n->occupied = occ;
    *out = n;
    return WR_OK;
}

extern "C" int wr_grid_clearance_ms(const wr_grid* g, float* ms)
{
    WR_REQUIRE(g && ms, WR_ERR_INVALID, "wr_grid_clearance_ms: null");
    *ms = g->clear_ms;
    return WR_OK;
}
