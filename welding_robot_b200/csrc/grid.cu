// K1 — voxeliser: triangles -> bit-packed occupancy grid, plus the per-node open-neighbour
// mask the ant walk reads.  Replaces GridMap<T>::creatGridMap (core/model_grid_map.hpp:151-273).
//
// Design (B200): node-parallel, atomics-free.  Every thread owns one 32-bit word of the
// occupancy grid (32 consecutive node ids), every CTA a slab of 8192 ids.  The triangle list
// is pre-reduced on the host to a 10-array SoA {n.xyz, D, box min.xyz, box max.xyz} (48 B of
// file data per triangle -> 40 B), streamed through shared memory in 512-triangle chunks
// with 1-D TMA bulk copies (cp.async.bulk + mbarrier, double buffered).  A CTA first culls a
// chunk against the slab's coordinate box (one triangle per thread, warp-aggregated
// compaction), then all threads evaluate the surviving triangles with the reference's exact
// predicate and operation order.  The reference tests every triangle against every node
// (O(T*N)); the cull only removes pairs whose box test (:258-260) cannot pass, so the result
// is bit-identical and independent of scheduling (pure OR).
#include <math.h>

#include <algorithm>

#include "tma.cuh"
#include "wr_internal.cuh"

namespace wr {

constexpr int kVoxThreads = 256;
constexpr int kVoxChunk = 512;      // triangles per TMA stage
constexpr int kVoxArrays = 10;      // nx ny nz D minx miny minz maxx maxy maxz
constexpr int kVoxNodesPerCta = kVoxThreads * 32;

struct VoxArgs {
    const float* soa;   // kVoxArrays arrays of Tpad floats
    int Tpad, nchunks;
    int rx, ry, rz;
    unsigned long long N;
    const float* coords;  // xs | ys | zs
    float thr;            // smallest float >= 1.2*(double)precision  (:256 compares in double)
    uint32_t* bits;
    unsigned long long* counters;  // [0] occupied [1] predicate evaluations
};

__device__ __forceinline__ float warp_min(float v)
{
    for (int o = 16; o; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_max(float v)
{
    for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__global__ void __launch_bounds__(kVoxThreads) k_voxelize(VoxArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* stage = reinterpret_cast<float*>(smem_raw);                           // [2][kVoxArrays][kVoxChunk]
    uint64_t* bar = reinterpret_cast<uint64_t*>(stage + 2 * kVoxArrays * kVoxChunk);  // [2]
    int* list = reinterpret_cast<int*>(bar + 2);                                 // [kVoxChunk]
    int* nlist = list + kVoxChunk;                                               // [2] (+2 pad), one counter per stage
    float* box = reinterpret_cast<float*>(nlist + 4);                            // [6][8 warps]
    float* xs = box + 6 * 8;
    float* ys = xs + a.rx;
    float* zs = ys + a.ry;

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int rx = a.rx, ry = a.ry;

    for (int i = tid; i < a.rx + a.ry + a.rz; i += kVoxThreads) xs[i] = a.coords[i];
    if (tid == 0) {
        tma::mbar_init(&bar[0], 1);
        tma::mbar_init(&bar[1], 1);
        tma::fence_barrier_init();
        nlist[0] = 0; nlist[1] = 0;
    }
    __syncthreads();

    constexpr uint32_t kStageBytes = kVoxArrays * kVoxChunk * sizeof(float);
    auto issue = [&](int chunk) {  // thread 0 only
        int s = chunk & 1;
        tma::mbar_arrive_expect_tx(&bar[s], kStageBytes);
#pragma unroll
        for (int f = 0; f < kVoxArrays; f++)
            tma::bulk_g2s(stage + (s * kVoxArrays + f) * kVoxChunk, a.soa + (size_t)f * a.Tpad + (size_t)chunk * kVoxChunk,
                          kVoxChunk * sizeof(float), &bar[s]);
    };
    if (tid == 0) issue(0);

    // ---- this thread's 32 nodes and their coordinate box --------------------------------
    const unsigned long long base = (unsigned long long)blockIdx.x * kVoxNodesPerCta + (unsigned long long)tid * 32;
    int cnt = 0;
    if (base < a.N) cnt = (int)min((unsigned long long)32, a.N - base);
    const unsigned long long rxy = (unsigned long long)rx * ry;
    int z0 = 0, y0 = 0, x0 = 0;
    if (cnt) {
        z0 = (int)(base / rxy);
        unsigned r = (unsigned)(base % rxy);
        y0 = r / rx; x0 = r % rx;
    }
    float tminx = INFINITY, tmaxx = -INFINITY, tminy = INFINITY, tmaxy = -INFINITY, tminz = INFINITY, tmaxz = -INFINITY;
    {
        int x = x0, y = y0, z = z0;
        for (int j = 0; j < cnt; j++) {
            float px = xs[x], py = ys[y], pz = zs[z];
            tminx = fminf(tminx, px); tmaxx = fmaxf(tmaxx, px);
            tminy = fminf(tminy, py); tmaxy = fmaxf(tmaxy, py);
            tminz = fminf(tminz, pz); tmaxz = fmaxf(tmaxz, pz);
            if (++x == rx) { x = 0; if (++y == ry) { y = 0; ++z; } }
        }
    }
    {   // CTA box = union of thread boxes
        float v0 = warp_min(tminx), v1 = warp_max(tmaxx), v2 = warp_min(tminy), v3 = warp_max(tmaxy), v4 = warp_min(tminz), v5 = warp_max(tmaxz);
        if (lane == 0) { box[0 * 8 + warp] = v0; box[1 * 8 + warp] = v1; box[2 * 8 + warp] = v2; box[3 * 8 + warp] = v3; box[4 * 8 + warp] = v4; box[5 * 8 + warp] = v5; }
    }
    __syncthreads();
    float cminx = box[0], cmaxx = box[8], cminy = box[16], cmaxy = box[24], cminz = box[32], cmaxz = box[40];
    for (int w = 1; w < 8; w++) {
        cminx = fminf(cminx, box[w]); cmaxx = fmaxf(cmaxx, box[8 + w]);
        cminy = fminf(cminy, box[16 + w]); cmaxy = fmaxf(cmaxy, box[24 + w]);
        cminz = fminf(cminz, box[32 + w]); cmaxz = fmaxf(cmaxz, box[40 + w]);
    }

    uint32_t word = 0;
    unsigned long long ntests = 0;
    const float thr = a.thr;

    for (int c = 0; c < a.nchunks; c++) {
        const int s = c & 1;
        if (tid == 0 && c + 1 < a.nchunks) issue(c + 1);  // stage (c+1)&1 was released by the barrier ending iteration c-1
        tma::mbar_wait(&bar[s], (c >> 1) & 1);
        const float* T = stage + s * kVoxArrays * kVoxChunk;
        // ---- cull this chunk against the CTA box -----------------------------------------
#pragma unroll
        for (int q = 0; q < kVoxChunk / kVoxThreads; q++) {
            int t = q * kVoxThreads + tid;
            bool keep = T[4 * kVoxChunk + t] <= cmaxx && cminx <= T[7 * kVoxChunk + t] &&
                        T[5 * kVoxChunk + t] <= cmaxy && cminy <= T[8 * kVoxChunk + t] &&
                        T[6 * kVoxChunk + t] <= cmaxz && cminz <= T[9 * kVoxChunk + t];
            unsigned m = __ballot_sync(0xffffffffu, keep);
            int pos = 0;
            if (lane == 0 && m) pos = atomicAdd(&nlist[s], __popc(m));
            pos = __shfl_sync(0xffffffffu, pos, 0);
            if (keep) list[pos + __popc(m & ((1u << lane) - 1))] = t;
        }
        __syncthreads();
        const int ns = nlist[s];
        if (tid == 0) nlist[s ^ 1] = 0;  // last read before the barrier that ended iteration c-1
        // ---- exact predicate on the survivors (model_grid_map.hpp:252-262) ----------------
        if (cnt) {
            for (int i = 0; i < ns; i++) {
                const int t = list[i];
                const float mnx = T[4 * kVoxChunk + t], mny = T[5 * kVoxChunk + t], mnz = T[6 * kVoxChunk + t];
                const float mxx = T[7 * kVoxChunk + t], mxy = T[8 * kVoxChunk + t], mxz = T[9 * kVoxChunk + t];
                if (!(mnx <= tmaxx && tminx <= mxx && mny <= tmaxy && tminy <= mxy && mnz <= tmaxz && tminz <= mxz)) continue;
                const float nx = T[t], ny = T[kVoxChunk + t], nz = T[2 * kVoxChunk + t], D = T[3 * kVoxChunk + t];
                int x = x0, y = y0, z = z0;
                float py = ys[y], pz = zs[z];
                bool row_in = mny <= py && py <= mxy && mnz <= pz && pz <= mxz;
                float pyny = __fmul_rn(py, ny), pznz = __fmul_rn(pz, nz);
                for (int j = 0; j < cnt; j++) {
                    float px = xs[x];
                    if (row_in && mnx <= px && px <= mxx) {
                        // distance = px*nx + py*ny + pz*nz + D, left to right, no contraction
                        float d = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(px, nx), pyny), pznz), D);
                        ntests++;
                        if (fabsf(d) < thr) word |= 1u << j;
                    }
                    if (++x == rx) {
                        x = 0;
                        if (++y == ry) { y = 0; ++z; }
                        if (j + 1 < cnt) {
                            py = ys[y]; pz = zs[z];
                            row_in = mny <= py && py <= mxy && mnz <= pz && pz <= mxz;
                            pyny = __fmul_rn(py, ny); pznz = __fmul_rn(pz, nz);
                        }
                    }
                }
            }
        }
        __syncthreads();  // `list` and stage s are free again
    }
    if (cnt) a.bits[base >> 5] = word;
    // counters
    unsigned occ = __popc(word);
    for (int o = 16; o; o >>= 1) {
        occ += __shfl_xor_sync(0xffffffffu, occ, o);
        ntests += __shfl_xor_sync(0xffffffffu, ntests, o);
    }
    if (lane == 0) {
        if (occ) atomicAdd(&a.counters[0], (unsigned long long)occ);
        if (ntests) atomicAdd(&a.counters[1], ntests);
    }
}

// Per-node open mask for the 6-neighbourhood in the reference's slot order
// [0]=-z [1]=-y [2]=-x [3]=+x [4]=+y [5]=+z (ACSRank_3D.hpp:355-359): bit k set <=> the
// neighbour exists (in bounds, :391-393) and is free (:148).
__global__ void k_open6(const uint32_t* __restrict__ bits, uint8_t* __restrict__ open6, int rx, int ry, int rz, unsigned long long N)
{
    unsigned long long id = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= N) return;
    const unsigned long long rxy = (unsigned long long)rx * ry;
    int z = (int)(id / rxy);
    unsigned r = (unsigned)(id % rxy);
    int y = r / rx, x = r % rx;
    auto is_free = [&](unsigned long long n) { return !((bits[n >> 5] >> (n & 31)) & 1u); };
    unsigned m = 0;
    if (z > 0 && is_free(id - rxy)) m |= 1u;
    if (y > 0 && is_free(id - rx)) m |= 2u;
    if (x > 0 && is_free(id - 1)) m |= 4u;
    if (x + 1 < rx && is_free(id + 1)) m |= 8u;
    if (y + 1 < ry && is_free(id + rx)) m |= 16u;
    if (z + 1 < rz && is_free(id + rxy)) m |= 32u;
    open6[id] = (uint8_t)m;
}

__global__ void k_pack_isfree(const uint8_t* __restrict__ isfree, uint32_t* __restrict__ bits, unsigned long long N, unsigned long long* occupied)
{
    __shared__ unsigned cta_occ;
    if (threadIdx.x == 0) cta_occ = 0;
    __syncthreads();
    unsigned long long id = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    bool occ = id < N && isfree[id] == 0;
    unsigned m = __ballot_sync(0xffffffffu, occ);
    if ((threadIdx.x & 31) == 0) {
        if (id < N) bits[id >> 5] = m;
        if (m) atomicAdd(&cta_occ, (unsigned)__popc(m));
    }
    __syncthreads();
    if (threadIdx.x == 0 && cta_occ) atomicAdd(occupied, (unsigned long long)cta_occ);
}
__global__ void k_unpack_isfree(const uint32_t* __restrict__ bits, uint8_t* __restrict__ isfree, unsigned long long N)
{
    unsigned long long id = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id < N) isfree[id] = ((bits[id >> 5] >> (id & 31)) & 1u) ? 0 : 1;
}

static float axis_coord(int i, int range, int wall, float mn, float mx, float precision)
{   // model_grid_map.hpp:204-205: three branches; the max-side wall restarts from max, so the
    // lattice is irregular there (possibly a duplicate plane) — kept on purpose (SURVEY.md §0.5)
    return i < wall ? mn - (wall - i) * precision : (i >= (range - wall) ? mx + (i - range + wall) * precision : mn + (i - wall) * precision);
}

int grid_alloc_common(wr_grid* g)
{
    WR_CUDA(cudaGetDevice(&g->device));
    g->N = (size_t)g->rx * g->ry * g->rz;
    g->nwords = (g->N + 31) / 32;
    size_t nc = (size_t)g->rx + g->ry + g->rz;
    WR_CUDA(dmalloc(&g->d_coords, nc * sizeof(float), 0));
    std::vector<float> c(nc);
    std::copy(g->h_xs.begin(), g->h_xs.end(), c.begin());
    std::copy(g->h_ys.begin(), g->h_ys.end(), c.begin() + g->rx);
    std::copy(g->h_zs.begin(), g->h_zs.end(), c.begin() + g->rx + g->ry);
    WR_CUDA(cudaMemcpy(g->d_coords, c.data(), nc * sizeof(float), cudaMemcpyHostToDevice));
    WR_CUDA(dmalloc(&g->d_bits, (g->nwords + 4) * sizeof(uint32_t), 0));
    WR_CUDA(cudaMemset(g->d_bits, 0, (g->nwords + 4) * sizeof(uint32_t)));
    return WR_OK;
}

int grid_ensure_open6(wr_grid* g, cudaStream_t s)
{
    if (g->d_open6) return WR_OK;
    WR_CUDA(dmalloc(&g->d_open6, g->N, s));
    unsigned blocks = (unsigned)((g->N + 255) / 256);
    k_open6<<<blocks, 256, 0, s>>>(g->d_bits, g->d_open6, g->rx, g->ry, g->rz, g->N);
    WR_CUDA(cudaGetLastError());
    return WR_OK;
}

int grid_ensure_host_bits(wr_grid* g)
{
    if (!g->h_bits.empty()) return WR_OK;
    g->h_bits.resize(g->nwords);
    WR_CUDA(cudaMemcpy(g->h_bits.data(), g->d_bits, g->nwords * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return WR_OK;
}

}  // namespace wr

using namespace wr;

extern "C" int wr_grid_create_from_triangles(const float* t12, int ntri, float precision, int wall, wr_grid** out)
{
    WR_REQUIRE(t12 && out && ntri > 0 && wall >= 0 && precision > 0, WR_ERR_INVALID, "wr_grid_create_from_triangles: bad argument");
    *out = nullptr;
    wr_grid* g = new wr_grid();
    g->precision = precision; g->wall = wall;
    // global box, model_grid_map.hpp:165-181
    float min_x = t12[3], min_y = t12[4], min_z = t12[5];
    float max_x = min_x, max_y = min_y, max_z = min_z;
    for (int t = 0; t < ntri; t++)
        for (int i = 0; i < 3; i++) {
            const float* v = t12 + 12 * (size_t)t + 3 + 3 * i;
            max_x = v[0] > max_x ? v[0] : max_x; max_y = v[1] > max_y ? v[1] : max_y; max_z = v[2] > max_z ? v[2] : max_z;
            min_x = v[0] < min_x ? v[0] : min_x; min_y = v[1] < min_y ? v[1] : min_y; min_z = v[2] < min_z ? v[2] : min_z;
        }
    g->gmin[0] = min_x; g->gmin[1] = min_y; g->gmin[2] = min_z;
    g->gmax[0] = max_x; g->gmax[1] = max_y; g->gmax[2] = max_z;
    // ranges, :198-200
    double ex = (double)((max_x - min_x) / precision), ey = (double)((max_y - min_y) / precision), ez = (double)((max_z - min_z) / precision);
    if (!(ex < 1e6 && ey < 1e6 && ez < 1e6)) { delete g; set_error("grid extent too large for precision %g", precision); return WR_ERR_INVALID; }
    g->rx = (int)((max_x - min_x) / precision) + 1 + 2 * wall;
    g->ry = (int)((max_y - min_y) / precision) + 1 + 2 * wall;
    g->rz = (int)((max_z - min_z) / precision) + 1 + 2 * wall;
    if ((double)g->rx * g->ry * g->rz >= 2147483648.0) { delete g; set_error("grid has >= 2^31 nodes"); return WR_ERR_INVALID; }
    g->h_xs.resize(g->rx); g->h_ys.resize(g->ry); g->h_zs.resize(g->rz);
    for (int x = 0; x < g->rx; x++) g->h_xs[x] = axis_coord(x, g->rx, wall, min_x, max_x, precision);
    for (int y = 0; y < g->ry; y++) g->h_ys[y] = axis_coord(y, g->ry, wall, min_y, max_y, precision);
    for (int z = 0; z < g->rz; z++) g->h_zs[z] = axis_coord(z, g->rz, wall, min_z, max_z, precision);
    int st = grid_alloc_common(g);
    if (st != WR_OK) { wr_grid_destroy(g); return st; }

    // per-triangle plane + padded box, :224-248 (host: O(T), same float expressions)
    const int Tpad = (ntri + kVoxChunk - 1) / kVoxChunk * kVoxChunk;
    std::vector<float> soa((size_t)kVoxArrays * Tpad);
    for (int t = 0; t < Tpad; t++) {
        float v[kVoxArrays];
        if (t < ntri) {
            const float* n = t12 + 12 * (size_t)t;
            const float* v0 = n + 3;
            float D = -(v0[0] * n[0] + v0[1] * n[1] + v0[2] * n[2]);
            float mnx = v0[0], mny = v0[1], mnz = v0[2], mxx = mnx, mxy = mny, mxz = mnz;
            for (int i = 0; i < 3; i++) {
                const float* p = n + 3 + 3 * i;
                mxx = p[0] > mxx ? p[0] : mxx; mxy = p[1] > mxy ? p[1] : mxy; mxz = p[2] > mxz ? p[2] : mxz;
                mnx = p[0] < mnx ? p[0] : mnx; mny = p[1] < mny ? p[1] : mny; mnz = p[2] < mnz ? p[2] : mnz;
            }
            mnx -= precision; mny -= precision; mnz -= precision;
            mxx += precision; mxy += precision; mxz += precision;
            v[0] = n[0]; v[1] = n[1]; v[2] = n[2]; v[3] = D; v[4] = mnx; v[5] = mny; v[6] = mnz; v[7] = mxx; v[8] = mxy; v[9] = mxz;
        } else {  // padding: empty box, never survives the cull
            v[0] = v[1] = v[2] = v[3] = 0; v[4] = v[5] = v[6] = INFINITY; v[7] = v[8] = v[9] = -INFINITY;
        }
        for (int f = 0; f < kVoxArrays; f++) soa[(size_t)f * Tpad + t] = v[f];
    }
    // |distance| < 1.2*precision is evaluated in double (:256); for a float lhs that is the same
    // as comparing against the smallest float >= the double threshold.
    double thr_d = 1.2 * (double)precision;
    float thr = (float)thr_d;
    if ((double)thr < thr_d) thr = nextafterf(thr, INFINITY);

    float* d_soa = nullptr;
    unsigned long long* d_cnt = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    auto fail = [&](int code) { pool_free(d_soa, 0); pool_free(d_cnt, 0); if (e0) cudaEventDestroy(e0); if (e1) cudaEventDestroy(e1); wr_grid_destroy(g); return code; };
#define WR_CUDA_F(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { set_error("%s failed: %s", #expr, cudaGetErrorString(_e)); return fail(WR_ERR_CUDA); } } while (0)
    WR_CUDA_F(dmalloc(&d_soa, soa.size() * sizeof(float), 0));
    WR_CUDA_F(cudaMemcpy(d_soa, soa.data(), soa.size() * sizeof(float), cudaMemcpyHostToDevice));
    WR_CUDA_F(dmalloc(&d_cnt, 2 * sizeof(unsigned long long), 0));
    WR_CUDA_F(cudaMemset(d_cnt, 0, 2 * sizeof(unsigned long long)));
    VoxArgs a;
    a.soa = d_soa; a.Tpad = Tpad; a.nchunks = Tpad / kVoxChunk; a.rx = g->rx; a.ry = g->ry; a.rz = g->rz; a.N = g->N;
    a.coords = g->d_coords; a.thr = thr; a.bits = g->d_bits; a.counters = d_cnt;
    size_t smem = 2 * kVoxArrays * kVoxChunk * sizeof(float) + 2 * sizeof(uint64_t) + (kVoxChunk + 4) * sizeof(int) + 48 * sizeof(float) +
                  ((size_t)g->rx + g->ry + g->rz) * sizeof(float);
    if (smem > 227 * 1024) { set_error("grid axes too long for the voxeliser's shared-memory coordinate tables"); return fail(WR_ERR_INVALID); }
    WR_CUDA_F(cudaFuncSetAttribute(k_voxelize, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    unsigned blocks = (unsigned)((g->N + kVoxNodesPerCta - 1) / kVoxNodesPerCta);
    WR_CUDA_F(cudaEventCreate(&e0));
    WR_CUDA_F(cudaEventCreate(&e1));
    WR_CUDA_F(cudaEventRecord(e0, 0));
    k_voxelize<<<blocks, kVoxThreads, smem, 0>>>(a);
    WR_CUDA_F(cudaGetLastError());
    WR_CUDA_F(cudaEventRecord(e1, 0));
    WR_CUDA_F(cudaEventSynchronize(e1));
    WR_CUDA_F(cudaEventElapsedTime(&g->vox_ms, e0, e1));
    unsigned long long h_cnt[2];
    WR_CUDA_F(cudaMemcpy(h_cnt, d_cnt, sizeof h_cnt, cudaMemcpyDeviceToHost));
#undef WR_CUDA_F
    g->occupied = h_cnt[0]; g->tests = h_cnt[1];
    pool_free(d_soa, 0); pool_free(d_cnt, 0); cudaEventDestroy(e0); cudaEventDestroy(e1);
    *out = g;
    return WR_OK;
}

extern "C" int wr_grid_create_from_occupancy(const uint8_t* isfree, int rx, int ry, int rz, const float* xs, const float* ys,
                                             const float* zs, float precision, wr_grid** out)
{
    WR_REQUIRE(isfree && out && xs && ys && zs && rx > 0 && ry > 0 && rz > 0, WR_ERR_INVALID, "wr_grid_create_from_occupancy: bad argument");
    WR_REQUIRE((double)rx * ry * rz < 2147483648.0, WR_ERR_INVALID, "grid has >= 2^31 nodes");
    *out = nullptr;
    wr_grid* g = new wr_grid();
    g->rx = rx; g->ry = ry; g->rz = rz; g->precision = precision; g->wall = 0;
    g->h_xs.assign(xs, xs + rx); g->h_ys.assign(ys, ys + ry); g->h_zs.assign(zs, zs + rz);
    int st = grid_alloc_common(g);
    if (st != WR_OK) { wr_grid_destroy(g); return st; }
    uint8_t* d_free = nullptr;
    unsigned long long* d_occ = nullptr;
    unsigned long long occ = 0;
    cudaError_t e = dmalloc(&d_free, g->N, 0);
    if (e == cudaSuccess) e = dmalloc(&d_occ, sizeof(unsigned long long), 0);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_occ, 0, sizeof(unsigned long long), 0);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_free, isfree, g->N, cudaMemcpyHostToDevice, 0);
    if (e == cudaSuccess) {
        unsigned blocks = (unsigned)((g->N + 255) / 256);
        k_pack_isfree<<<blocks, 256>>>(d_free, g->d_bits, g->N, d_occ);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpy(&occ, d_occ, sizeof occ, cudaMemcpyDeviceToHost);   // also orders the upload before the caller reuses `isfree`
    }
    pool_free(d_free, 0); pool_free(d_occ, 0);
    if (e != cudaSuccess) { set_error("occupancy upload failed: %s", cudaGetErrorString(e)); wr_grid_destroy(g); return WR_ERR_CUDA; }
    g->occupied = occ;
    *out = g;
    return WR_OK;
}

extern "C" int wr_grid_destroy(wr_grid* g)
{
    if (!g) return WR_OK;
    pool_free(g->d_coords, 0); pool_free(g->d_bits, 0); pool_free(g->d_open6, 0); pool_free(g->d_clear, 0);
    delete g;
    return WR_OK;
}
extern "C" int wr_grid_dims(const wr_grid* g, int d[3])
{
    WR_REQUIRE(g && d, WR_ERR_INVALID, "wr_grid_dims: null");
    d[0] = g->rx; d[1] = g->ry; d[2] = g->rz;
    return WR_OK;
}
extern "C" int wr_grid_precision(const wr_grid* g, float* precision, int* wall)
{
    WR_REQUIRE(g, WR_ERR_INVALID, "wr_grid_precision: null");
    if (precision) *precision = g->precision;
    if (wall) *wall = g->wall;
    return WR_OK;
}
extern "C" int wr_grid_bbox(const wr_grid* g, float mn[3], float mx[3])
{
    WR_REQUIRE(g && mn && mx, WR_ERR_INVALID, "wr_grid_bbox: null");
    for (int k = 0; k < 3; k++) { mn[k] = g->gmin[k]; mx[k] = g->gmax[k]; }
    return WR_OK;
}
extern "C" int wr_grid_coords(const wr_grid* g, float* xs, float* ys, float* zs)
{
    WR_REQUIRE(g && xs && ys && zs, WR_ERR_INVALID, "wr_grid_coords: null");
    std::copy(g->h_xs.begin(), g->h_xs.end(), xs);
    std::copy(g->h_ys.begin(), g->h_ys.end(), ys);
    std::copy(g->h_zs.begin(), g->h_zs.end(), zs);
    return WR_OK;
}
extern "C" int wr_grid_download_bits(const wr_grid* g, uint32_t* bits, size_t nwords)
{
    WR_REQUIRE(g && bits, WR_ERR_INVALID, "wr_grid_download_bits: null");
    WR_REQUIRE(nwords >= g->nwords, WR_ERR_CAPACITY, "wr_grid_download_bits: buffer too small");
    WR_CUDA(cudaMemcpy(bits, g->d_bits, g->nwords * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return WR_OK;
}
extern "C" int wr_grid_download_isfree(const wr_grid* g, uint8_t* isfree, size_t n)
{
    WR_REQUIRE(g && isfree, WR_ERR_INVALID, "wr_grid_download_isfree: null");
    WR_REQUIRE(n >= g->N, WR_ERR_CAPACITY, "wr_grid_download_isfree: buffer too small");
    uint8_t* d = nullptr;
    WR_CUDA(dmalloc(&d, g->N, 0));
    k_unpack_isfree<<<(unsigned)((g->N + 255) / 256), 256>>>(g->d_bits, d, g->N);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpy(isfree, d, g->N, cudaMemcpyDeviceToHost);
    pool_free(d, 0);
    if (e != cudaSuccess) { set_error("wr_grid_download_isfree: %s", cudaGetErrorString(e)); return WR_ERR_CUDA; }
    return WR_OK;
}
extern "C" int wr_grid_stats(const wr_grid* g, uint64_t* occupied, uint64_t* tests, float* kernel_ms)
{
    WR_REQUIRE(g, WR_ERR_INVALID, "wr_grid_stats: null");
    if (occupied) *occupied = g->occupied;
    if (tests) *tests = g->tests;
    if (kernel_ms) *kernel_ms = g->vox_ms;
    return WR_OK;
}
