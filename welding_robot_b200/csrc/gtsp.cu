// K4 — batched seam-ordering ant colony (ACS_GTSP, core/ACS_GTSP.hpp): B independent colonies on
// one distance matrix, colony b drawing from Philox stream (seed, colony_first + b).
//
// One CTA owns one colony for the whole call (no grid-wide sync, colonies never interact);
// thread k is ant k (colony size = city count, ACS_GTSP.hpp:192).  All arithmetic is FP64 in the
// reference's order: the roulette sums `info` over the unvisited cities in ASCENDING city order
// (:129-141), a 255-term dependent DADD chain per ant and step that cannot be re-associated, so the
// parallelism is ants x colonies, not cities.
//
// Memory plan.  info = pheromone * heuristic^6 is symmetric (pheromone is kept symmetric by :183,
// the heuristic by construction), so ant k standing on city r reads info[c][r] instead of
// info[r][c]: all ants of the colony then walk the SAME rows c = 0..N-1 in lockstep, and a row
// chunk (8 rows, 16 KB) is staged ONCE per CTA in shared memory with a 1-D TMA bulk copy
// (double-buffered, mbarrier completion) instead of once per ant.  The reference scans the row
// twice (total, then prefix until >= rnd*total); here the running sum is check-pointed every 16
// cities in shared memory during the single streaming pass, and the second scan re-adds only the
// 16 cities of the interval that contains the threshold, starting from the exact check-pointed
// partial sum — the same additions in the same order, 1/16 of the traffic.
// Per colony-iteration the matrix (N^2 doubles, 512 KB at N = 256) is streamed N times from L2/HBM: that
// stream (134 GB per iteration of 1024 colonies) is what bounds the kernel — measured 34.7k colony-iterations/s
// = 4.6 TB/s of matrix rows at N = 256, B = 1024 (the resident colonies' matrices exceed L2, so most of it is HBM).
#include <math.h>
#include <stdlib.h>

#include <vector>

#include "tma.cuh"
#include "wr_internal.cuh"

namespace wr {

constexpr int kGtspRows = 8;     // rows per TMA chunk
constexpr int kGtspMaxStages = 4; // TMA ring depth is a template parameter of the kernel (2..4)
constexpr int kGtspIv = 16;      // check-point interval (cities)
constexpr double kGtspInf = 1061109567.0;   // INF 0x3f3f3f3f (ACS_GTSP.hpp:19), ACS_Tour::clean :29-34

// computeSolution's locals (:258-259) for one colony during one wr_gtsp_solve call
struct GtspSolve {
    double last;                 // lowest best L seen in this call
    int bad_times;               // consecutive iterations that did not lower it
    int ran;                     // iterations run in this call
};

// the stopping rule of computeSolution (:262-264), with the iteration cap of the call
__device__ __forceinline__ bool gtsp_stopped(const GtspSolve& s, int n, int cap) { return s.bad_times > n || s.ran >= cap; }

struct GtspArgs {
    int n, npad;                 // cities; row stride of every matrix (multiple of 2 doubles = 16 B)
    int stages;                  // TMA ring depth
    size_t mat_stride;           // doubles between consecutive colonies' matrices
    int iterations;              // per colony in this launch (a solve launch: at most this many)
    int* iter;                   // [B] iterations each colony has run so far: the Philox iteration index of its next one
    GtspSolve* solve;            // [B] stopping-rule state of a wr_gtsp_solve launch; nullptr: wr_gtsp_iterate, no stopping rule
    int cap;                     // solve: iterations per colony in the whole call
    double* hist;                // solve (nullable): [B][iterations] best L after each iteration of this launch
    int* running;                // solve: incremented by every colony that has not stopped at the end of the launch
    int colony_first;
    uint32_t seed_lo, seed_hi;
    double evap;                 // 1 - alpha (:177), computed in double on the host
    const double* dis;           // [n][npad]
    const double* h6;            // [n][npad]  heuristic^beta, beta = 6 (:117-118), identical for all colonies
    double* ph;                  // [B][n][npad]
    double* info;                // [B][n][npad]
    uint16_t* tours;             // [B][n steps][n ants]  next city per (step, ant)
    uint16_t* best_tour;         // [B][n]  next-city list of the best ant
    int* best_start;             // [B]
    double* best_L;              // [B]
    unsigned long long* phase_ns;  // [3] summed over CTAs: info rebuild, construction, update
};

__device__ __forceinline__ unsigned long long gtimer()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

template <int kGtspStages>
__global__ void k_gtsp_iterate(GtspArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int n = a.n, npad = a.npad;
    const int nthreads = blockDim.x;
    const int k = threadIdx.x;             // ant
    const bool ant = k < n;
    const int nck = (n + kGtspIv - 1) / kGtspIv;
    const int nwords = (n + 31) / 32;
    // shared layout
    double* rows = reinterpret_cast<double*>(smem_raw);                       // [kGtspStages][kGtspRows][npad]
    double* ckpt = rows + kGtspStages * kGtspRows * npad;                               // [nck][nthreads]
    uint32_t* vis = reinterpret_cast<uint32_t*>(ckpt + (size_t)nck * nthreads);   // [nwords][nthreads]  bit set = visited
    double* redL = reinterpret_cast<double*>(vis + (size_t)nwords * nthreads);    // [32]
    int* redK = reinterpret_cast<int*>(redL + 32);                            // [32]
    uint64_t* bar = reinterpret_cast<uint64_t*>(redK + 32);                   // [kGtspStages]
    int* bcast = reinterpret_cast<int*>(bar + kGtspMaxStages);                // [4]: winner, improved, stopped, first iteration

    const size_t mat = (size_t)n * npad;
    const int colony = blockIdx.x;
    double* ph = a.ph + (size_t)colony * a.mat_stride;
    double* info = a.info + (size_t)colony * a.mat_stride;
    uint16_t* tours = a.tours + (size_t)colony * n * n;
    const uint32_t stream = kStreamGtsp + (uint32_t)(a.colony_first + colony);

    if (k == 0) {
        for (int s = 0; s < kGtspStages; s++) tma::mbar_init(&bar[s], 1);
        tma::fence_barrier_init();
        bcast[2] = a.solve ? gtsp_stopped(a.solve[colony], n, a.cap) : 0;   // a colony that stopped in an earlier launch returns at once
        bcast[3] = a.iter[colony];
    }
    __syncthreads();
    unsigned phase_bits = 0;   // bit s: parity of the next wait on bar[s]
    unsigned consumed = 0, issued = 0;   // chunks waited for / requested so far (ring positions persist across iterations)
    const int nchunks = (n + kGtspRows - 1) / kGtspRows;
    const int total = n * nchunks;       // chunks per iteration: every step streams the whole matrix once
    auto issue = [&](int j) {            // thread 0: request chunk j of this iteration into ring slot issued % S
        const int c0 = (j % nchunks) * kGtspRows, nr = min(kGtspRows, n - c0);
        const unsigned st = issued % kGtspStages;
        tma::mbar_arrive_expect_tx(&bar[st], (uint32_t)(nr * npad * sizeof(double)));
        tma::bulk_g2s(rows + (size_t)st * kGtspRows * npad, info + (size_t)c0 * npad, (uint32_t)(nr * npad * sizeof(double)), &bar[st]);
    };
    unsigned long long t_info = 0, t_cons = 0, t_upd = 0;

    // bcast[2] is set by thread 0 before the barrier that ends an iteration and read by all threads after it, so the stop
    // is uniform over the CTA.  Leaving between iterations is safe for the TMA ring: an iteration issues and waits for
    // exactly `total` chunks, so no bulk copy is in flight into shared memory there.
    int it = 0;
    for (; it < a.iterations && !bcast[2]; it++) {
        const uint32_t iter = (uint32_t)(bcast[3] + it);
        unsigned long long t0 = gtimer();
        // ---- reset(): info = pheromone^1 * heuristic^6 (:114-119) --------------------------------
        for (size_t i = k; i < mat; i += nthreads) info[i] = __dmul_rn(__dmul_rn(1.0, ph[i]), a.h6[i]);
        for (int w = 0; w < nwords; w++) vis[w * nthreads + k] = 0;
        int r = k, left = n - 1;           // r1[k] = k (:109), J[k] = all \ {k} (:110-111)
        if (ant) vis[(k >> 5) * nthreads + k] = 1u << (k & 31);
        double L = 0.0;
        asm volatile("fence.proxy.async;" ::: "memory");   // generic-proxy writes of info -> visible to the TMA reads below
        __syncthreads();
        unsigned long long t1 = gtimer();
        // ---- construct_solution(): n steps, every ant moves once per step (:146-159) ------------
        int it_issued = 0;
        for (; it_issued < kGtspStages - 1 && it_issued < total; it_issued++, issued++) if (k == 0) issue(it_issued);
        for (int step = 0; step < n; step++) {
            double sum = 0.0;
            for (int ch = 0; ch < nchunks; ch++) {
                // ring slot (consumed-1) % S was released by the barrier that ended the previous chunk: refill it
                // (this runs ahead across step boundaries: `info` does not change within an iteration)
                if (it_issued < total) { if (k == 0) issue(it_issued); it_issued++; issued++; }
                const unsigned b = consumed % kGtspStages;
                tma::mbar_wait(&bar[b], (phase_bits >> b) & 1u);
                phase_bits ^= 1u << b;
                consumed++;
                if (ant && left > 0) {
                    // column r of the staged rows: info[c][r] == info[r][c]
                    const double* col = rows + (int)b * (kGtspRows * npad) + r;
                    const int c0 = ch * kGtspRows, nr = min(kGtspRows, n - c0);
                    // kGtspRows divides 32 and c0 is a multiple of it: the chunk's visited bits are one byte
                    const uint32_t vb = vis[(c0 >> 5) * nthreads + k] >> (c0 & 31);
                    if (nr == kGtspRows) {
                        // all eight loads first (unconditional), then the dependent chain; a visited city contributes
                        // +0.0, which is the identity of the (non-negative) running sum, so no load sits under a predicate
                        double x[kGtspRows];
#pragma unroll
                        for (int j = 0; j < kGtspRows; j++) x[j] = col[j * npad];
#pragma unroll
                        for (int j = 0; j < kGtspRows; j++) sum = __dadd_rn(sum, ((vb >> j) & 1u) ? 0.0 : x[j]);
                    } else {
                        for (int j = 0; j < nr; j++) {
                            const double x = col[j * npad];
                            if (!((vb >> j) & 1u)) sum = __dadd_rn(sum, x);
                        }
                    }
                    // check-point after cities 16i+15 and after the last city (warp-uniform condition)
                    const int cend = c0 + nr;
                    if ((cend & (kGtspIv - 1)) == 0 || cend == n) ckpt[((cend - 1) / kGtspIv) * nthreads + k] = sum;
                }
                __syncthreads();
            }
            // ---- select_next (:122-144) ----------------------------------------------------------
            int next = k;                                     // J empty -> home city r1[k] (:124-125); also the fall-through (:143)
            if (ant && left > 0) {
                const uint32_t r31 = rand31(a.seed_lo, a.seed_hi, iter, (uint32_t)k, (uint32_t)step, stream);
                double rnd = __ddiv_rn((double)(int)r31, 2147483647.0);   // (double)rand()/(double)RAND_MAX (:126)
                rnd = __dmul_rn(rnd, sum);
                int iv = -1;
                if (rnd <= 0.0) {
                    // every prefix sum is >= 0 >= rnd: the reference takes the lowest unvisited city.  The check-point search
                    // would stop at interval 0 even when all its cities are visited (a zero draw, a zero or subnormal sum),
                    // so the city comes from the visited words; left > 0 puts it below n.  A NaN rnd skips both branches.
                    for (int w = 0;; w++) {
                        const uint32_t fr = ~vis[w * nthreads + k];
                        if (fr) { next = w * 32 + __ffs(fr) - 1; break; }
                    }
                } else {
                    for (int j = 0; j < nck; j++) if (ckpt[j * nthreads + k] >= rnd) { iv = j; break; }
                }
                if (iv >= 0) {
                    double s = iv > 0 ? ckpt[(iv - 1) * nthreads + k] : 0.0;
                    const int c0 = iv * kGtspIv;
                    const uint32_t vb = vis[(c0 >> 5) * nthreads + k] >> (c0 & 31);   // kGtspIv divides 32
                    // the 16 candidates of the interval are fetched together (independent L2 gathers), then re-added
                    // in city order from the exact check-pointed partial sum
                    double xv[kGtspIv];
#pragma unroll
                    for (int j = 0; j < kGtspIv; j++) {
                        const int c = c0 + j;
                        xv[j] = (c < n && !((vb >> j) & 1u)) ? info[(size_t)c * npad + r] : 0.0;
                    }
                    bool hit = false;
#pragma unroll
                    for (int j = 0; j < kGtspIv; j++) {
                        const int c = c0 + j;
                        if (c < n && !((vb >> j) & 1u)) {
                            s = __dadd_rn(s, xv[j]);
                            if (!hit && s >= rnd) { next = c; hit = true; }
                        }
                    }
                }
            }
            if (ant) {
                const uint32_t bit = 1u << (next & 31);
                uint32_t* w = &vis[(next >> 5) * nthreads + k];
                if (!(*w & bit)) { *w |= bit; left--; }           // J[k].erase(next) (:153)
                tours[(size_t)step * n + k] = (uint16_t)next;        // tour[k].push_back(r, next) (:155)
                if (step < n - 1) L = __dadd_rn(L, a.dis[(size_t)r * npad + next]);   // ACS_Tour::calc skips the closing edge (:36-44)
                r = next;
            }
        }
        unsigned long long t2 = gtimer();
        // ---- update_pheromone (:161-185) ------------------------------------------------------------
        // now_best = first strict minimum over ants in index order (:165-170)
        double bl = ant ? L : INFINITY;
        int bk = ant ? k : 0x7fffffff;
        for (int o = 16; o; o >>= 1) {
            double ol = __shfl_xor_sync(0xffffffffu, bl, o);
            int ok = __shfl_xor_sync(0xffffffffu, bk, o);
            if (ol < bl || (ol == bl && ok < bk)) { bl = ol; bk = ok; }
        }
        if ((k & 31) == 0) { redL[k >> 5] = bl; redK[k >> 5] = bk; }
        __syncthreads();
        if (k < 32) {
            const int nw = (nthreads + 31) / 32;
            bl = k < nw ? redL[k] : INFINITY; bk = k < nw ? redK[k] : 0x7fffffff;
            for (int o = 16; o; o >>= 1) {
                double ol = __shfl_xor_sync(0xffffffffu, bl, o);
                int ok = __shfl_xor_sync(0xffffffffu, bk, o);
                if (ol < bl || (ol == bl && ok < bk)) { bl = ol; bk = ok; }
            }
            if (k == 0) {
                const bool have = bl < kGtspInf;                 // tour[i] < now_best with now_best.L = INF (:164-169)
                redL[0] = bl; bcast[0] = have ? bk : -1;
                bcast[1] = (have && bl < a.best_L[colony]) ? 1 : 0;   // now_best < best (:171-174)
                if (bcast[1]) { a.best_L[colony] = bl; a.best_start[colony] = bk; }
                if (a.solve) {   // computeSolution :266-275
                    GtspSolve s = a.solve[colony];
                    const double best = a.best_L[colony];
                    if (s.last > best) { s.last = best; s.bad_times = 0; } else s.bad_times++;
                    if (a.hist) a.hist[(size_t)colony * a.iterations + it] = best;
                    s.ran++;
                    a.solve[colony] = s;
                    bcast[2] = gtsp_stopped(s, n, a.cap);
                }
            }
        }
        __syncthreads();
        const int win = bcast[0];
        const double winL = redL[0];
        if (bcast[1]) for (int s = k; s < n; s += nthreads) a.best_tour[(size_t)colony * n + s] = tours[(size_t)s * n + win];
        for (size_t i = k; i < mat; i += nthreads) ph[i] = __dmul_rn(ph[i], a.evap);   // :175-177 (padding columns included, harmless)
        __syncthreads();
        if (win >= 0 && k == 0) {
            // :179-184, in edge order (a valid tour never repeats an unordered pair, but the roulette
            // fall-through of :143 can produce one, so the deposits stay sequential: 2n updates)
            const double dep = __ddiv_rn(1.0, winL);
            int rr = win;
            for (int s = 0; s < n; s++) {
                const int ss = tours[(size_t)s * n + win];
                const double v = __dadd_rn(ph[(size_t)rr * npad + ss], dep);
                ph[(size_t)rr * npad + ss] = v;
                ph[(size_t)ss * npad + rr] = v;
                rr = ss;
            }
        }
        __syncthreads();
        unsigned long long t3 = gtimer();
        t_info += t1 - t0; t_cons += t2 - t1; t_upd += t3 - t2;
    }
    if (k == 0) {
        atomicAdd(&a.phase_ns[0], t_info); atomicAdd(&a.phase_ns[1], t_cons); atomicAdd(&a.phase_ns[2], t_upd);
        a.iter[colony] = bcast[3] + it;
        if (a.solve && !bcast[2]) atomicAdd(a.running, 1);
    }
}

}  // namespace wr

using namespace wr;

struct wr_gtsp {
    int device = 0;
    int n = 0, npad = 0, batch = 0, colony_first = 0;
    uint64_t seed = 0;
    double tau0 = 0;
    double *d_dis = nullptr, *d_h6 = nullptr, *d_ph = nullptr, *d_info = nullptr, *d_best_L = nullptr;
    uint16_t *d_tours = nullptr, *d_best_tour = nullptr;
    int* d_best_start = nullptr;
    int* d_iter = nullptr;                 // [batch] iterations run per colony
    GtspSolve* d_solve = nullptr;          // [batch], allocated by the first wr_gtsp_solve
    double* d_hist = nullptr;              // [batch][kGtspSolveSlice]
    int* d_running = nullptr;
    unsigned long long* d_phase = nullptr;
    cudaStream_t stream = nullptr;
    float ms_total = 0;
    size_t smem = 0;
    int threads = 0;
    int stages = 6;
    size_t mat_stride = 0;
};

template <class T> static T host_power(T x, int y)
{   // power<T>() ACSRank_3D.hpp:48-60
    T ans = 1;
    while (y) { if (y & 1) ans *= x; x *= x; y >>= 1; }
    return ans;
}

extern "C" int wr_gtsp_destroy(wr_gtsp* g)
{
    if (!g) return WR_OK;
    if (g->stream) { cudaStreamSynchronize(g->stream); cudaStreamDestroy(g->stream); }
    cudaFree(g->d_dis); cudaFree(g->d_h6); cudaFree(g->d_ph); cudaFree(g->d_info); cudaFree(g->d_best_L);
    cudaFree(g->d_tours); cudaFree(g->d_best_tour); cudaFree(g->d_best_start); cudaFree(g->d_phase);
    cudaFree(g->d_iter); cudaFree(g->d_solve); cudaFree(g->d_hist); cudaFree(g->d_running);
    delete g;
    return WR_OK;
}

// TMA ring depth 3 (two CTAs per SM at N = 256) measured best: 2 -> 33.0k, 3 -> 34.7k, 4 -> 31.9k, 6 -> 21.3k colony-iterations/s
// at N = 256 x 1024 colonies (per-CTA latency wants more CTAs per SM, L2 capacity wants fewer resident matrices)
constexpr int kGtspStages = 3;
constexpr size_t kGtspSmemMax = 227 * 1024;

// dynamic shared memory of k_gtsp_iterate for n cities: the ring of matrix rows, then per ant (one per thread) its
// check-points and visited bits, then the reduction and barrier words
static size_t gtsp_smem(int n, int stages)
{
    const size_t npad = (size_t)((n + 1) & ~1), threads = (size_t)(n + 31) / 32 * 32;
    const size_t nck = (size_t)(n + kGtspIv - 1) / kGtspIv, nwords = (size_t)(n + 31) / 32;
    return (size_t)stages * kGtspRows * npad * sizeof(double) + nck * threads * sizeof(double) + nwords * threads * sizeof(uint32_t) +
           32 * sizeof(double) + 32 * sizeof(int) + kGtspMaxStages * sizeof(uint64_t) + 4 * sizeof(int);
}

// the largest city count whose shared memory fits one CTA (464)
static int gtsp_max_cities()
{
    int n = 2;
    while (n < 1024 && gtsp_smem(n + 1, kGtspStages) <= kGtspSmemMax) n++;
    return n;
}

// readFromGraphFile :224-253 (matrix passed in memory) + init_param :187-218
extern "C" int wr_gtsp_create(const double* dis, int n, int cnt, int batch, int colony_first, uint64_t seed, wr_gtsp** out)
{
    WR_REQUIRE(dis && out && n >= 2 && batch >= 1 && colony_first >= 0, WR_ERR_INVALID, "wr_gtsp_create: bad argument");
    const int nmax = gtsp_max_cities();
    if (n > nmax) {
        set_error("wr_gtsp_create: at most %d cities (one ant per thread: its check-points and visited bits, with a %d-stage ring of "
                  "matrix rows, must fit %zu B of shared memory; %d cities need %zu B)", nmax, kGtspStages, kGtspSmemMax, n, gtsp_smem(n, kGtspStages));
        return WR_ERR_INVALID;
    }
    WR_REQUIRE(colony_first + batch <= 65536, WR_ERR_INVALID, "wr_gtsp_create: colony ids must stay below 65536 (Philox stream tag)");
    *out = nullptr;
    wr_gtsp* g = new wr_gtsp();
    g->n = n; g->npad = (n + 1) & ~1; g->batch = batch; g->colony_first = colony_first; g->seed = seed;
    const int npad = g->npad;
    double tmp = 0;
    for (int i = 0; i < n; i++)
        for (int j = i + 1; j < n; j++) tmp += dis[(size_t)i * n + j];   // :246, file order
    g->tau0 = (double)cnt / (tmp * n);                                 // :249
    std::vector<double> hd((size_t)n * npad, 0.0), hh((size_t)n * npad, 0.0);
    for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) {
            const double d = i == j ? 0.0 : dis[(size_t)i * n + j];    // the reference never reads its (uninitialised) diagonal
            hd[(size_t)i * npad + j] = d;
            hh[(size_t)i * npad + j] = host_power(1 / (d + 1e-8), 6);  // herustic :211, beta = 6 :191, power() :117-118
        }
    const size_t mat = (size_t)n * npad;
    g->stages = kGtspStages;
    g->mat_stride = mat;
#define WR_CUDA_G(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { set_error("%s failed: %s", #expr, cudaGetErrorString(_e)); wr_gtsp_destroy(g); return WR_ERR_CUDA; } } while (0)
    WR_CUDA_G(cudaGetDevice(&g->device));
    WR_CUDA_G(cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking));
    WR_CUDA_G(cudaMalloc(&g->d_dis, mat * sizeof(double)));
    WR_CUDA_G(cudaMalloc(&g->d_h6, mat * sizeof(double)));
    WR_CUDA_G(cudaMalloc(&g->d_ph, g->mat_stride * batch * sizeof(double)));
    WR_CUDA_G(cudaMalloc(&g->d_info, g->mat_stride * batch * sizeof(double)));
    WR_CUDA_G(cudaMalloc(&g->d_tours, (size_t)n * n * batch * sizeof(uint16_t)));
    WR_CUDA_G(cudaMalloc(&g->d_best_tour, (size_t)n * batch * sizeof(uint16_t)));
    WR_CUDA_G(cudaMalloc(&g->d_best_start, batch * sizeof(int)));
    WR_CUDA_G(cudaMalloc(&g->d_best_L, batch * sizeof(double)));
    WR_CUDA_G(cudaMalloc(&g->d_phase, 3 * sizeof(unsigned long long)));
    WR_CUDA_G(cudaMemset(g->d_phase, 0, 3 * sizeof(unsigned long long)));
    WR_CUDA_G(cudaMalloc(&g->d_iter, batch * sizeof(int)));
    WR_CUDA_G(cudaMemset(g->d_iter, 0, batch * sizeof(int)));
    WR_CUDA_G(cudaMemcpy(g->d_dis, hd.data(), mat * sizeof(double), cudaMemcpyHostToDevice));
    WR_CUDA_G(cudaMemcpy(g->d_h6, hh.data(), mat * sizeof(double), cudaMemcpyHostToDevice));
    {
        std::vector<double> p0(g->mat_stride * batch, g->tau0);        // pheromone[i][j] = pheromone_0 (:209)
        WR_CUDA_G(cudaMemcpy(g->d_ph, p0.data(), p0.size() * sizeof(double), cudaMemcpyHostToDevice));
        std::vector<double> bl(batch, kGtspInf);                       // best.clean() (:214)
        WR_CUDA_G(cudaMemcpy(g->d_best_L, bl.data(), batch * sizeof(double), cudaMemcpyHostToDevice));
        std::vector<int> bs(batch, -1);
        WR_CUDA_G(cudaMemcpy(g->d_best_start, bs.data(), batch * sizeof(int), cudaMemcpyHostToDevice));
    }
    g->threads = (n + 31) / 32 * 32;
    g->smem = gtsp_smem(n, g->stages);   // <= kGtspSmemMax: n <= gtsp_max_cities()
    WR_CUDA_G(cudaFuncSetAttribute(k_gtsp_iterate<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g->smem));
    WR_CUDA_G(cudaFuncSetAttribute(k_gtsp_iterate<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g->smem));
    WR_CUDA_G(cudaFuncSetAttribute(k_gtsp_iterate<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g->smem));
#undef WR_CUDA_G
    *out = g;
    return WR_OK;
}

static GtspArgs gtsp_args(const wr_gtsp* g, int iterations)
{
    GtspArgs a;
    a.n = g->n; a.npad = g->npad; a.stages = g->stages; a.mat_stride = g->mat_stride; a.iterations = iterations; a.iter = g->d_iter;
    a.solve = nullptr; a.cap = 0; a.hist = nullptr; a.running = nullptr; a.colony_first = g->colony_first;
    a.seed_lo = (uint32_t)g->seed; a.seed_hi = (uint32_t)(g->seed >> 32);
    a.evap = 1 - 0.1;   // (1 - alpha), alpha = 0.1 (:189)
    a.dis = g->d_dis; a.h6 = g->d_h6; a.ph = g->d_ph; a.info = g->d_info; a.tours = g->d_tours; a.best_tour = g->d_best_tour;
    a.best_start = g->d_best_start; a.best_L = g->d_best_L; a.phase_ns = g->d_phase;
    return a;
}

// one launch of k_gtsp_iterate over every colony, event-timed into wr_gtsp_kernel_ms; returns after it has finished
static int gtsp_launch(wr_gtsp* g, const GtspArgs& a)
{
    cudaEvent_t e0, e1;
    WR_CUDA(cudaEventCreate(&e0));
    WR_CUDA(cudaEventCreate(&e1));
    WR_CUDA(cudaEventRecord(e0, g->stream));
    if (g->stages == 2) k_gtsp_iterate<2><<<g->batch, g->threads, g->smem, g->stream>>>(a);
    else if (g->stages == 3) k_gtsp_iterate<3><<<g->batch, g->threads, g->smem, g->stream>>>(a);
    else k_gtsp_iterate<4><<<g->batch, g->threads, g->smem, g->stream>>>(a);
    WR_CUDA(cudaGetLastError());
    WR_CUDA(cudaEventRecord(e1, g->stream));
    WR_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    WR_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    g->ms_total += ms;
    return WR_OK;
}

// the loop body of computeSolution :261-276, `iterations` times per colony, without the early stop
extern "C" int wr_gtsp_iterate(wr_gtsp* g, int iterations)
{
    WR_REQUIRE(g && iterations >= 0, WR_ERR_INVALID, "wr_gtsp_iterate: bad argument");
    if (iterations == 0) return WR_OK;
    WR_CUDA(cudaSetDevice(g->device));
    return gtsp_launch(g, gtsp_args(g, iterations));
}

// Iterations per wr_gtsp_solve launch.  One iteration takes milliseconds at a few hundred cities, and the cap (n*n) reaches
// 215 296 at 464 cities: the solve is a sequence of bounded launches, with one word (colonies still running) read back after
// each.  The history goes through a [batch][kGtspSolveSlice] device buffer copied out after each launch.
constexpr int kGtspSolveSlice = 32;

// computeSolution :255-284 for every colony, each stopping by its own rule
extern "C" int wr_gtsp_solve(wr_gtsp* g, int max_iterations, int* iterations, double* best_L_history, int* best_colony)
{
    WR_REQUIRE(g && max_iterations >= 0, WR_ERR_INVALID, "wr_gtsp_solve: bad argument");
    WR_CUDA(cudaSetDevice(g->device));
    const int cap = max_iterations > 0 ? max_iterations : g->n * g->n;   // MAX_itera (:257)
    const int B = g->batch;
    if (!g->d_solve) {
        WR_CUDA(cudaMalloc(&g->d_solve, B * sizeof(GtspSolve)));
        WR_CUDA(cudaMalloc(&g->d_hist, (size_t)B * kGtspSolveSlice * sizeof(double)));
        WR_CUDA(cudaMalloc(&g->d_running, sizeof(int)));
    }
    std::vector<GtspSolve> st(B, GtspSolve{kGtspInf, 0, 0});   // last = INF, bad_times = 0 (:258-259), afresh with every call
    WR_CUDA(cudaMemcpyAsync(g->d_solve, st.data(), B * sizeof(GtspSolve), cudaMemcpyHostToDevice, g->stream));
    GtspArgs a = gtsp_args(g, kGtspSolveSlice);
    a.solve = g->d_solve; a.cap = cap; a.hist = best_L_history ? g->d_hist : nullptr; a.running = g->d_running;
    std::vector<double> h(best_L_history ? (size_t)B * kGtspSolveSlice : 0);
    for (int start = 0;; start += kGtspSolveSlice) {
        WR_CUDA(cudaMemsetAsync(g->d_running, 0, sizeof(int), g->stream));
        const int rc = gtsp_launch(g, a);
        if (rc != WR_OK) return rc;
        int running = 0;
        WR_CUDA(cudaMemcpyAsync(&running, g->d_running, sizeof(int), cudaMemcpyDeviceToHost, g->stream));
        if (best_L_history) {
            WR_CUDA(cudaMemcpyAsync(st.data(), g->d_solve, B * sizeof(GtspSolve), cudaMemcpyDeviceToHost, g->stream));
            WR_CUDA(cudaMemcpyAsync(h.data(), g->d_hist, h.size() * sizeof(double), cudaMemcpyDeviceToHost, g->stream));
        }
        WR_CUDA(cudaStreamSynchronize(g->stream));
        // a colony that ran in this launch had run exactly `start` iterations before it (it never stopped earlier)
        for (int b = 0; best_L_history && b < B; b++)
            for (int j = 0; j < st[b].ran - start; j++) best_L_history[(size_t)b * cap + start + j] = h[(size_t)b * kGtspSolveSlice + j];
        if (!running) break;
    }
    if (iterations) {
        WR_CUDA(cudaMemcpy(st.data(), g->d_solve, B * sizeof(GtspSolve), cudaMemcpyDeviceToHost));
        for (int b = 0; b < B; b++) iterations[b] = st[b].ran;
    }
    if (best_colony) {
        std::vector<double> L(B);
        WR_CUDA(cudaMemcpy(L.data(), g->d_best_L, B * sizeof(double), cudaMemcpyDeviceToHost));
        int bc = 0;
        for (int b = 1; b < B; b++) if (L[b] < L[bc]) bc = b;
        *best_colony = bc;
    }
    return WR_OK;
}

extern "C" int wr_gtsp_sync(wr_gtsp* g)
{
    WR_REQUIRE(g, WR_ERR_INVALID, "wr_gtsp_sync: null");
    WR_CUDA(cudaStreamSynchronize(g->stream));
    return WR_OK;
}

extern "C" int wr_gtsp_best(wr_gtsp* g, int colony, int* tour_pairs, int* nedges, double* L)
{
    WR_REQUIRE(g && nedges && L && colony >= 0 && colony < g->batch, WR_ERR_INVALID, "wr_gtsp_best: bad argument");
    WR_CUDA(cudaStreamSynchronize(g->stream));
    int start = -1;
    WR_CUDA(cudaMemcpy(L, g->d_best_L + colony, sizeof(double), cudaMemcpyDeviceToHost));
    WR_CUDA(cudaMemcpy(&start, g->d_best_start + colony, sizeof(int), cudaMemcpyDeviceToHost));
    if (start < 0) { *nedges = 0; return WR_OK; }
    *nedges = g->n;
    if (tour_pairs) {
        std::vector<uint16_t> t(g->n);
        WR_CUDA(cudaMemcpy(t.data(), g->d_best_tour + (size_t)colony * g->n, g->n * sizeof(uint16_t), cudaMemcpyDeviceToHost));
        int r = start;
        for (int i = 0; i < g->n; i++) { tour_pairs[2 * i] = r; tour_pairs[2 * i + 1] = t[i]; r = t[i]; }
    }
    return WR_OK;
}

extern "C" int wr_gtsp_download_pheromone(wr_gtsp* g, int colony, double* out)
{
    WR_REQUIRE(g && out && colony >= 0 && colony < g->batch, WR_ERR_INVALID, "wr_gtsp_download_pheromone: bad argument");
    WR_CUDA(cudaStreamSynchronize(g->stream));
    WR_CUDA(cudaMemcpy2D(out, (size_t)g->n * sizeof(double), g->d_ph + (size_t)colony * g->mat_stride, (size_t)g->npad * sizeof(double),
                         (size_t)g->n * sizeof(double), g->n, cudaMemcpyDeviceToHost));
    return WR_OK;
}

extern "C" int wr_gtsp_tau0(wr_gtsp* g, double* tau0)
{
    WR_REQUIRE(g && tau0, WR_ERR_INVALID, "wr_gtsp_tau0: null");
    *tau0 = g->tau0;
    return WR_OK;
}

// event-timed total of all wr_gtsp_iterate and wr_gtsp_solve launches, split by the CTAs' own phase clocks
extern "C" int wr_gtsp_kernel_ms(wr_gtsp* g, float out[3])
{
    WR_REQUIRE(g && out, WR_ERR_INVALID, "wr_gtsp_kernel_ms: null");
    WR_CUDA(cudaStreamSynchronize(g->stream));
    unsigned long long ns[3];
    WR_CUDA(cudaMemcpy(ns, g->d_phase, sizeof ns, cudaMemcpyDeviceToHost));
    const double tot = (double)ns[0] + (double)ns[1] + (double)ns[2];
    for (int i = 0; i < 3; i++) out[i] = tot > 0 ? (float)(g->ms_total * ((double)ns[i] / tot)) : 0.f;
    return WR_OK;
}
