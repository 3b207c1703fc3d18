/* wr_gpu.h — C ABI of libwrgpu.so, the B200 (sm_100a) device layer of the welding-robot
 * ACS hot path.
 *
 * The reference (mhsitu/welding_robot) has no FFI: its boundary is a header-only C++ class
 * surface (SURVEY.md §8b).  This header is the C-ABI a replacement must export for that
 * surface; every entry point names the reference code it replaces (paths relative to the
 * reference root).  The C++ facade in include/welding_robot_b200/ re-creates the reference's
 * class and method names on top of these calls; INTEGRATION.md shows the binding.
 *
 * Conventions
 *  - plain C types only; all buffers are caller-owned HOST memory unless a name says `dev`;
 *  - every call returns a wr_status (0 = ok, negative = error); wr_last_error() gives the
 *    message of the calling thread's last failure; nothing throws or exits;
 *  - a handle is used by one host thread at a time; different handles may be used from
 *    different threads / on different devices; a handle lives on the device that was
 *    current (wr_set_device) when it was created;
 *  - there is NO CPU fallback: without a usable CUDA device every compute call fails with
 *    WR_ERR_CUDA.
 */
#ifndef WR_GPU_H
#define WR_GPU_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    WR_OK = 0,
    WR_ERR_INVALID = -1,  /* bad argument */
    WR_ERR_CUDA = -2,     /* CUDA runtime error / no device */
    WR_ERR_NOMEM = -3,
    WR_ERR_STATE = -4,    /* call order (e.g. iterate before endpoints are set) */
    WR_ERR_NOTFOUND = -5, /* route point does not snap to a free node */
    WR_ERR_CAPACITY = -6, /* caller buffer too small */
    WR_ERR_FORMAT = -7    /* malformed STL / grid / graph input */
} wr_status;

typedef struct wr_grid wr_grid;   /* bit-packed occupancy grid + axis coordinates, resident in HBM */
typedef struct wr_acs wr_acs;     /* one rank-based 3-D ant-colony search (pheromone field in HBM) */
typedef struct wr_gtsp wr_gtsp;   /* a batch of seam-ordering colonies */

const char* wr_last_error(void);
int wr_version(void);
int wr_device_count(int* count);
int wr_set_device(int device);

/* ------------------------------------------------------------------------------------------
 * STL — replaces STLReader::readFile / ReadBinary (core/read_STL.hpp:26-77, 131-174).
 * buf/len: the whole file.  tris12: 12 floats per triangle (normal, v0, v1, v2).
 * *ntri receives the triangle count in the file; at most `cap` triangles are written.
 * The ASCII branch (read_STL.hpp:99-129) is not supported -> WR_ERR_FORMAT.
 * ---------------------------------------------------------------------------------------- */
int wr_stl_parse(const uint8_t* buf, size_t len, float* tris12, int cap, int* ntri);

/* ------------------------------------------------------------------------------------------
 * Voxel grid — replaces GridMap<T>::creatGridMap (core/model_grid_map.hpp:151-273).
 * Node id = z*ry*rx + y*rx + x (model_grid_map.hpp:214); occupancy is bit-packed, bit
 * (id & 31) of word (id >> 5), 1 = occupied (isFree == false).
 * ---------------------------------------------------------------------------------------- */
int wr_grid_create_from_triangles(const float* tris12, int ntri, float precision, int wall, wr_grid** out);
/* synthetic / reloaded grids: isfree is N bytes in z,y,x order (what readGridMap,
 * model_grid_map.hpp:300-356, produces); xs/ys/zs are the per-axis node coordinates. */
int wr_grid_create_from_occupancy(const uint8_t* isfree, int rx, int ry, int rz, const float* xs, const float* ys,
                                  const float* zs, float precision, wr_grid** out);
int wr_grid_destroy(wr_grid* g);
int wr_grid_dims(const wr_grid* g, int dims[3]);                       /* rangeX, rangeY, rangeZ (:381-383) */
int wr_grid_precision(const wr_grid* g, float* precision, int* wall);
int wr_grid_bbox(const wr_grid* g, float mn[3], float mx[3]);          /* global mesh box (:165-181) */
int wr_grid_coords(const wr_grid* g, float* xs, float* ys, float* zs); /* node coordinates (:204-211) */
int wr_grid_download_bits(const wr_grid* g, uint32_t* bits, size_t nwords);
int wr_grid_download_isfree(const wr_grid* g, uint8_t* isfree, size_t n);
/* occupied nodes, triangle-node predicate evaluations, device ms of the voxelise kernel */
int wr_grid_stats(const wr_grid* g, uint64_t* occupied, uint64_t* tests, float* kernel_ms);

/* ------------------------------------------------------------------------------------------
 * Rank-based 3-D ant colony search — replaces ACS_Rank (core/ACSRank_3D.hpp).
 * ---------------------------------------------------------------------------------------- */
typedef struct {
    int alpha;            /* pheromone exponent, ACSRank_3D.hpp:319 (1)            */
    float beta;           /* heuristic weight in tau^alpha*(1+beta*cos), :320 (0.6) */
    float rho;            /* evaporation factor, :321 (0.8)                        */
    float tau0;           /* initial pheromone, :324 (1)                           */
    int fixed_colony;     /* 0: adaptive colony_num of :247; >0: that many ants    */
    int step_cap;         /* 0: auto (min(N-1, 65532)); else max steps per ant     */
    int K;                /* neighbourhood: 6 (reference) or 26 (the extension disabled at :367-385; one GPU) */
    uint64_t seed;        /* Philox key; draw = f(seed; search, iteration, ant, step) */
    int update_mode;      /* WR_UPDATE_*; default WR_UPDATE_RANKSET (adaptive)     */
    int walk_table_log2;  /* log2 of per-ant shared-memory visited-tile slots (0: default 9) */
} wr_acs_params;

enum {
    WR_UPDATE_FUSED = 0,     /* one HBM pass: tile streamed through registers, rank-ordered deposits applied while the tile is in L2 */
    WR_UPDATE_SPLIT = 1,     /* float4 evaporation pass, then rank-ordered deposit pass (same bits) */
    WR_UPDATE_ATOMIC = 2,    /* evaporation pass + atomicAdd deposits (fast, order not reproducible) */
    /* 3 was a measurement variant (every tile through a TMA ring in shared memory); removed, rejected by wr_acs_create */
    WR_UPDATE_RANKSET = 4    /* adaptive: per touched slot the SET of depositing ranks (a deposit's value depends only on the rank and one
                                bit of the slot) is built with atomicOr and applied as one ordered chain — no record sort — on the
                                iterations where the colony's deposits are concentrated; sorted records + the fused pass (WR_UPDATE_FUSED)
                                while it still wanders.  The choice for iteration n is a pure function of the statistics of iteration
                                n-5 (read by the host without synchronising); same additions in the same order either way, same bits.
                                Any colony size, one GPU or sharded; the table has a fixed capacity (142 MB) and a build that would
                                exceed it falls back to an exact serial pass. */
};

/* Handles created in a loop (one search per request) re-use a few large buffers of their predecessors instead of allocating and
 * zeroing them again: the rank-set table of WR_UPDATE_RANKSET, the peer slab of a sharded handle and the IPC mappings of the
 * peers' slabs stay parked in the process after wr_acs_destroy.  wr_release_caches frees them (no search may be in flight). */
int wr_release_caches(void);
int wr_acs_default_params(wr_acs_params* p);                        /* literals of initFromGridMap :319-325 */
int wr_acs_create(wr_grid* g, const wr_acs_params* p, wr_acs** out); /* initFromGridMap :317-410 */
int wr_acs_destroy(wr_acs* a);
/* setPoints :537-565 — snap two world points to the last free node (z,y,x scan order) within
 * 1.2*precision on every axis.  ids[0]/ids[1] = start/goal node id (-1 if none). */
int wr_acs_set_points(wr_acs* a, const float start[3], const float goal[3], int64_t ids[2]);
int wr_acs_set_endpoints(wr_acs* a, int64_t start_id, int64_t goal_id);
/* setPoints' full-grid scan (:545-562) as a kernel, for any number of points at once: ids[i] = the node point i
 * (3 floats each) snaps to, -1 if none.  checkRoutePoints (:511-535) = this call over route_points. */
int wr_acs_snap_points(wr_acs* a, const float* pts_xyz, int npoints, int64_t* ids);
/* The all-pairs loop of searchBestPathOfPoints (:472-499) on the device: for every pair, wr_acs_begin(predict) +
 * n_iterations iterations + reset(), enqueued back to back with no host synchronisation; one read-back at the end.
 * L[p] = best.L (+inf: no path), path_nodes[p] = node count of the best path (0: none); row p of path_ids / path_dirs
 * (path_cap entries per row; both may be NULL with path_cap 0) gets min(path_nodes[p], path_cap) ids and one slot
 * index less.  Independent queries (BASELINE config 5) shard by giving every rank its own pairs. */
int wr_acs_search_pairs(wr_acs* a, const int64_t* start_ids, const int64_t* goal_ids, int npairs, float predict_path_len,
                        int n_iterations, float* L, int* path_nodes, int64_t* path_ids, int* path_dirs, int path_cap);
/* The same searches advanced CONCURRENTLY: one launch per phase covers every (query, ant) pair — a 35- or 256-ant search
 * alone leaves the GPU idle.  Per-query pheromone lives in one hash table keyed by (query, node) (a node without an entry
 * is worth the scalar every never-deposited slot holds), the geometric factor is computed per step.  Results are
 * bit-identical to wr_acs_search_pairs on the same handle state (query q takes Philox search index next_search + q either
 * way).  Both neighbourhoods batch; K = 26 entries hold the node's 26 slots, and a K = 26 batch never builds the dense
 * N x 26 heuristic table (the factor is computed per step for each query's goal).  Colonies above 4096 ants,
 * WR_UPDATE_ATOMIC and handles whose field is not in its initial / reset() state run as the sequential loop; so does a
 * single query, and a chunk whose table or overflow pool fills up.  Same arguments as wr_acs_search_pairs. */
int wr_acs_search_batch(wr_acs* a, const int64_t* start_ids, const int64_t* goal_ids, int nqueries, float predict_path_len,
                        int n_iterations, float* L, int* path_nodes, int64_t* path_ids, int* path_dirs, int path_cap);
/* Result `index` of the last wr_acs_search_pairs / wr_acs_search_batch (kept in the handle, packed by true length — call
 * those with path_cap = 0 and fetch the paths here instead of passing rows of step_cap + 1 entries).  Like wr_acs_best. */
int wr_acs_result_path(wr_acs* a, int index, int64_t* ids, int* dirs, int cap, int* n, float* L);
/* batch path: [0] queries per chunk [1] entries of the pheromone table [2] entries used by the last chunk
 * [3] chunks that fell back to the sequential loop since the handle was created */
int wr_acs_batch_stats(wr_acs* a, uint64_t out[4]);
/* computeSolution :220-305 = wr_acs_begin(predict) + wr_acs_iterate(max_iteration).
 * Random draws: the reference draws every search of an ACS_Rank object from ONE continuous rand() stream (:169, seeded
 * once at :327), so successive searches are independent.  Here a draw is Philox(seed; search, iteration, ant, step) and
 * `search` is the number of wr_acs_begin calls the handle has seen before this one (0, 1, 2 ...; the pairs of
 * wr_acs_search_pairs and the queries of wr_acs_search_batch take consecutive indices the same way).
 * wr_acs_set_next_search overrides the index the NEXT wr_acs_begin takes (e.g. to re-run query q of a batch alone). */
int wr_acs_begin(wr_acs* a, float predict_path_len);                /* :229-233 */
int wr_acs_set_next_search(wr_acs* a, uint32_t index);
int wr_acs_iterate(wr_acs* a, int n_iterations);                    /* loop body :237-299, n times; asynchronous; one GPU or sharded */
int wr_acs_sync(wr_acs* a);
int wr_acs_reset(wr_acs* a);                                        /* reset() :307-315 */
/* getSolution :506-509 / Agent::getPath, nodeIndex :93-100.  *n = node count of the best path
 * (0 if none yet); ids gets min(*n, cap) node ids, dirs min(*n-1, cap) slot indices; *L = best.L
 * (+inf if none). */
int wr_acs_best(wr_acs* a, int64_t* ids, int* dirs, int cap, int* n, float* L);
int wr_acs_download_pheromone(wr_acs* a, float* tau, size_t n);     /* N*K floats, node-major; K = 6: slots [-z,-y,-x,+x,+y,+z]; K = 26: the (dz,dy,dx) enumeration of :355-359 without the centre */
/* upload materialises the field (every tile takes part in the evaporation from then on); on a clean-tile handle a
 * -0.0f in the input is stored as +0.0f (the bit pattern of -0.0f is the handle's "never deposited" marker) */
int wr_acs_upload_pheromone(wr_acs* a, const float* tau, size_t n);
/* last iteration's colony (parity checks): size, lambda, Q of :247-249 */
int wr_acs_last_colony(wr_acs* a, int* colony, float* lambda, float* Q);
/* ant k of the last iteration: node ids visited (start first), *n = node count, *L = its length
 * (+inf if it died), *order = 1-based rank after the sort of :273 */
int wr_acs_last_ant(wr_acs* a, int k, int64_t* ids, int* dirs, int cap, int* n, float* L, int* order);
/* cumulative counters: [0] ant-steps [1] ants [2] arrived [3] dead: no candidate [4] dead: roulette
 * fall-through/NaN [5] dead: step cap [6] iterations [7] deposit records [8] visited-table overflows */
int wr_acs_counters(wr_acs* a, uint64_t out[9]);
/* cumulative device milliseconds per kernel since begin (CUDA events on the handle's stream):
 * [0] walk [1] rank+best [2] deposit build+sort [3] update (evaporate+deposit) [4] whole iterations */
int wr_acs_kernel_ms(wr_acs* a, float out[5]);
int wr_acs_set_timing(wr_acs* a, int enabled);
/* WR_UPDATE_RANKSET: [0] the last iteration took the rank-set path, [1] pheromone tiles that received deposits in the last
 * record-path iteration, [2] distinct slots in the last rank-set iteration, [3] rank-set iterations since begin */
int wr_acs_update_stats(wr_acs* a, uint32_t out[4]);
/* Clean-tile pheromone field (FUSED / RANKSET handles): [0] 16 KB tiles that hold at least one slot that ever received a
 * deposit since init/reset() — the only tiles the evaporation pass reads and writes — [1] tiles of the field.  Slots that
 * never received a deposit all hold the same value (tau0 * rho per iteration, kept as one scalar); downloads materialise it. */
int wr_acs_field_stats(wr_acs* a, uint64_t out[2]);
/* cumulative device ms and launch count, since begin and with timing enabled, of the kernel that streams the pheromone field
 * (k_update_fused or k_evaporate_tiles) measured by its own event pair inside the iteration loop */
int wr_acs_stream_kernel_ms(wr_acs* a, float* ms, int* launches);
/* measurement hook: run ONE kernel of the update path `reps` times back to back on the handle's
 * stream and report the average device time per launch (CUDA events).  which: 0 = fused update
 * (evaporation + the last iteration's deposit records), 1 = float4 evaporation pass alone,
 * 2 = device-to-device copy of the pheromone field (in-run copy ceiling).  The field is
 * multiplied by rho each time (which 0/1), so call it on a scratch search only. */
int wr_acs_bench_kernel(wr_acs* a, int which, int reps, float* ms_per_launch);
/* use an existing CUDA stream (cudaStream_t as void*); default: a private non-blocking stream.  (Round 1's sharded protocol issued
 * collectives from the host and needed the handle on the collectives' stream — the advisor's finding; since round 2 the exchange
 * of a sharded iteration lives inside the library's kernels, so any stream will do.  The default streams cannot be captured into
 * the steady-state CUDA graph: a handle on one of them runs plain launches.) */
int wr_acs_set_stream(wr_acs* a, void* cuda_stream);

/* ---- ant sharding across ranks (SURVEY.md §8e): one process per GPU ------------------------------------------------
 * The pheromone field and the grid are replicated; rank r constructs ants [r*chunk, (r+1)*chunk) of the global colony,
 * chunk = ceil(colony_max / nranks).  Philox is keyed by the GLOBAL ant index, so the result does not depend on the rank
 * count: pheromone field (on every rank), best path and ranks are bit-identical to the 1-GPU run.
 *
 * The exchange runs over NVLink peer memory inside the library's own kernels — no collective library and no host
 * synchronisation in the iteration loop.  Everything a peer reads lives in ONE slab per rank (barrier flags, step
 * counts, ant trails, final slot values, published rank-set blocks), exported with one CUDA IPC handle per search.
 * One iteration of wr_acs_iterate on a sharded handle:
 *     walk (local ants; trails + step counts into the slab)
 *     barrier (k_peer_barrier: release/acquire epoch words in the peers' slabs) ; gather of every rank's step counts
 *     global ranking + best decision on every rank; the new best trail is read from its owner's HBM
 *     deposits, by the path the search is in (chosen identically on every rank, see WR_UPDATE_RANKSET):
 *       rank sets:      each rank builds the per-slot rank sets of ITS eligible ants (bits = global ranks), publishes its
 *                       row blocks; barrier; every rank ORs the peers' blocks into its table, evaporates its field and
 *                       applies the ordered chains — work per rank independent of the rank count
 *       sorted records: each rank generates the records of all eligible ants from their owners' trails, keeps, sorts and
 *                       applies the records of ITS slot slice while evaporating the whole field, lists the final values;
 *                       barrier; every rank overwrites the slots the others own with their final values
 *
 * Setting up, either
 *   (a) wr_comm_unique_id on one rank -> distribute the 128 bytes (any means) -> wr_acs_comm_init on every rank;
 *       wr_acs_begin then exchanges the slab handles itself (ncclAllGather; libnccl.so.2 is opened at run time), or
 *   (b) wr_acs_set_shard; after every wr_acs_begin: wr_acs_peer_export -> all_gather the 64-byte handles by your own
 *       means (welding_robot_b200/dist.py uses torch.distributed) -> wr_acs_peer_import.
 * raw_pointer / wr_acs_peer_set_pointers: the same for handles that live in ONE process on one GPU (tests); such
 * handles must run on different streams and be iterated in turn, one iteration at a time.
 * A sharded handle's stream must not be shared with work that could delay it behind a peer's (each barrier waits for
 * every rank); a barrier that is not reached within 20 s (WR_PEER_TIMEOUT_MS) is reported by wr_acs_sync. */
#define WR_COMM_ID_BYTES 128
int wr_comm_unique_id(void* id128);                                       /* ncclGetUniqueId */
int wr_acs_comm_init(wr_acs* a, const void* nccl_unique_id, int rank, int nranks);   /* before wr_acs_begin */
int wr_acs_set_shard(wr_acs* a, int rank, int nranks);                    /* before wr_acs_begin */
int wr_acs_peer_export(wr_acs* a, void* ipc_handle, void** raw_pointer);  /* ipc_handle: 64 bytes (cudaIpcMemHandle_t) */
int wr_acs_peer_import(wr_acs* a, const void* all_ipc_handles);           /* nranks x 64 bytes in rank order */
int wr_acs_peer_set_pointers(wr_acs* a, void* const* all_raw_pointers);

/* ------------------------------------------------------------------------------------------
 * Seam ordering — replaces ACS_GTSP (core/ACS_GTSP.hpp), batched: B independent colonies on
 * the same distance matrix, colony b drawing from Philox stream (seed, colony_first + b).
 * ---------------------------------------------------------------------------------------- */
/* dis: n*n doubles, symmetric, diagonal ignored (readFromGraphFile :224-253 + init_param :187-218);
 * cnt = the edge count used in tau0 = cnt/(sum*n) (:249). */
int wr_gtsp_create(const double* dis, int n, int cnt, int batch, int colony_first, uint64_t seed, wr_gtsp** out);
int wr_gtsp_destroy(wr_gtsp* g);
int wr_gtsp_iterate(wr_gtsp* g, int iterations);   /* loop body of computeSolution :261-276, no early stop */
/* computeSolution :255-284 for EVERY colony of the handle, on the device.  Colony b repeats the loop body until it has run
 * max_iterations iterations (0: the reference's MAX_itera = n*n) or until more than n consecutive iterations did not
 * lower its best (bad_times > city_num, :263-275; `last` and bad_times start afresh with every call, like the reference's
 * locals) -- each colony on its own.  iterations[b] (optional): iterations colony b ran in this call.
 * best_L_history (optional, [batch][max_iterations or n*n]): colony b's best L after each of its iterations (what the facade
 * prints); entries past iterations[b] are not written.  *best_colony (optional): the colony with the lowest best L, lowest
 * index on ties.  Later wr_gtsp_iterate / wr_gtsp_solve calls continue every colony from its own iteration count. */
int wr_gtsp_solve(wr_gtsp* g, int max_iterations, int* iterations, double* best_L_history, int* best_colony);
int wr_gtsp_sync(wr_gtsp* g);
/* best tour of colony b: 2 ints per edge (r, s), n edges (closing edge last); L excludes the
 * closing edge (ACS_Tour::calc :36-44). */
int wr_gtsp_best(wr_gtsp* g, int colony, int* tour_pairs, int* nedges, double* L);
int wr_gtsp_download_pheromone(wr_gtsp* g, int colony, double* out); /* n*n */
int wr_gtsp_tau0(wr_gtsp* g, double* tau0);
int wr_gtsp_kernel_ms(wr_gtsp* g, float out[3]); /* [0] info rebuild [1] construction [2] update */

/* ------------------------------------------------------------------------------------------
 * Trajectory smoothing — replaces BS_Basic<float, 3, DEGREE, CI, CF> (core/BSplineBasic.h) as
 * main.cpp:299-300 and :337-338 use it: SetParam (:70-76) on the host, getCurvePoint (:85-111)
 * for m sample times on the GPU.  init / fin: 3*(ci+1) / 3*(cf+1) floats (position, velocity,
 * acceleration); middle: n_middle rows of middle_stride floats, the first three of each are used
 * (main.cpp:325-334 passes rows of nine).  ok[i] (optional) = getCurvePoint's return value; the
 * out row of a failed call keeps the caller's contents, as `res` does in the demo.  knots_out
 * (degree+n_middle+ci+cf+3 floats) and cps_out ((n_middle+2+ci+cf)*3 floats) are optional.
 * degree <= 5, ci, cf <= min(2, degree).  Host pointers. */
int wr_bspline_eval(int degree, int ci, int cf, const float* init, const float* fin, const float* middle, int n_middle, int middle_stride,
                    float fin_time, const float* u, int m, float* out, unsigned char* ok, float* knots_out, float* cps_out);

#ifdef __cplusplus
}
#endif
#endif /* WR_GPU_H */
