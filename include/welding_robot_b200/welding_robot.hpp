// welding_robot.hpp — C++ host-side facade of the B200-native ACS hot path.
//
// Source-compatible with the class surface main.cpp (reference, :33-35, :273-283) uses:
//   STLReader, GridMap<float>, ACS_Rank, ACS_GTSP, Agent<float>, ACS_Node<float>, Point3<T>,
//   Triangles<T>, Vertex3<T>
// with the same method names, argument meaning and printed messages, but every computation runs in
// libwrgpu.so (hand-written sm_100a CUDA kernels) behind the C ABI of include/wr_gpu.h.  Header-only;
// link with -lwrgpu.  Nothing here falls back to the CPU: a missing GPU surfaces as wr::Error.
//
// Differences a caller can observe (all documented in DESIGN.md):
//  * the node cuboid (Vertex3*** / ACS_Node***) is never built eagerly: ptr_grid_map() materialises
//    it on first use, and paths return ACS_Node objects created on demand (their adjacency vectors
//    stay empty) — at 512^3 the reference's cuboid would need ~38 GB of host memory;
//  * rand() is replaced by Philox keyed (seed; iteration, ant, step); the unstable std::sort of
//    ACSRank_3D.hpp:273 by the total order (L, ant index);
//  * the grid dump carries the global mesh box (the reference writes the last triangle's box,
//    model_grid_map.hpp:279) and the graph file a whole header (the reference's in-place rewrite,
//    ACSRank_3D.hpp:500-501, clobbers the first distance once there are >= 10 points);
//  * additions: ACS_Rank::params, begin()/iterate()/bestPath(), counters(); ACS_GTSP::setDistanceMatrix().
#pragma once
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <deque>
#include <fstream>
#include <functional>
#include <iostream>
#include <memory>
#include <set>
#include <stdexcept>
#include <type_traits>
#include <string>
#include <utility>
#include <vector>

#include "../wr_gpu.h"

#ifndef INF_FLOAT
#define INF_FLOAT (1.0 / 0.0)
#endif

namespace wr {
struct Error : std::runtime_error {
    int status;
    Error(int s, const std::string& m) : std::runtime_error(m), status(s) {}
};
inline void check(int status)
{
    if (status != WR_OK) throw Error(status, std::string(wr_last_error()));
}
}  // namespace wr

// ---- value types (model_grid_map.hpp:34-88) ------------------------------------------------------
template <class T>
class Point3 {
public:
    Point3() : x(0), y(0), z(0) {}
    Point3(T _x, T _y, T _z) : x(_x), y(_y), z(_z) {}
    T x, y, z;
    Point3<T> operator+(const Point3<T>& b) const { return Point3<T>(x + b.x, y + b.y, z + b.z); }
    Point3<T> operator-(const Point3<T>& b) const { return Point3<T>(x - b.x, y - b.y, z - b.z); }
    T norm() const { return sqrt(x * x + y * y + z * z); }
    static T manhattan_distance(const Point3<T>& a, const Point3<T>& b) { return (a.x - b.x) + (a.y - b.y) + (a.z - b.z); }
    static T euler_distance(const Point3<T>& a, const Point3<T>& b) { return (a - b).norm(); }
    static T dot(const Point3<T>& a, const Point3<T>& b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
};
typedef Point3<float> Point3f;
typedef Point3<int> Point3i;

template <class T>
struct Triangles {
    Point3<T> nor_vec;
    Point3<T> vertex[3];
    int trait;
};

template <class T>
class Vertex3 {
public:
    Point3<T> pt;
    bool isFree;
    unsigned long int id;
};

// ---- node-cuboid helpers (model_grid_map.hpp:90-138) ---------------------------------------------
// Same contract as the reference's three templates: matrix[z][y][x], the callback sees every (z, y, x) in z -> y -> x
// order, creat_* wants a NULL pointer and delete_* a live one.  The storage differs: one contiguous block of T plus two
// pointer tables (three allocations instead of rz*ry + rz + 1), so a sweep over the cuboid is a linear scan.
template <class T>
void creat_all_nodes(T***& matrix, int rx, int ry, int rz, std::function<void(int, int, int)> f)
{
    if (matrix != NULL) throw wr::Error(WR_ERR_STATE, "creat_all_nodes: matrix already exists");
    T* cells = new T[(size_t)rx * ry * rz];
    T** rows = new T*[(size_t)ry * rz];
    matrix = new T**[rz];
    for (int z = 0; z < rz; z++) {
        matrix[z] = rows + (size_t)z * ry;
        for (int y = 0; y < ry; y++) rows[(size_t)z * ry + y] = cells + ((size_t)z * ry + y) * rx;
    }
    for (int z = 0; z < rz; z++)
        for (int y = 0; y < ry; y++)
            for (int x = 0; x < rx; x++) f(z, y, x);
}

template <class T>
void for_each_nodes(T***& matrix, int rx, int ry, int rz, std::function<void(int, int, int)> f)
{
    if (matrix == NULL) throw wr::Error(WR_ERR_STATE, "for_each_nodes: no matrix");
    for (int z = 0; z < rz; z++)
        for (int y = 0; y < ry; y++)
            for (int x = 0; x < rx; x++) f(z, y, x);
}

template <class T>
void delete_all_nodes(T***& matrix, int /*rx*/, int /*ry*/, int /*rz*/)
{
    if (matrix == NULL) throw wr::Error(WR_ERR_STATE, "delete_all_nodes: no matrix");
    delete[] matrix[0][0];   // the cells
    delete[] matrix[0];      // the row table
    delete[] matrix;
    matrix = NULL;
}

template <class T>
struct _Inf_of_Points_t {
    _Inf_of_Points_t() {}
    _Inf_of_Points_t(T a, T b, T c) : distance(a), pheromone(b), info(c) {}
    T distance, pheromone, info;
};

template <class T>
class ACS_Node : public Vertex3<T> {
public:
    std::vector<ACS_Node<T>*> adjacency_nodes;        // left empty: adjacency lives in HBM as index arithmetic
    std::vector<_Inf_of_Points_t<T>> adjacency_infos; // left empty: the pheromone field lives in HBM
};

// ---- STLReader (read_STL.hpp:23-175) -----------------------------------------------------------
class STLReader {
public:
    bool readFile(std::string file_name)
    {
        std::ifstream f(file_name.c_str(), std::ios::binary);
        if (!f) throw wr::Error(WR_ERR_FORMAT, "File error: " + file_name);   // the reference exit(1)s (:36-37)
        std::vector<char> buf((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
        int n = 0;
        wr::check(wr_stl_parse(reinterpret_cast<const uint8_t*>(buf.data()), buf.size(), nullptr, 0, &n));
        std::vector<float> t((size_t)n * 12);
        wr::check(wr_stl_parse(reinterpret_cast<const uint8_t*>(buf.data()), buf.size(), t.data(), n, &n));
        triangleMesh.resize(n);
        for (int i = 0; i < n; i++) {
            const float* p = &t[(size_t)i * 12];
            triangleMesh[i].nor_vec = Point3f(p[0], p[1], p[2]);
            for (int j = 0; j < 3; j++) triangleMesh[i].vertex[j] = Point3f(p[3 + 3 * j], p[4 + 3 * j], p[5 + 3 * j]);
            triangleMesh[i].trait = 0;
        }
        unTriangles = (unsigned)n;
        return true;
    }
    int NumTri() { return (int)unTriangles; }
    std::vector<Point3f>& PointList() { return pointList; }
    const std::vector<Triangles<float>>& TriangleList() { return triangleMesh; }

private:
    std::vector<Point3f> pointList;
    std::vector<Triangles<float>> triangleMesh;
    unsigned int unTriangles = 0;
};

// ---- GridMap (model_grid_map.hpp:140-421) ------------------------------------------------------
template <class T>
class GridMap {
public:
    GridMap() {}
    GridMap(const GridMap&) = delete;
    GridMap& operator=(const GridMap&) = delete;
    virtual ~GridMap() { release_grid(); }

    Vertex3<T>*** creatGridMap(const std::vector<Triangles<T>>& mesh, T _precision, int _wall, std::string file_name = "")
    {
        static_assert(sizeof(T) == sizeof(float), "the device layer is float32, like the reference's only instantiation");
        release_grid();
        std::vector<float> t(mesh.size() * 12);
        for (size_t i = 0; i < mesh.size(); i++) {
            float* p = &t[i * 12];
            p[0] = mesh[i].nor_vec.x; p[1] = mesh[i].nor_vec.y; p[2] = mesh[i].nor_vec.z;
            for (int j = 0; j < 3; j++) { p[3 + 3 * j] = mesh[i].vertex[j].x; p[4 + 3 * j] = mesh[i].vertex[j].y; p[5 + 3 * j] = mesh[i].vertex[j].z; }
        }
        wr::check(wr_grid_create_from_triangles(t.data(), (int)mesh.size(), _precision, _wall, &grid_));
        adopt();
        float mn[3], mx[3];
        wr::check(wr_grid_bbox(grid_, mn, mx));
        printf("[Grid Map]max(%.2f, %.2f, %.2f), min(%.2f, %.2f, %.2f) \n", mx[0], mx[1], mx[2], mn[0], mn[1], mn[2]);
        printf("[Grid Map] %d triangles is scanned... \n", (int)mesh.size());
        printf("[Grid Map] %d nodes is created... \n", size_of_map());
        if (file_name != "") writeGridMap(file_name);
        printf("[Grid Map] Done! \r\n");
        // the reference returns its node cuboid (model_grid_map.hpp:297).  It is built here (24 B of host memory per
        // node) unless the caller switched it off; ptr_grid_map() builds it on first use either way.
        return materialise_cuboid ? ptr_grid_map() : nullptr;
    }

    // synthetic-grid entry point (an addition)
    void creatFromOccupancy(const std::vector<uint8_t>& isfree, const std::vector<float>& xs, const std::vector<float>& ys,
                            const std::vector<float>& zs, T _precision)
    {
        release_grid();
        wr::check(wr_grid_create_from_occupancy(isfree.data(), (int)xs.size(), (int)ys.size(), (int)zs.size(), xs.data(), ys.data(), zs.data(),
                                                _precision, &grid_));
        adopt();
    }

    void writeGridMap(const std::string& file_name)
    {   // layout of model_grid_map.hpp:277-291
        std::vector<uint8_t> free(size_of_map());
        wr::check(wr_grid_download_isfree(grid_, free.data(), free.size()));
        float mn[3], mx[3];
        wr::check(wr_grid_bbox(grid_, mn, mx));
        FILE* fp = fopen(file_name.c_str(), "w");
        if (!fp) throw wr::Error(WR_ERR_FORMAT, "cannot write " + file_name);
        fprintf(fp, "%d %d %d %d %f %d\n", size_of_map(), rangeX, rangeY, rangeZ, precision, wall);
        fprintf(fp, "%f %f %f %f %f %f\n", mn[0], mn[1], mn[2], mx[0], mx[1], mx[2]);
        size_t id = 0;
        for (int i = 0; i < rangeZ; i++)
            for (int j = 0; j < rangeY; j++) {
                for (int k = 0; k < rangeX; k++) fprintf(fp, "%d ", (int)free[id++]);
                fprintf(fp, "\n");
            }
        fclose(fp);
        printf("\n[Grid Map] Successfully write to %s \r\n", file_name.c_str());
    }

    void readGridMap(std::string file_name)
    {   // model_grid_map.hpp:300-356
        FILE* fp = fopen(file_name.c_str(), "r");
        if (fp == NULL) { std::cout << "[Grid Map] Failed to read file, skipping..." << std::endl; return; }
        int n = 0, rx = 0, ry = 0, rz = 0, w = 0;
        float p = 0, mn[3], mx[3];
        bool ok = fscanf(fp, "%d %d %d %d %f %d", &n, &rx, &ry, &rz, &p, &w) == 6 &&
                  fscanf(fp, "%f %f %f %f %f %f", &mn[0], &mn[1], &mn[2], &mx[0], &mx[1], &mx[2]) == 6 && rx > 0 && ry > 0 && rz > 0;
        if (!ok) { fclose(fp); throw wr::Error(WR_ERR_FORMAT, "malformed grid file " + file_name); }
        std::vector<uint8_t> free((size_t)rx * ry * rz);
        for (size_t i = 0; i < free.size(); i++) { int v = 1; if (fscanf(fp, "%d", &v) != 1) v = 1; free[i] = v != 0; }
        fclose(fp);
        std::vector<float> xs(rx), ys(ry), zs(rz);
        for (int i = 0; i < rx; i++) xs[i] = axis(i, rx, w, mn[0], mx[0], p);
        for (int i = 0; i < ry; i++) ys[i] = axis(i, ry, w, mn[1], mx[1], p);
        for (int i = 0; i < rz; i++) zs[i] = axis(i, rz, w, mn[2], mx[2], p);
        creatFromOccupancy(free, xs, ys, zs, p);
        wall = w;
        printf("\n[Grid Map] Successfully read grid map from %s \r\n", file_name.c_str());
    }

    // Built on first use; NULL before a grid exists.  24 B per node of host memory.
    Vertex3<T>*** ptr_grid_map() const
    {
        if (!grid_) return NULL;
        if (cuboid_.empty()) {
            GridMap* self = const_cast<GridMap*>(this);
            std::vector<uint8_t> free(size_of_map());
            wr::check(wr_grid_download_isfree(grid_, free.data(), free.size()));
            self->load_coords();
            self->nodes_.resize(free.size());
            self->rows_.resize((size_t)rangeZ * rangeY);
            self->cuboid_.resize(rangeZ);
            size_t id = 0;
            for (int z = 0; z < rangeZ; z++) {
                self->cuboid_[z] = &self->rows_[(size_t)z * rangeY];
                for (int y = 0; y < rangeY; y++) {
                    self->rows_[(size_t)z * rangeY + y] = &self->nodes_[id];
                    for (int x = 0; x < rangeX; x++, id++) {
                        self->nodes_[id].pt = Point3<T>(xs_[x], ys_[y], zs_[z]);
                        self->nodes_[id].isFree = free[id] != 0;
                        self->nodes_[id].id = id;
                    }
                }
            }
        }
        return const_cast<Vertex3<T>***>(cuboid_.data());
    }
    // additions: clearance (include/wr_gpu.h, "Clearance").  Squared INDEX distance of every node to the nearest occupied
    // node, z,y,x order; UINT32_MAX everywhere when none is occupied.
    std::vector<uint32_t> clearanceMap()
    {
        std::vector<uint32_t> d2((size_t)size_of_map());
        wr::check(wr_grid_clearance(grid_, d2.data(), d2.size()));
        return d2;
    }
    // nearest node per point (per axis argmin |p - c[i]| in double, lowest index on ties) and its d2; either output may be NULL
    void clearanceAt(const std::vector<Point3<T>>& pts, std::vector<int64_t>* ids, std::vector<uint32_t>* d2)
    {
        std::vector<float> xyz(3 * pts.size() + 3);
        for (size_t i = 0; i < pts.size(); i++) { xyz[3 * i] = pts[i].x; xyz[3 * i + 1] = pts[i].y; xyz[3 * i + 2] = pts[i].z; }
        if (ids) ids->resize(pts.size());
        if (d2) d2->resize(pts.size());
        wr::check(wr_grid_clearance_at(grid_, xyz.data(), (int)pts.size(), ids ? ids->data() : nullptr, d2 ? d2->data() : nullptr));
    }
    // replace the grid by its obstacles inflated by `radius` (world units): occupied iff d2 <= floor((radius / precision)^2).
    // precision and wall keep their values; an ACS_Rank releases its search handle (release_grid) and creates a new one on next use.
    void inflateGridMap(T radius)
    {
        const uint32_t r2 = radius_r2(radius, "inflateGridMap");
        wr_grid* inflated = nullptr;
        wr::check(wr_grid_inflate(grid_, r2, &inflated));
        const T p = precision;
        const int w = wall;
        release_grid();
        grid_ = inflated;
        adopt();
        precision = p; wall = w;
    }

    // addition: greedy line-of-sight shortcutting of node rows (include/wr_gpu.h, wr_grid_shortcut_paths), all rows in one
    // launch.  Segments keep clear of every node with d2 <= floor((radius / precision)^2) (radius 0: of occupied nodes); from
    // each waypoint the next is the furthest row node, at most max_span ahead (0: no bound), whose segment is clear, else the
    // next node (counted in `blocked`).
    struct ShortcutRow {
        std::vector<int64_t> ids;    // waypoint node ids
        std::vector<int32_t> keep;   // their indices into the row
        int blocked = 0;             // segments kept by the fallback
        double length = 0;           // world length of the waypoint polyline
    };
    std::vector<ShortcutRow> shortcutPaths(const std::vector<std::vector<int64_t>>& paths, T radius = 0, int max_span = 0)
    {
        const uint32_t r2 = radius_r2(radius, "shortcutPaths");
        const int nrows = (int)paths.size();
        std::vector<int64_t> off(paths.size() + 1, 0), ids;
        for (int p = 0; p < nrows; p++) {
            off[p + 1] = off[p] + (int64_t)paths[p].size();
            ids.insert(ids.end(), paths[p].begin(), paths[p].end());
        }
        std::vector<int32_t> keep(ids.size() + 1), nkeep(paths.size() + 1), blocked(paths.size() + 1);
        std::vector<double> length(paths.size() + 1);
        wr::check(wr_grid_shortcut_paths(grid_, ids.data(), off.data(), nrows, r2, max_span, keep.data(), nkeep.data(), blocked.data(),
                                         length.data()));
        std::vector<ShortcutRow> out(paths.size());
        for (int p = 0; p < nrows; p++) {
            out[p].keep.assign(keep.begin() + off[p], keep.begin() + off[p] + nkeep[p]);
            for (int32_t k : out[p].keep) out[p].ids.push_back(paths[p][k]);
            out[p].blocked = blocked[p];
            out[p].length = length[p];
        }
        return out;
    }

    int size_of_map() const { return rangeX * rangeY * rangeZ; }
    void plot_grid_map(int) {}   // plotting (model_grid_map.hpp:368-379) is out of scope
    void show_plot() {}

    T precision = 0;
    int wall = 0;
    int rangeX = 0, rangeY = 0, rangeZ = 0;
    bool materialise_cuboid = true;   // addition: false = creatGridMap returns NULL and leaves the cuboid to ptr_grid_map()

protected:
    wr_grid* grid_ = nullptr;
    std::vector<float> xs_, ys_, zs_;
    // a world radius as a squared index radius: floor((radius / precision)^2), saturating at UINT32_MAX
    uint32_t radius_r2(T radius, const char* who) const
    {
        if (!grid_) throw wr::Error(WR_ERR_STATE, std::string(who) + ": no grid map");
        if (!(radius >= 0)) throw wr::Error(WR_ERR_INVALID, std::string(who) + ": radius must be >= 0");
        const double r = (double)radius / (double)precision;
        const double r2 = floor(r * r);
        return r2 >= 4294967295.0 ? 0xffffffffu : (uint32_t)r2;
    }
    void load_coords()
    {
        if (!xs_.empty()) return;
        xs_.resize(rangeX); ys_.resize(rangeY); zs_.resize(rangeZ);
        wr::check(wr_grid_coords(grid_, xs_.data(), ys_.data(), zs_.data()));
    }
    Point3<T> node_point(unsigned long id)
    {
        load_coords();
        const unsigned long rxy = (unsigned long)rangeX * rangeY;
        return Point3<T>(xs_[(id % rxy) % rangeX], ys_[(id % rxy) / rangeX], zs_[id / rxy]);
    }
    virtual void release_grid()
    {
        if (grid_) wr_grid_destroy(grid_);
        grid_ = nullptr;
        xs_.clear(); ys_.clear(); zs_.clear(); nodes_.clear(); rows_.clear(); cuboid_.clear();
    }

private:
    std::vector<Vertex3<T>> nodes_;
    std::vector<Vertex3<T>*> rows_;
    std::vector<Vertex3<T>**> cuboid_;
    void adopt()
    {
        int d[3];
        wr::check(wr_grid_dims(grid_, d));
        rangeX = d[0]; rangeY = d[1]; rangeZ = d[2];
        float p; int w;
        wr::check(wr_grid_precision(grid_, &p, &w));
        precision = p; wall = w;
    }
    static float axis(int i, int range, int w, float mn, float mx, float p)
    {   // model_grid_map.hpp:204-205
        return i < w ? mn - (w - i) * p : (i >= (range - w) ? mx + (i - range + w) * p : mn + (i - w) * p);
    }
};

// ---- Agent (ACSRank_3D.hpp:62-109) ---------------------------------------------------------------
template <class T>
class Agent {
private:
    std::vector<ACS_Node<T>*> path;
    std::vector<int> node_index;

public:
    std::set<unsigned long int> tabu_list;
    T L = (T)INF_FLOAT;
    const std::vector<ACS_Node<T>*>* getPath() const { return &path; }
    const std::vector<int>* nodeIndex() const { return &node_index; }
    bool findPathNode(ACS_Node<T>* target)
    {
        for (auto node : path) if (target == node) return true;
        return false;
    }
    // filled by ACS_Rank from the device read-out
    void assign(const std::vector<ACS_Node<T>*>& p, const std::vector<int>& idx, T len)
    {
        path = p; node_index = idx; L = len;
        tabu_list.clear();
        for (auto n : p) tabu_list.insert(n->id);
    }
};

// ---- ACS_Rank (ACSRank_3D.hpp:111-599) -----------------------------------------------------------
class ACS_Rank : public GridMap<float> {
public:
    Agent<float>** best_matrix = NULL;
    std::vector<Point3<float>> route_points;
    wr_acs_params params;          // addition: colony parameters (defaults = the literals of :319-325)
    int max_iteration = 150;       // :322

    ACS_Rank() { wr_acs_default_params(&params); }
    ~ACS_Rank() override
    {
        release_acs();
        free_matrix();
    }

    void initFromGridMap()
    {   // :317-410
        if (!grid_) throw wr::Error(WR_ERR_STATE, "initFromGridMap: no grid map");
        release_acs();
        wr::check(wr_acs_create(grid_, &params, &acs_));
        printf("[ACS 3D] Created %d nodes, node cubiod [x: %d, y: %d, z: %d]\r\n", size_of_map(), rangeX, rangeY, rangeZ);
    }

    bool setPoints(Point3<float>& start, Point3<float>& end)
    {   // :537-565
        need();
        float s[3] = {start.x, start.y, start.z}, e[3] = {end.x, end.y, end.z};
        int64_t ids[2];
        int st = wr_acs_set_points(acs_, s, e, ids);
        if (st == WR_ERR_NOTFOUND) return false;
        wr::check(st);
        return true;
    }

    void checkRoutePoints()
    {   // :511-535
        for (size_t i = 0; i < route_points.size(); i++) {
            Point3<float> p = route_points[i];
            if (!setPoints(p, p))
                printf("[ACS 3D] Invalid route point, please reset point(%.3f, %.3f, %.3f) \n", p.x, p.y, p.z);
        }
        printf("[ACS 3D] %d route points have been checked. \n", (int)route_points.size());
    }

    // additions: explicit stepping (north_star: "iterate, best-path readout")
    void begin(float predict_path_len) { need(); wr::check(wr_acs_begin(acs_, predict_path_len)); }
    void iterate(int n = 1) { need(); wr::check(wr_acs_iterate(acs_, n)); }
    void computeSolution(float predict_path_len)
    {   // :220-305
        begin(predict_path_len);
        iterate(max_iteration);
        fetch_best(best_);
    }
    void reset() { need(); wr::check(wr_acs_reset(acs_)); }   // :307-315
    const Agent<float>* getSolution() const { return &best_; }   // :506-509
    const Agent<float>* bestPath()
    {
        fetch_best(best_);
        return &best_;
    }
    void counters(uint64_t out[9]) { need(); wr::check(wr_acs_counters(acs_, out)); }
    // additions: the colony sharded by ants over `nranks` processes (one GPU each).  `nccl_unique_id`: the WR_COMM_ID_BYTES
    // bytes rank 0 got from wr_comm_unique_id, handed to every rank by the caller's own means.  Call before computeSolution
    // / begin; iterate() and computeSolution() then run the sharded protocol (include/wr_gpu.h) with the same results.
    void commInit(const void* nccl_unique_id, int rank, int nranks) { need(); wr::check(wr_acs_comm_init(acs_, nccl_unique_id, rank, nranks)); }
    void setEndpoints(int64_t start_id, int64_t goal_id) { need(); wr::check(wr_acs_set_endpoints(acs_, start_id, goal_id)); }
    void sync() { need(); wr::check(wr_acs_sync(acs_)); }
    std::vector<float> pheromone()
    {
        need();
        std::vector<float> tau((size_t)size_of_map() * (size_t)params.K);
        wr::check(wr_acs_download_pheromone(acs_, tau.data(), tau.size()));
        return tau;
    }
    std::vector<uint8_t> isFreeArray()
    {
        std::vector<uint8_t> f((size_t)size_of_map());
        wr::check(wr_grid_download_isfree(grid_, f.data(), f.size()));
        return f;
    }
    wr_acs* handle() { need(); return acs_; }

    void searchBestPathOfPoints(float predict_path_len = 10, std::string read_file = "", std::string output_file = "")
    {   // :427-504
        int point_num = 0;
        if (read_file == "") {
            std::cout << "[ACS 3D] Please enter passing point number: ";
            std::cin >> point_num;
            route_points.resize(point_num);
            std::cout << "[ACS 3D] Please enter passing point in order: " << std::endl;
            for (int i = 0; i < point_num; i++) std::cin >> route_points[i].x >> route_points[i].y >> route_points[i].z;
        } else {
            FILE* fp = fopen(read_file.c_str(), "r");
            if (fp == NULL) { std::cout << "[ACS 3D] Failed to read file, reject to init." << std::endl; return; }
            if (fscanf(fp, "%d", &point_num) != 1 || point_num < 0) { fclose(fp); return; }
            route_points.resize(point_num);
            for (int i = 0; i < point_num; i++)
                if (fscanf(fp, "%f %f %f", &route_points[i].x, &route_points[i].y, &route_points[i].z) != 3) break;
            fclose(fp);
        }
        free_matrix();
        matrix_n_ = point_num;
        best_matrix = new Agent<float>*[point_num];
        for (int i = 0; i < point_num; i++) best_matrix[i] = new Agent<float>[point_num];
        initFromGridMap();
        checkRoutePoints();
        // the pair loop of :472-499 runs on the device: snap every point once, search all pairs up to the first one the
        // reference would reject, read everything back once
        std::vector<float> xyz(3 * (size_t)point_num + 3);
        for (int i = 0; i < point_num; i++) { xyz[3 * i] = route_points[i].x; xyz[3 * i + 1] = route_points[i].y; xyz[3 * i + 2] = route_points[i].z; }
        std::vector<int64_t> node(point_num + 1, -1);
        wr::check(wr_acs_snap_points(acs_, xyz.data(), point_num, node.data()));
        std::vector<std::pair<int, int>> pairs;
        for (int i = 0; i < point_num; i++) for (int j = i + 1; j < point_num; j++) pairs.push_back(std::make_pair(i, j));
        size_t good = 0;
        while (good < pairs.size() && node[pairs[good].first] >= 0 && node[pairs[good].second] >= 0) good++;
        std::vector<float> lens;
        if (good > 0) {
            std::vector<int64_t> s_ids(good), g_ids(good);
            std::vector<int> cnt(good);
            lens.resize(good);
            for (size_t q = 0; q < good; q++) { s_ids[q] = node[pairs[q].first]; g_ids[q] = node[pairs[q].second]; }
            // all pairs advance concurrently (wr_acs_search_batch: same results as the pair-by-pair loop, bit for bit);
            // the paths are fetched by their true length afterwards
            wr::check(wr_acs_search_batch(acs_, s_ids.data(), g_ids.data(), (int)good, predict_path_len, max_iteration, lens.data(), cnt.data(), nullptr, nullptr, 0));
            for (size_t q = 0; q < good; q++) {
                const int i = pairs[q].first, j = pairs[q].second;
                std::vector<int64_t> ids((size_t)std::max(cnt[q], 1));
                std::vector<int> dirs((size_t)std::max(cnt[q], 1));
                int m = 0; float Lq = 0;
                wr::check(wr_acs_result_path(acs_, (int)q, ids.data(), dirs.data(), cnt[q], &m, &Lq));
                make_agent(best_, ids.data(), dirs.data(), cnt[q], lens[q]);
                best_matrix[i][j] = best_;
                best_matrix[j][i] = best_;
                printf("[ACS 3D] <Point (%.3f, %.3f, %.3f) : Point (%.3f, %.3f, %.3f)> Path length: %.3f\r\n", route_points[i].x,
                       route_points[i].y, route_points[i].z, route_points[j].x, route_points[j].y, route_points[j].z, best_.L);
            }
        }
        if (good < pairs.size()) {
            const int i = pairs[good].first, j = pairs[good].second;
            printf("[ACS 3D] Wrong point : (%.3f, %.3f, %.3f) or (%.3f, %.3f, %.3f), program will exit immediately \r\n",
                   route_points[i].x, route_points[i].y, route_points[i].z, route_points[j].x, route_points[j].y, route_points[j].z);
            return;
        }
        if (output_file != "") {
            FILE* fp = fopen(output_file.c_str(), "w");
            if (fp) {
                fprintf(fp, "%d %d\n", point_num, (int)lens.size());
                for (float L : lens) fprintf(fp, "%.3f\n", L);
                fclose(fp);
                printf("[ACS 3D] %d Result has been written to \"%s\" \r\n", (int)lens.size(), output_file.c_str());
            }
        }
    }

    // addition: best_matrix with every best path shortcut (shortcutPaths, one launch for all pairs): Agents whose path is the
    // waypoint nodes, with no node_index and L = the waypoint polyline's world length; read_all_segments stitches it like
    // best_matrix.  Entries without a path are copied as they are.  Owned by this object and freed with best_matrix (by the
    // next searchBestPathOfPoints or shortcutBestMatrix, or the destructor).
    Agent<float>** shortcutBestMatrix(float radius = 0, int max_span = 0)
    {
        if (!best_matrix) throw wr::Error(WR_ERR_STATE, "shortcutBestMatrix: no best_matrix (run searchBestPathOfPoints first)");
        std::vector<std::pair<int, int>> pairs;
        std::vector<std::vector<int64_t>> rows;
        for (int i = 0; i < matrix_n_; i++)
            for (int j = i + 1; j < matrix_n_; j++) {
                const std::vector<ACS_Node<float>*>* path = best_matrix[i][j].getPath();
                if (path->empty()) continue;
                pairs.push_back(std::make_pair(i, j));
                rows.emplace_back();
                for (auto nd : *path) rows.back().push_back((int64_t)nd->id);
            }
        const std::vector<ShortcutRow> res = shortcutPaths(rows, radius, max_span);
        free_shortcut_matrix();
        shortcut_matrix_ = new Agent<float>*[matrix_n_];
        for (int i = 0; i < matrix_n_; i++) {
            shortcut_matrix_[i] = new Agent<float>[matrix_n_];
            for (int j = 0; j < matrix_n_; j++) shortcut_matrix_[i][j] = best_matrix[i][j];
        }
        for (size_t q = 0; q < pairs.size(); q++) {
            const int i = pairs[q].first, j = pairs[q].second;
            make_agent(shortcut_matrix_[i][j], res[q].ids.data(), nullptr, (int)res[q].ids.size(), (float)res[q].length);
            shortcut_matrix_[j][i] = shortcut_matrix_[i][j];
        }
        return shortcut_matrix_;
    }

    void plot_path(Agent<float>&, int) {}   // :567-598, plotting out of scope
    void plot_route_point(int) {}

protected:
    void release_grid() override
    {
        release_acs();
        GridMap<float>::release_grid();
    }

private:
    wr_acs* acs_ = nullptr;
    Agent<float> best_;
    std::deque<ACS_Node<float>> pool_;   // nodes handed out through paths; stable addresses for the object's lifetime
    int matrix_n_ = 0;
    Agent<float>** shortcut_matrix_ = NULL;

    void need() { if (!acs_) initFromGridMap(); }
    void release_acs()
    {
        if (acs_) wr_acs_destroy(acs_);
        acs_ = nullptr;
    }
    void free_shortcut_matrix()
    {
        if (!shortcut_matrix_) return;
        for (int i = 0; i < matrix_n_; i++) delete[] shortcut_matrix_[i];
        delete[] shortcut_matrix_;
        shortcut_matrix_ = NULL;
    }
    void free_matrix()
    {
        free_shortcut_matrix();
        if (!best_matrix) return;
        for (int i = 0; i < matrix_n_; i++) delete[] best_matrix[i];
        delete[] best_matrix;
        best_matrix = NULL;
    }
    // dirs == NULL: a path of waypoints, which has no node_index
    void make_agent(Agent<float>& out, const int64_t* ids, const int* dirs, int n, float L)
    {
        std::vector<ACS_Node<float>*> p;
        for (int i = 0; i < n; i++) {
            pool_.emplace_back();
            ACS_Node<float>& nd = pool_.back();
            nd.id = (unsigned long)ids[i]; nd.isFree = true; nd.pt = node_point(nd.id);
            p.push_back(&nd);
        }
        std::vector<int> d;
        if (dirs) d.assign(dirs, dirs + (n > 0 ? n - 1 : 0));
        out.assign(p, d, L);
    }
    void fetch_best(Agent<float>& out)
    {
        need();
        int n = 0; float L = 0;
        wr::check(wr_acs_best(acs_, nullptr, nullptr, 0, &n, &L));
        std::vector<int64_t> ids(n > 0 ? n : 1);
        std::vector<int> dirs(n > 0 ? n : 1);
        if (n > 0) wr::check(wr_acs_best(acs_, ids.data(), dirs.data(), n, &n, &L));
        make_agent(out, ids.data(), dirs.data(), n, L);
    }
};

// ---- ACS_GTSP (ACS_GTSP.hpp:82-328) ----------------------------------------------------------------
class ACS_GTSP {
public:
    std::vector<float> g_path_x, g_path_y, g_path_z;
    uint64_t seed = 0;   // addition
    int colonies = 1;    // addition: colonies setDistanceMatrix creates; computeSolution keeps the best one's tour

    ~ACS_GTSP() { if (g_) wr_gtsp_destroy(g_); }

    bool readFromGraphFile(std::string filename)
    {   // :224-253
        FILE* fp = fopen(filename.c_str(), "r");
        if (!fp) return false;
        int n = 0, cnt = 0;
        if (fscanf(fp, "%d %d", &n, &cnt) != 2 || n < 2) { fclose(fp); return false; }
        std::vector<double> dis((size_t)n * n, 0.0);
        for (int i = 0; i < n; i++)
            for (int j = i + 1; j < n; j++) {
                double v = 0;
                if (fscanf(fp, "%lf", &v) != 1) { fclose(fp); return false; }
                dis[(size_t)i * n + j] = dis[(size_t)j * n + i] = v;
                printf("distance: %lf \r\n", v);
            }
        fclose(fp);
        return setDistanceMatrix(dis, n, cnt);
    }
    bool setDistanceMatrix(const std::vector<double>& dis, int n, int cnt)
    {
        if (g_) wr_gtsp_destroy(g_);
        g_ = nullptr;
        city_num = n;
        wr::check(wr_gtsp_create(dis.data(), n, cnt, colonies, 0, seed, &g_));
        batch_ = colonies;
        init_flag = true;
        best_L = 0x3f3f3f3f;
        return true;
    }
    bool computeSolution()
    {   // :255-284, every colony on the device with its own stopping rule
        if (!init_flag) return false;
        const int cap = city_num * city_num;
        std::vector<int> ran(batch_);
        // left uninitialised: only the pages up to each colony's iteration count are ever touched
        std::unique_ptr<double[]> hist(new double[(size_t)batch_ * cap]);
        int b = 0;
        wr::check(wr_gtsp_solve(g_, cap, ran.data(), hist.get(), &b));
        for (int index_itera = 0; index_itera < ran[b]; index_itera++)
            printf("iteration %d:Best so far = %.2lf\n", index_itera, hist[(size_t)b * cap + index_itera]);
        fetch(b);
        printf("Best in all = %.2lf\n", best_L);
        for (size_t i = 0; i < best_path.size(); i++) printf("%d->", best_path[i].first + 1);
        if (!best_path.empty()) printf("%d\n", best_path.back().second + 1);
        return true;
    }
    void read_all_segments(Agent<float>**& best_matrix)
    {   // :286-298
        for (size_t i = 1; i < best_path.size(); i++) read_segment(best_matrix, (int)i);
    }
    void read_segment(Agent<float>** best_matrix, int i)
    {   // :303-312 (i starts from 1)
        const std::vector<ACS_Node<float>*>* segment = best_matrix[best_path[i - 1].first][best_path[i - 1].second].getPath();
        for (size_t j = 0; j < segment->size(); j++) {
            g_path_x.push_back((*segment)[j]->pt.x);
            g_path_y.push_back((*segment)[j]->pt.y);
            g_path_z.push_back((*segment)[j]->pt.z);
        }
    }
    int path_segment_nums() { return (int)best_path.size() - 1; }
    void plot_route_path(int) {}
    const std::vector<std::pair<int, int>>& bestTour() const { return best_path; }
    double bestLength() const { return best_L; }

private:
    wr_gtsp* g_ = nullptr;
    int city_num = 0;
    int batch_ = 0;
    bool init_flag = false;
    std::vector<std::pair<int, int>> best_path;
    double best_L = 0x3f3f3f3f;
    void fetch(int colony)
    {
        std::vector<int> t((size_t)2 * city_num);
        int ne = 0;
        wr::check(wr_gtsp_best(g_, colony, t.data(), &ne, &best_L));
        best_path.resize(ne);
        for (int i = 0; i < ne; i++) best_path[i] = std::make_pair(t[2 * i], t[2 * i + 1]);
    }
};

// ---- BS_Basic (BSplineBasic.h:33-120): trajectory smoothing of the stitched path (main.cpp:287-352) ---------------------------
// Same template parameters and SetParam as the reference (T = float, DIM = 3: what main.cpp instantiates); the curve is evaluated
// for a whole vector of times in one kernel launch (getCurvePoints) — the demo's wall-clock sampling loop (main.cpp:309-320)
// becomes a list of times.  getCurvePoint(u, ret) is kept for source compatibility (one launch per call).
template <typename T, int DIM, int DEGREE, int CONST_LEVEL_INI, int CONST_LEVEL_FIN>
class BS_Basic {
    static_assert(std::is_same<T, float>::value && DIM == 3, "the GPU path implements BS_Basic<float, 3, ...> (main.cpp:299, :337)");

public:
    explicit BS_Basic(int num_middle) : NUM_MIDDLE(num_middle)
    {
        if (num_knots() < 2 * (DEGREE + 1)) printf("Invalid setup (num_knots, degree): %d, %d\n", num_knots(), DEGREE);   // :54-56
    }
    bool SetParam(T* init, T* fin, T** middle_pt, T fin_time)
    {   // :70-76
        init_.assign(init, init + DIM * (CONST_LEVEL_INI + 1));
        fin_.assign(fin, fin + DIM * (CONST_LEVEL_FIN + 1));
        mid_.resize((size_t)NUM_MIDDLE * DIM);
        for (int i = 0; i < NUM_MIDDLE; i++)
            for (int j = 0; j < DIM; j++) mid_[(size_t)i * DIM + j] = middle_pt[i][j];   // _CalcCPoints :441-447 copies DIM values per point
        tf_ = fin_time;
        knots_.assign(num_knots(), 0.f);
        cps_.assign((size_t)num_cps() * DIM, 0.f);
        return eval(nullptr, 0, nullptr, nullptr);
    }
    // getCurvePoint (:85-111) at every time of `u`; out: m rows of DIM; ok[i] (optional) = its return value
    bool getCurvePoints(const std::vector<T>& u, std::vector<T>& out, std::vector<unsigned char>* ok = nullptr)
    {
        out.resize(u.size() * DIM);
        std::vector<unsigned char> flags(u.size());
        const bool r = eval(u.data(), (int)u.size(), out.data(), flags.data());
        if (ok) *ok = flags;
        return r;
    }
    bool getCurvePoint(T u, T* ret)
    {
        unsigned char f = 0;
        T tmp[DIM];
        for (int i = 0; i < DIM; i++) tmp[i] = ret[i];
        if (!eval(&u, 1, tmp, &f) || !f) return false;
        for (int i = 0; i < DIM; i++) ret[i] = tmp[i];
        return true;
    }
    const std::vector<T>& knots() const { return knots_; }
    const std::vector<T>& controlPoints() const { return cps_; }

private:
    int NUM_MIDDLE;
    T tf_ = 0;
    std::vector<T> init_, fin_, mid_, knots_, cps_;
    int num_knots() const { return DEGREE + NUM_MIDDLE + 2 + CONST_LEVEL_INI + CONST_LEVEL_FIN + 1; }
    int num_cps() const { return NUM_MIDDLE + 2 + CONST_LEVEL_INI + CONST_LEVEL_FIN; }
    bool eval(const T* u, int m, T* out, unsigned char* ok)
    {
        wr::check(wr_bspline_eval(DEGREE, CONST_LEVEL_INI, CONST_LEVEL_FIN, init_.data(), fin_.data(), mid_.data(), NUM_MIDDLE, DIM, tf_, u, m, out, ok,
                                  knots_.data(), cps_.data()));
        return true;
    }
};
