// GPU test of the C++ facade's clearance methods (GridMap<T>::clearanceMap / clearanceAt / inflateGridMap): voxelises an STL at
// (0.005, wall 10), inflates it by one precision, searches all pairs of the weld points on the inflated grid and prints, on lines
// that start with "clearance ", the occupied counts, per best path its minimum clearance on the plain grid (by node id) and the
// minimum that clearanceAt reports for its node coordinates on the inflated grid, and the length of the first pair's path.  Usage: clearance_test <stl file> <weld points file>
#include <stdio.h>

#include <algorithm>

#include "welding_robot.hpp"

int main(int argc, char** argv)
{
    if (argc < 3) { fprintf(stderr, "usage: %s <stl file> <weld points file>\n", argv[0]); return 2; }
    try {
        STLReader model;
        model.readFile(argv[1]);
        ACS_Rank search;
        search.params.seed = 0;
        search.creatGridMap(model.TriangleList(), 0.005f, 10);
        const std::vector<uint32_t> plain = search.clearanceMap();
        search.initFromGridMap();
        search.inflateGridMap(0.005f);   // r2 = 1; releases the search handle
        const std::vector<uint32_t> thick = search.clearanceMap();
        printf("clearance occupied %ld inflated %ld\n", (long)std::count(plain.begin(), plain.end(), 0u),
               (long)std::count(thick.begin(), thick.end(), 0u));
        search.searchBestPathOfPoints(0.5f, argv[2], "");
        const int n = (int)search.route_points.size();
        for (int i = 0; i < n; i++)
            for (int j = i + 1; j < n; j++) {
                const std::vector<ACS_Node<float>*>* path = search.best_matrix[i][j].getPath();
                std::vector<Point3<float>> pts;
                for (size_t k = 0; k < path->size(); k++) pts.push_back((*path)[k]->pt);
                std::vector<int64_t> ids;
                std::vector<uint32_t> d2;
                search.clearanceAt(pts, &ids, &d2);
                uint32_t mn = 0xffffffffu, at = 0xffffffffu;
                for (size_t k = 0; k < path->size(); k++) {
                    mn = std::min(mn, plain[(size_t)(*path)[k]->id]);
                    at = std::min(at, d2[k]);
                }
                printf("clearance pair %d %d min_d2 %u inflated_at %u\n", i, j, mn, at);
            }
        printf("clearance path 0 1 L %.6f\n", (double)search.best_matrix[0][1].L);
    } catch (const wr::Error& e) {
        fprintf(stderr, "wr::Error %d: %s\n", e.status, e.what());
        return 1;
    }
    return 0;
}
