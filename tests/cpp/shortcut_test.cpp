// GPU test of the C++ facade's shortcutting (GridMap<T>::shortcutPaths, ACS_Rank::shortcutBestMatrix): voxelises an STL at
// (0.005, wall 10), searches all pairs of the weld points, shortcuts every best path at radius 0 and at one precision and
// prints, on lines that start with "shortcut ", per pair and radius the waypoint count, the fallback count and the length,
// then orders the seams and prints how many points read_all_segments stitches from best_matrix and from the shortcut matrix.
// Usage: shortcut_test <stl file> <weld points file> <graph file to write>
#include <stdio.h>

#include "welding_robot.hpp"

int main(int argc, char** argv)
{
    if (argc < 4) { fprintf(stderr, "usage: %s <stl file> <weld points file> <graph file>\n", argv[0]); return 2; }
    try {
        STLReader model;
        model.readFile(argv[1]);
        ACS_Rank search;
        search.params.seed = 0;
        search.creatGridMap(model.TriangleList(), 0.005f, 10);
        search.searchBestPathOfPoints(0.5f, argv[2], argv[3]);
        const int n = (int)search.route_points.size();
        std::vector<std::vector<int64_t>> rows;
        std::vector<std::pair<int, int>> pairs;
        for (int i = 0; i < n; i++)
            for (int j = i + 1; j < n; j++) {
                const std::vector<ACS_Node<float>*>* path = search.best_matrix[i][j].getPath();
                rows.emplace_back();
                for (auto nd : *path) rows.back().push_back((int64_t)nd->id);
                pairs.push_back(std::make_pair(i, j));
            }
        const float radii[2] = {0.0f, 0.005f};
        for (float radius : radii) {
            const std::vector<ACS_Rank::ShortcutRow> res = search.shortcutPaths(rows, radius);
            for (size_t q = 0; q < res.size(); q++)
                printf("shortcut pair %d %d radius %g nkeep %d blocked %d length %.17g\n", pairs[q].first, pairs[q].second, radius,
                       (int)res[q].keep.size(), res[q].blocked, res[q].length);
        }
        ACS_GTSP route;
        if (!route.readFromGraphFile(argv[3]) || !route.computeSolution()) { fprintf(stderr, "seam ordering failed\n"); return 1; }
        route.read_all_segments(search.best_matrix);
        const size_t full = route.g_path_x.size();
        Agent<float>** shortcut = search.shortcutBestMatrix(0.0f);
        route.g_path_x.clear(); route.g_path_y.clear(); route.g_path_z.clear();
        route.read_all_segments(shortcut);
        printf("shortcut stitched %zu of %zu\n", route.g_path_x.size(), full);
        printf("shortcut agent 0 1 nodes %zu dirs %zu L %.9g\n", shortcut[0][1].getPath()->size(), shortcut[0][1].nodeIndex()->size(),
               (double)shortcut[1][0].L);
    } catch (const wr::Error& e) {
        fprintf(stderr, "wr::Error %d: %s\n", e.status, e.what());
        return 1;
    }
    return 0;
}
