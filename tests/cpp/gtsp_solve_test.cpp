// GPU test of the C++ facade's ACS_GTSP::computeSolution (ACS_GTSP.hpp:255-284): reads a graph file and prints what the
// facade prints.  Usage: gtsp_solve_test <graph file> <seed> <colonies>
#include <stdio.h>
#include <stdlib.h>

#include "welding_robot.hpp"

int main(int argc, char** argv)
{
    if (argc < 4) { fprintf(stderr, "usage: %s <graph file> <seed> <colonies>\n", argv[0]); return 2; }
    ACS_GTSP g;
    g.seed = strtoull(argv[2], nullptr, 10);
    g.colonies = atoi(argv[3]);
    if (!g.readFromGraphFile(argv[1]) || !g.computeSolution()) return 1;
    return 0;
}
