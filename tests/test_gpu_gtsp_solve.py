"""GPU: seam ordering run to convergence on the device (wr_gtsp_solve, computeSolution ACS_GTSP.hpp:255-284) against the CPU
oracle.  Colony b of a solve is oracle.Gtsp(D, seed, colony_id=first + b).iterate(cap, early_stop=True): same iteration count,
tour, L and pheromone matrix bit for bit, and its best L after every iteration."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

SLICE = 32   # kGtspSolveSlice (csrc/gtsp.cu): iterations per solve launch


def matrix(n, seed):
    P = np.random.default_rng(seed).random((n, 3))
    D = np.sqrt(((P[:, None] - P[None]) ** 2).sum(-1))
    return np.array([[float("%.6f" % v) for v in row] for row in D])   # as a graph file would carry it


def handle(D, seed, batch, first):
    import welding_robot_b200 as wr
    n = D.shape[0]
    g = wr.ACS_GTSP(seed=seed)
    g.dis, g.city_num, g.cnt = D, n, n * (n - 1) // 2
    g._create(batch, first)
    return g


class Colony:
    """One oracle colony, plus a twin stepped one iteration at a time for the best L after each iteration."""

    def __init__(self, oracle, D, seed, cid):
        self.T = oracle.Gtsp(D, seed=seed, colony_id=cid)
        self.H = oracle.Gtsp(D, seed=seed, colony_id=cid)

    def solve(self, cap):
        ran = self.T.iterate(cap, early_stop=True)
        hist = []
        for _ in range(ran):
            self.H.iterate(1)
            hist.append(self.H.best()[1])
        return ran, np.array(hist)

    def iterate(self, k):
        self.T.iterate(k)
        self.H.iterate(k)


def assert_colony(g, b, T):
    tour, L = T.best()
    gt, gL = g.best(b)
    assert np.array_equal(gt, tour), b
    assert gL == L, b
    assert np.array_equal(g.pheromone(b).view(np.uint64), T.pheromone().view(np.uint64)), b


def check_solve(g, cols, cap):
    ran, hist, bc = g.solve(cap)
    n = g.city_num
    for b, col in enumerate(cols):
        r, h = col.solve(cap if cap > 0 else n * n)
        assert ran[b] == r, (b, ran[b], r)
        assert np.array_equal(hist[b, :r].view(np.uint64), h.view(np.uint64)), b
        assert_colony(g, b, col.T)
    Ls = [c.T.best()[1] for c in cols]
    assert bc == int(np.argmin(Ls))
    return ran


@pytest.mark.parametrize("n,batch,first,seed", [(5, 8, 0, 1), (12, 6, 3, 2), (33, 4, 0, 5), (64, 3, 7, 9)])
def test_solve_stops_by_stagnation(oracle, n, batch, first, seed):
    D = matrix(n, n)
    g = handle(D, seed, batch, first)
    cols = [Colony(oracle, D, seed, first + b) for b in range(batch)]
    ran = check_solve(g, cols, 0)
    assert (ran < n * n).all()             # every colony stopped by the rule, not the cap
    if n == 33:
        # colonies of one batch stop at different iterations; one runs past two launches and stops inside a third
        assert len(set(ran.tolist())) == batch
        assert any(r > 2 * SLICE and r % SLICE for r in ran)
    # continuing: every colony's next draws are keyed by its own iteration count
    g.iterate(5)
    for b, col in enumerate(cols):
        col.iterate(5)
        assert_colony(g, b, col.T)
    # a second solve starts `last` and bad_times afresh, like the reference's locals
    check_solve(g, cols, 0)
    ms = g.kernelMs()
    assert ms["construct"] > 0


@pytest.mark.parametrize("n,batch,cap", [(256, 2, 20), (464, 2, 3)])
def test_solve_stops_at_the_cap(oracle, n, batch, cap):
    D = matrix(n, n)
    g = handle(D, 11, batch, 0)
    cols = [Colony(oracle, D, 11, b) for b in range(batch)]
    ran = check_solve(g, cols, cap)
    assert (ran == cap).all()


def test_solve_optional_outputs(oracle):
    """iterations, history and best_colony may each be NULL."""
    from welding_robot_b200 import _lib
    n = 33
    D = matrix(n, n)
    g = handle(D, 5, 4, 0)
    assert _lib.lib().wr_gtsp_solve(g._g, 0, None, None, None) == 0
    for b in range(4):
        T = oracle.Gtsp(D, seed=5, colony_id=b)
        T.iterate(n * n, early_stop=True)
        assert_colony(g, b, T)


def test_best_colony_ties_take_the_lowest_index(oracle):
    n = 9
    D = matrix(n, 109)
    g = handle(D, 2, 8, 0)
    Ls = []
    for b in range(8):
        T = oracle.Gtsp(D, seed=2, colony_id=b)
        T.iterate(n * n, early_stop=True)
        Ls.append(T.best()[1])
    ties = [b for b in range(8) if Ls[b] == min(Ls)]
    assert len(ties) > 1 and ties[0] > 0      # several colonies share the optimum, colony 0 is not one of them
    _, _, bc = g.solve()
    assert bc == ties[0]


def test_solve_rejects_negative_cap():
    import welding_robot_b200 as wr
    g = handle(matrix(5, 5), 0, 2, 0)
    with pytest.raises(wr.WrError) as e:
        g.solve(-1)
    assert e.value.status == -1   # WR_ERR_INVALID


def write_graph(path, D):
    n = D.shape[0]
    with open(path, "w") as fp:
        fp.write("%d %d\n" % (n, n * (n - 1) // 2))
        for i in range(n):
            for j in range(i + 1, n):
                fp.write("%.6f\n" % D[i, j])


def facade_python(path, seed, colonies, capsys):
    import welding_robot_b200 as wr
    capsys.readouterr()
    g = wr.ACS_GTSP(seed=seed, colonies=colonies)
    assert g.readFromGraphFile(str(path)) and g.computeSolution()
    return g, capsys.readouterr().out


@pytest.fixture(scope="module")
def cpp_exe(tmp_path_factory):
    from welding_robot_b200 import _lib
    exe = str(tmp_path_factory.mktemp("cpp") / "gtsp_solve_test")
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.run(["g++", "-std=c++14", "-O1", "-Wall", "-I" + os.path.join(ROOT, "include", "welding_robot_b200"),
                    os.path.join(ROOT, "tests", "cpp", "gtsp_solve_test.cpp"), "-o", exe, "-L" + libdir, "-lwrgpu",
                    "-Wl,-rpath," + libdir, "-ldl", "-lpthread", "-lrt"], check=True)
    return exe


def test_facades_multi_start(oracle, tmp_path, capsys, cpp_exe):
    """computeSolution with 8 colonies reports colony 1's tour and history (the lowest best L, colonies 2, 5, 6, 7 tie with
    it); the C++ facade prints the same bytes as the Python one, with 8 colonies and with the default single colony."""
    n = 9
    D = matrix(n, 109)
    f = tmp_path / "graph.in"
    write_graph(f, D)
    T = oracle.Gtsp(D, seed=2, colony_id=1)
    ran = T.iterate(n * n, early_stop=True)
    tour, L = T.best()
    g, out = facade_python(f, 2, 8, capsys)
    assert np.array_equal(g.best_path, tour) and g.best_L == L
    lines = [l for l in out.splitlines() if l.startswith("iteration ")]
    assert len(lines) == ran and lines[-1].startswith("iteration %d:Best so far" % (ran - 1))
    assert "Best in all = %.2f" % L in out
    assert "->".join(str(r + 1) for r, _ in tour) + "->%d" % (tour[-1][1] + 1) in out
    for colonies in (8, 1):
        _, py = facade_python(f, 2, colonies, capsys)
        r = subprocess.run([cpp_exe, str(f), "2", str(colonies)], capture_output=True, timeout=600)   # bytes: keep the "\r" of each line
        assert r.returncode == 0, r.stderr[-2000:]
        assert r.stdout.decode() == py, colonies


def test_facade_single_colony_is_colony_zero(oracle, tmp_path, capsys):
    """colonies = 1 (the default): the reference's single run, whose history is the oracle's best after each iteration."""
    n = 33
    D = matrix(n, 33)
    f = tmp_path / "graph.in"
    write_graph(f, D)
    col = Colony(oracle, D, 5, 0)
    ran, hist = col.solve(n * n)
    g, out = facade_python(f, 5, 1, capsys)
    lines = [l for l in out.splitlines() if l.startswith("iteration ")]
    assert lines == ["iteration %d:Best so far = %.2f" % (i, h) for i, h in enumerate(hist)]
    assert_colony(g, 0, col.T)
