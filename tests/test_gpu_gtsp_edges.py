"""GPU: seam ordering (k_gtsp_iterate) against the CPU oracle where the roulette degenerates, bit for bit.

The reference draws rnd = u * (sum of `info` over the unvisited cities) and takes the first unvisited city whose prefix sum
is >= rnd; rnd == 0 therefore means the lowest unvisited city.  The kernel finds the 16-city check-point interval first, and
interval 0 always qualifies for rnd == 0 even when all its cities are visited.  rnd == 0 happens on a zero draw, on a zero
sum (an `inf` distance makes tau0 = 0; a distance near 1e60 underflows the heuristic) and on a subnormal sum that u * sum
rounds to 0.  Every case compares the best tour and L (including the
no-tour state), tau0 and the whole pheromone matrix; solve cases also the iteration counts and the best L after every
iteration.  Float64 values are compared as bit patterns with every NaN mapped to one pattern (x86 keeps the input NaN's
payload, the GPU returns its canonical NaN).
"""
import ctypes as C

import numpy as np
import pytest

from test_gpu_gtsp import matrix
from test_gpu_gtsp_solve import Colony

gpu = pytest.mark.gpu

NO_TOUR_L = float(0x3f3f3f3f)        # ACS_Tour::clean (ACS_GTSP.hpp:29-34): the best L while no tour has been found
STREAM_GTSP = 0x65700000             # Philox stream tag of colony 0 (oracle/philox.h)
TINY = np.finfo(np.float64).tiny     # smallest normal float64
ULP0 = 5e-324                        # smallest subnormal float64

# a zero draw: rand() == 0 for ant 14 at step 62 of iteration 0, colony 0 (Philox counter (0, 14, 62, STREAM_GTSP))
ZERO_SEED, ZERO_ANT, ZERO_STEP = 37284317, 14, 62


def bits(a):
    a = np.asarray(a, np.float64)
    b = np.ascontiguousarray(a).view(np.uint64).copy()
    b[np.isnan(a)] = 0x7FF8000000000000
    return b


def rand31(oracle, seed, iteration, ant, step, colony):
    ctr = np.array([iteration, ant, step, STREAM_GTSP + colony], np.uint32)
    key = np.array([seed & 0xFFFFFFFF, seed >> 32], np.uint32)
    out = np.zeros(4, np.uint32)
    oracle.lib().wro_philox(ctr.ctypes.data_as(C.c_void_p), key.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    return int(out[0]) >> 1


def pow6(x):
    """power<double>(x, 6) of ACS_GTSP.hpp:117-118, in its multiplication order."""
    ans, y = 1.0, 6
    while y:
        if y & 1:
            ans *= x
        x *= x
        y >>= 1
    return ans


def tau0(D):
    n = len(D)
    tmp = 0.0
    for i in range(n):
        for j in range(i + 1, n):
            tmp += float(D[i, j])
    return (n * (n - 1) // 2) / (tmp * n)


def far_seam(n, seed, d):
    """matrix(n, seed) with seam n - 1 at distance d from every other seam."""
    D = matrix(n, seed)
    D[n - 1, :] = D[:, n - 1] = d
    D[n - 1, n - 1] = 0.0
    return D


def zero_draw_matrix():
    return far_seam(64, 64, 1000.0)


def unreachable(n, kind):
    """`inf` where a 3-D search failed: one pair, or every pair of the last seam."""
    D = matrix(n, n)
    if kind == "pair":
        D[2, 9] = D[9, 2] = np.inf
    else:
        D[n - 1, :] = D[:, n - 1] = np.inf
        D[n - 1, n - 1] = 0.0
    return D


def subnormal_matrix(n=20):
    """Seam n - 1 so far away that its information tau0 * heuristic^6 is exactly one subnormal ulp, while pair (0, 1) at
    1e290 makes tau0 ~ 1e-290 and keeps every other tour length finite (one such pair in a tour does not matter: a tour that
    uses it only loses to the others).  When seam n - 1 is the last one left, the sum is that one ulp and u * sum rounds to 0
    for every u <= 1/2."""
    base = matrix(n, 5)
    base[0, 1] = base[1, 0] = 1e290

    def info(d):
        D = base.copy()
        D[n - 1, :] = D[:, n - 1] = d
        D[n - 1, n - 1] = 0.0
        return D, tau0(D) * pow6(1 / (d + 1e-8))

    lo, hi = 1.0, 1e12                     # info(lo) is normal, info(hi) is 0: bisect on the log scale
    for _ in range(200):
        mid = float(np.sqrt(lo * hi))
        D, v = info(mid)
        if v == ULP0:
            return D
        lo, hi = (mid, hi) if v > ULP0 else (lo, mid)
    raise AssertionError("no distance gives one subnormal ulp")


def lattice(nx, ny, step=0.1):
    """Seams on a grid, distances as searchBestPathOfPoints writes them ("%.3f"): many tours of equal length."""
    P = np.array([(i * step, j * step, 0.0) for i in range(nx) for j in range(ny)])
    D = np.sqrt(((P[:, None] - P[None]) ** 2).sum(-1))
    return np.array([[float("%.3f" % v) for v in row] for row in D])


def duplicates(n, seed):
    """Every seam twice, at distance 0."""
    P = np.random.default_rng(seed).random((n // 2, 3))
    P = np.concatenate([P, P])
    D = np.sqrt(((P[:, None] - P[None]) ** 2).sum(-1))
    return np.array([[float("%.6f" % v) for v in row] for row in D])


def ant_tours(oracle, D, seed, colony, iteration, ph):
    """One iteration's construction (ACS_GTSP.hpp:103-159) from the pheromone matrix `ph`, in plain Python floats: every
    ant's tour and L."""
    n = len(D)
    Dl, ph = D.tolist(), ph.tolist()
    info = [[ph[i][j] * pow6(1 / (Dl[i][j] + 1e-8)) for j in range(n)] for i in range(n)]
    tours, Ls = [], []
    for k in range(n):
        free = [c != k for c in range(n)]
        r, left, tour = k, n - 1, []
        for step in range(n):
            nxt = k
            if left:
                row = info[r]
                s = 0.0
                for c in range(n):
                    if free[c]:
                        s += row[c]
                rnd = rand31(oracle, seed, iteration, k, step, colony) / 2147483647.0 * s
                p = 0.0
                for c in range(n):
                    if free[c]:
                        p += row[c]
                        if p >= rnd:
                            nxt = c
                            break
            if free[nxt]:
                free[nxt] = False
                left -= 1
            tour.append((r, nxt))
            r = nxt
        L = 0.0
        for a, b in tour[:-1]:
            L += Dl[a][b]
        tours.append(tour)
        Ls.append(L)
    return tours, Ls


def is_tour(tour, n):
    return len(tour) == n and sorted(int(r) for r, _ in tour) == list(range(n)) and all(tour[i][1] == tour[(i + 1) % n][0] for i in range(n))


def assert_colony(g, b, T):
    tour, L = T.best()
    gt, gL = g.best(b)
    assert np.array_equal(gt, tour), b
    assert bits(gL) == bits(L), (b, gL, L)
    assert np.array_equal(bits(g.pheromone(b)), bits(T.pheromone())), b


def oracle_run(oracle, D, seed, first, batch, iters, cnt=None):
    Ts = []
    for b in range(batch):
        T = oracle.Gtsp(D, seed=seed, colony_id=first + b, cnt=cnt)
        assert T.iterate(iters) == iters
        Ts.append(T)
    return Ts


def check_batch(oracle, D, seed, batch, iters, first=0):
    """computeBatch against the oracle; returns the oracle colonies."""
    import welding_robot_b200 as wr
    n = len(D)
    g = wr.ACS_GTSP(seed=seed)
    g.dis, g.city_num, g.cnt = D, n, n * (n - 1) // 2
    g.computeBatch(batch, iters, colony_first=first)
    Ts = oracle_run(oracle, D, seed, first, batch, iters)
    for b, T in enumerate(Ts):
        assert bits(g.tau0()) == bits(T.tau0())
        assert_colony(g, b, T)
    return Ts


def solve_handle(D, seed, batch, first=0):
    import welding_robot_b200 as wr
    n = len(D)
    g = wr.ACS_GTSP(seed=seed)
    g.dis, g.city_num, g.cnt = D, n, n * (n - 1) // 2
    g._create(batch, first)
    return g


def check_solve(g, cols, cap):
    ran, hist, bc = g.solve(cap)
    for b, col in enumerate(cols):
        r, h = col.solve(cap if cap > 0 else g.city_num ** 2)   # cap 0: MAX_itera = N^2 (ACS_GTSP.hpp:257)
        assert ran[b] == r, (b, ran[b], r)
        assert np.array_equal(bits(hist[b, :r]), bits(h)), b
        assert_colony(g, b, col.T)
    return ran


def check_solve_fresh(oracle, D, seed, batch, cap):
    g = solve_handle(D, seed, batch)
    return check_solve(g, [Colony(oracle, D, seed, b) for b in range(batch)], cap)


# ---- zero draw ---------------------------------------------------------------------------------------------------------

def test_zero_draw_constant(oracle):
    """The Philox draw the zero-draw cases rely on really is rand() == 0 (runs without a GPU)."""
    assert rand31(oracle, ZERO_SEED, 0, ZERO_ANT, ZERO_STEP, 0) == 0
    assert rand31(oracle, ZERO_SEED, 0, ZERO_ANT, ZERO_STEP - 1, 0) != 0


def test_degenerate_inputs_on_the_host():
    """The inputs below really are degenerate (runs without a GPU): the heuristic of 1e60 underflows to 0 while tau0 stays
    positive, and the subnormal case's information is one subnormal ulp."""
    D = far_seam(20, 20, 1e60)
    assert pow6(1 / (1e60 + 1e-8)) == 0.0 and tau0(D) > 0
    D = subnormal_matrix()
    v = tau0(D) * pow6(1 / (D[19, 0] + 1e-8))
    assert 0 < v < TINY and v == ULP0
    assert 0.5 * v == 0.0                 # u * sum rounds to 0 for u <= 1/2


@gpu
def test_zero_draw_batch(oracle):
    """n = 64 with seam 63 at distance 1000: every ant visits it last, so ant 14's zero draw at step 62 finds cities 0..15
    visited and must still take seam 63."""
    D = zero_draw_matrix()
    Ts = check_batch(oracle, D, ZERO_SEED, 2, 3)
    tour, L = Ts[0].best()
    assert is_tour(tour.tolist(), 64) and L > 1000


@gpu
def test_zero_draw_solve(oracle):
    check_solve_fresh(oracle, zero_draw_matrix(), ZERO_SEED, 2, 4096)


# ---- zero information: unreachable seams, heuristic underflow, subnormal sum ---------------------------------------

@gpu
@pytest.mark.parametrize("kind", ["pair", "seam"])
@pytest.mark.parametrize("n", [17, 20, 40, 64])
def test_unreachable_matrix(oracle, n, kind):
    """setDistanceMatrix with `inf` distances: tau0 = 0, so every ant of iteration 0 walks the lowest unvisited city."""
    import welding_robot_b200 as wr
    D = unreachable(n, kind)
    g = wr.ACS_GTSP(seed=3, colonies=2)
    assert g.setDistanceMatrix(D)
    g.iterate(4)
    Ts = oracle_run(oracle, D, 3, 0, 2, 4)
    for b, T in enumerate(Ts):
        assert bits(g.tau0()) == bits(T.tau0()) and T.tau0() == 0.0
        assert_colony(g, b, T)
        tour, L = T.best()
        if kind == "pair":
            assert is_tour(tour.tolist(), n) and L < NO_TOUR_L
        else:
            assert len(tour) == 0 and L == NO_TOUR_L   # every tour has an infinite edge: no best tour, no deposit


@gpu
@pytest.mark.parametrize("kind", ["pair", "seam"])
@pytest.mark.parametrize("n", [17, 20, 40, 64])
def test_unreachable_graph_file(oracle, tmp_path, n, kind):
    """readFromGraphFile + computeSolution on a graph file as searchBestPathOfPoints writes it ("%.3f", `inf` for a pair
    whose 3-D search failed)."""
    import welding_robot_b200 as wr
    D = np.array([[float("%.3f" % v) for v in row] for row in unreachable(n, kind)])
    f = tmp_path / "graph.in"
    with open(f, "w") as fp:
        fp.write("%d %d\n" % (n, n * (n - 1) // 2))
        for i in range(n):
            for j in range(i + 1, n):
                fp.write("%.3f\n" % D[i, j])
    assert "inf\n" in f.read_text()
    g = wr.ACS_GTSP(seed=8)
    assert g.readFromGraphFile(str(f)) and g.computeSolution()
    T = oracle.Gtsp(D, seed=8, colony_id=0)
    T.iterate(n * n, early_stop=True)
    tour, L = T.best()
    assert bits(g.tau0()) == bits(T.tau0())
    assert np.array_equal(g.best_path, tour) and bits(g.best_L) == bits(L)
    assert np.array_equal(bits(g.pheromone(0)), bits(T.pheromone()))


@gpu
@pytest.mark.parametrize("n", [17, 20, 40])
def test_heuristic_underflow(oracle, n):
    """Seam n - 1 at 1e60: its information is exactly 0 while tau0 > 0; when it is the last seam left the sum is 0.
    Every tour has an edge of 1e60 > the no-tour length, so the oracle never records a tour."""
    D = far_seam(n, n, 1e60)
    Ts = check_batch(oracle, D, 6, 2, 3)
    assert Ts[0].tau0() > 0 and len(Ts[0].best()[0]) == 0
    check_solve_fresh(oracle, D, 6, 2, 0)


@gpu
def test_subnormal_sum(oracle):
    D = subnormal_matrix()
    Ts = check_batch(oracle, D, 12, 3, 6)
    tour, L = Ts[0].best()
    assert is_tour(tour.tolist(), 20) and L < NO_TOUR_L
    check_solve_fresh(oracle, D, 12, 3, 0)


# ---- long runs: subnormal and zero pheromone -------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("n", [20, 40])
def test_long_run_subnormal_pheromone(oracle, n):
    """8000 iterations (0.9^8000 ~ 1e-366) on seams in a 2 x 2 x 2 box, then a solve with a large cap from there.  Off-tour
    pheromone sinks into the subnormals but never reaches 0: 0.9 rounds up in binary, so 5 ulps * 0.9 rounds back to 5 ulps.
    Its information, 5 ulps * heuristic^6, is subnormal, or exactly 0 for pairs farther apart than ~1.47."""
    D = matrix(n, n) * 2
    g = solve_handle(D, 21, 2)
    g.iterate(8000)
    cols = [Colony(oracle, D, 21, b) for b in range(2)]
    off = ~np.eye(n, dtype=bool)
    h = 1 / (D + 1e-8)
    h6 = (h * h) * ((h * h) * (h * h))
    for b, col in enumerate(cols):
        col.iterate(8000)
        ph = col.T.pheromone()
        info = ph * h6
        assert ((ph < TINY) & off).any() and (ph > 0).all(), b
        assert ((info != 0) & (info < TINY) & off).any() and ((info == 0) & off).any(), b
        assert_colony(g, b, col.T)
    check_solve(g, cols, 1 << 17)


# ---- NaN distance ----------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("n", [20, 40])
def test_nan_distance(oracle, n):
    """tau0 = NaN: every roulette falls through to the ant's home city (:143), every L is 0, the deposit is 1/0."""
    D = matrix(n, n)
    D[2, 9] = D[9, 2] = np.nan
    Ts = check_batch(oracle, D, 4, 2, 3)
    tour, L = Ts[0].best()
    assert np.isnan(Ts[0].tau0()) and L == 0.0 and (tour == 0).all()
    check_solve_fresh(oracle, D, 4, 2, 0)


# ---- ties --------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("nx,ny,seed,it", [(4, 5, 22, 0), (6, 6, 0, 9), (6, 8, 1, 8)])
def test_ties_take_the_lowest_ant(oracle, nx, ny, seed, it):
    """Seams on a lattice: in iteration `it` of colony 0 several ants share the shortest L with different tours (in the
    last two cases ants of different warps), and the deposit goes along the lowest such ant's tour (:165-170).  At
    (4, 5, 22, 0) that tour is also the new best."""
    D = lattice(nx, ny)
    n = len(D)
    T = oracle.Gtsp(D, seed=seed, colony_id=0)
    T.iterate(it)
    ph = T.pheromone()
    tours, Ls = ant_tours(oracle, D, seed, 0, it, ph)
    ties = [k for k in range(n) if Ls[k] == min(Ls)]
    assert len(ties) > 1 and len({tuple(tours[k]) for k in ties}) > 1
    T.iterate(1)
    ph *= 0.9
    for r, s in tours[ties[0]]:
        ph[r, s] += 1.0 / Ls[ties[0]]
        ph[s, r] = ph[r, s]
    assert np.array_equal(bits(ph), bits(T.pheromone()))
    check_batch(oracle, D, seed, 2, it + 1)
    check_solve_fresh(oracle, D, seed, 2, 0)


@gpu
def test_duplicate_seams(oracle):
    """Every seam twice: distance 0, heuristic (1 / 1e-8)^6 ~ 1e48 next to information of order 1."""
    D = duplicates(40, 2)
    check_batch(oracle, D, 9, 3, 8)
    check_solve_fresh(oracle, D, 9, 3, 0)


# ---- city counts at the kernel's boundaries ---------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("n", [16, 17, 31, 32, 47, 48, 63, 65, 127, 128, 129, 463])
def test_city_counts(oracle, n):
    """Check-point interval 16, visited word 32, row chunk 8 and thread warps, each side of the boundary."""
    check_batch(oracle, matrix(n, n + 1000), 13, 2, 3 if n < 400 else 2)


# ---- colony ids at the top of the Philox stream tag ------------------------------------------------------------------

@gpu
def test_top_colony_ids(oracle):
    import welding_robot_b200 as wr
    D = matrix(20, 20)
    check_batch(oracle, D, 14, 3, 4, first=65533)
    g = wr.ACS_GTSP(seed=14)
    g.dis, g.city_num, g.cnt = D, 20, 190
    with pytest.raises(wr.WrError, match="65536"):
        g.computeBatch(3, 1, colony_first=65534)
