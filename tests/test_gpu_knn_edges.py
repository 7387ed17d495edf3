"""GPU: the batched kNN query (knn_count/fill/select, rcs_query_knn) and the radius query next to it at their
exactness edges, against the oracle: exact distance ties around the query (the stable order is the visiting order),
coincident points, crowded cells past the select kernel's lane stride, non-square grids and aliased query rows, NaN
distances (the reference's sort panics: an error, and nothing written) and saturated query cells (the ring bounds
wrap).  Lists bit-exact.  Each family asserts that its edge class is hit."""
import math

import numpy as np
import pytest

import oracle_ffi as O
import parity as P
import rmf_crowdsim_b200 as R
from rmf_crowdsim_b200 import _native as N

pytestmark = pytest.mark.gpu

NAN = float("nan")
NAN_MSG = "get_nearest_neighbours: NaN distance"


def _pair(grid, pts, ids=None):
    w, h, cell, off = grid
    ids = np.arange(len(pts), dtype=np.uint64) if ids is None else np.asarray(ids, dtype=np.uint64)
    g = R.LocationHash2D(w, h, cell, off, capacity=max(len(pts) + 16, 64))
    o = O.OracleSim(w, h, cell, off)
    if len(pts):
        g.add_or_update_many(ids, pts)
    for i, p in zip(ids, pts):
        o.index_add_or_update(int(i), p)
    return g, o


def _check_knn(g, o, qs, k):
    """One batched device call against the oracle query by query; returns the oracle's lists."""
    qs = np.asarray(qs, dtype=np.float64).reshape(-1, 2)
    got, cnt = g.query_knn(qs, k)
    out = []
    for r, q in enumerate(qs):
        want = list(o.query_knn(k, q))
        assert int(cnt[r]) == len(want), (k, r, q)
        assert [int(v) for v in got[r, :len(want)]] == want, (k, r, q)
        out.append(want)
    return out


def _dist(p, q):
    return math.sqrt((p[0] - q[0]) ** 2 + (p[1] - q[1]) ** 2)


def test_knn_exact_ties_follow_the_visiting_order():
    """Agents placed symmetrically around cell-centre queries (exact distances 1, 2, sqrt 2, sqrt 8) on all four ring
    sides, at the doubled (x-s, y-s) corner and at the never-visited (x+s, y+s) corner, with ids shuffled so that id
    order and visiting order differ; plus coincident points spread over several cells."""
    rng = np.random.default_rng(7)
    grid = (20.0, 20.0, 1.0, (0.0, 0.0))
    pts = []
    for cx, cy in ((10.5, 10.5), (4.5, 15.5), (15.5, 4.5)):
        for dx, dy in ((1, 0), (-1, 0), (0, 1), (0, -1), (2, 0), (-2, 0), (0, 2), (0, -2),
                       (1, 1), (-1, -1), (1, -1), (-1, 1), (2, 2), (-2, -2), (2, -2), (-2, 2)):
            pts.append((cx + dx, cy + dy))
    for c in ((2.25, 2.75), (7.25, 3.5), (12.75, 17.25), (18.5, 18.5)):  # 5 coincident agents in each of 4 cells
        pts += [c] * 5
    pts = np.array(pts)
    ids = rng.permutation(len(pts)).astype(np.uint64)
    g, o = _pair(grid, pts, ids)
    loc = {int(i): tuple(p) for i, p in zip(ids, pts)}
    qs = [(10.5, 10.5), (4.5, 15.5), (15.5, 4.5), (2.25, 2.75), (7.25, 3.5), (12.75, 17.25), (18.5, 18.5), (9.0, 9.0)]
    ties = twice = unsorted_ties = 0
    for k in (1, 4, 5, 8, 13, 20, 64, 200):
        for q, lst in zip(qs, _check_knn(g, o, qs, k)):
            d = [_dist(loc[i], q) for i in lst]
            assert d == sorted(d)
            for a in range(len(lst) - 1):
                if d[a] == d[a + 1]:
                    ties += 1
                    unsorted_ties += lst[a] > lst[a + 1]  # equal distances NOT in id order: the visiting order rules
            twice += len(lst) - len(set(lst))
    assert ties > 100 and unsorted_ties > 10 and twice > 0


@pytest.mark.parametrize("m", [40, 1100])
def test_knn_crowded_cell_past_the_lane_stride(m):
    """One cell with m > 32 (and > 1024) candidates, some coincident, next to a few sparse agents: the select kernel
    ranks m candidates 32 lanes at a time.  k in {0, 1, 31, 32, 33, m-1, m, m+1} and k >= the live count, where the walk
    runs to the grid edge."""
    rng = np.random.default_rng(m)
    grid = (8.0, 8.0, 1.0, (0.0, 0.0))
    crowd = rng.uniform(3.0, 4.0, size=(m, 2))
    crowd[m // 2: m // 2 + 8] = crowd[:8]
    sparse = np.array([[0.5, 0.5], [7.5, 7.5], [3.5, 6.25], [1.25, 3.75]])
    pts = np.concatenate([crowd, sparse])
    ids = rng.permutation(len(pts)).astype(np.uint64)
    g, o = _pair(grid, pts, ids)
    qs = [(3.5, 3.5), (3.0, 3.0), (3.999, 3.001), (0.1, 7.9), (6.0, 2.0), (-3.0, 3.5)]
    for k in (0, 1, 31, 32, 33, m - 1, m, m + 1, len(pts), len(pts) + 50):
        res = _check_knn(g, o, qs, k)
        if k == m:
            assert len(res[0]) == m  # the crowded cell alone: ring 0 is enough


@pytest.mark.parametrize("grid", [(12.0, 5.0, 1.0, (0.0, 0.0)), (5.0, 12.0, 0.7, (-3.3, 2.1)),
                                  (30.0, 2.0, 2.0, (-10.0, -1.0))])
def test_knn_non_square_grids_and_aliased_queries(grid):
    """Non-square grids (the width cell count is the stride of both coordinates, so rows >= n_y alias into the next
    column), agents on aliased rows, and queries above the grid top, left of and below the origin and far outside."""
    w, h, cell, off = grid
    nx = int(w / cell)
    rng = np.random.default_rng(int(w * h))
    cells = rng.integers(0, nx * int(h / cell), size=120)
    pts = P._cell_centres(cells, nx, cell) + np.array(off) + rng.uniform(-0.45, 0.45, size=(120, 2)) * cell
    g, o = _pair(grid, pts)
    ys = off[1] + rng.uniform(h, h + 3 * w, size=10)
    qs = np.concatenate([
        np.stack([off[0] + rng.uniform(0, min(w, h), size=10), ys], axis=1),        # aliased rows above the top
        np.stack([off[0] - rng.uniform(0, 3 * w, size=8), off[1] + rng.uniform(0, h, size=8)], axis=1),
        np.stack([off[0] + rng.uniform(0, w, size=8), off[1] - rng.uniform(0, 3 * h, size=8)], axis=1),
        np.array([[1e6, 1e6], [-1e12, 3.0], [3.0, 1e12], [1e15, -1e15]]),
    ])
    aliased_hits = 0
    for k in (1, 5, 40, 200):
        res = _check_knn(g, o, qs, k)
        aliased_hits += sum(len(r) for r in res[:10])
    assert aliased_hits > 0


def test_knn_nan_distance_is_an_error_and_the_handle_recovers():
    """Every case of parity.NAN_KNN_CASES: where the reference's sort panics the call fails with the oracle's message;
    elsewhere the lists are the oracle's.  One bad query in a batch of good ones fails the whole call, and the next
    call on the same handle answers correctly."""
    grid = (8.0, 8.0, 1.0, (0.0, 0.0))
    errors = 0
    for agents, q, k, err in P.NAN_KNN_CASES:
        g, o = _pair(grid, np.array(agents))
        if err:
            with pytest.raises(O.OracleError, match=NAN_MSG):
                o.query_knn(k, q)
            with pytest.raises(R.CrowdsimError, match=NAN_MSG):
                g.query_knn(np.array([q]), k)
            errors += 1
        else:
            _check_knn(g, o, [q], k)
    assert errors == 6
    g, o = _pair(grid, np.array([(NAN, NAN), (0.5, 0.5), (3.5, 3.5), (6.5, 1.5)]))
    good = [(3.5, 3.6), (6.2, 1.1), (5.0, 5.0)]
    with pytest.raises(R.CrowdsimError, match=NAN_MSG):
        g.query_knn(np.array(good[:2] + [(0.2, 0.3)] + good[2:]), 1)
    # the C entry point writes neither ids nor counts when it refuses
    q = np.ascontiguousarray(good[:2] + [(0.2, 0.3)], dtype=np.float64)
    ids, cnt = np.full(6, 777, dtype=np.uint64), np.full(3, 777, dtype=np.uint64)
    rc = g._lib.rcs_query_knn(g._h, 3, q.ctypes.data_as(N.c_f64p), 2, ids.ctypes.data_as(N.c_u64p),
                              cnt.ctypes.data_as(N.c_u64p))
    assert rc == N.RCS_ERR_ARG and (ids == 777).all() and (cnt == 777).all()
    _check_knn(g, o, good, 1)


def test_knn_nan_reached_through_a_simulation_step():
    """Two agents whose relative speed squares to zero get t_i = 0 and a NaN force: after two steps both sit at NaN
    positions in cell 0 of the index the Simulation shares, and a kNN query that reaches cell 0 is the error."""
    za = (0.05, 1.0, 0.0, 0.5, 1.0, 0.2)
    o = O.OracleSim(16.0, 16.0, 2.0, (0.0, 0.0))
    o.add_agents(np.array([[5.0, 5.0], [6.0, 5.0]]), o.hl_parity((7e-163, 0.0)), o.lp_zanlungo(*za), 2.0)
    idx = R.LocationHash2D(16.0, 16.0, 2.0, (0.0, 0.0), capacity=16)
    sim = R.Simulation(idx)
    sim.add_agents([(5.0, 5.0), (6.0, 5.0)], R.ParityVelocityPlan((7e-163, 0.0)), R.Zanlungo(*za), 2.0)
    for _ in range(2):
        sim.step(R.Duration(0, 16_666_667))
        o.step(0, 16_666_667)
    assert np.isnan(sim.read_state()["x"]).all() and np.isnan(o.read_state()["x"]).all()
    for q, k in (((5.0, 5.0), 1), ((0.5, 0.5), 1), ((15.0, 1.0), 2)):
        with pytest.raises(O.OracleError, match=NAN_MSG):
            o.query_knn(k, q)
        with pytest.raises(R.CrowdsimError, match=NAN_MSG):
            idx.query_knn(np.array([q]), k)
    assert idx.query_knn(np.array([(5.0, 5.0)]), 0)[1][0] == 0


def test_knn_saturated_query_cells():
    """parity.saturated_knn_cases (their answers are pinned against the independent restatement on the CPU): +inf on an
    even- and an odd-nx grid, the last aliased row, +-inf in either coordinate, and x = (2^63 - 1024) cells on a row far
    up, whose walk runs 1025 rings.  Each case alone and all queries of a grid in one batch."""
    by_grid = {}
    found = 0
    for name, grid, pts, q, k in P.saturated_knn_cases():
        g, o = _pair(grid, pts)
        found += len(_check_knn(g, o, [q], k)[0])
        by_grid.setdefault((grid, pts.tobytes()), (grid, pts, []))[2].append((q, k))
    assert found > 50
    for grid, pts, qk in by_grid.values():
        g, o = _pair(grid, pts)
        for k in sorted({k for _, k in qk}):
            _check_knn(g, o, [q for q, _ in qk], k)


def test_query_radius_degenerate_radii():
    """get_neighbours_in_radius with radius NaN, +0, -0, negative, -inf, the smallest subnormal (only a coincident agent
    is inside) and 3x the grid width (the aliased rows list agents several times over)."""
    rng = np.random.default_rng(3)
    grid = (8.0, 6.0, 1.0, (-1.0, 0.5))
    pts = rng.uniform([-1.0, 0.5], [4.9, 6.5], size=(60, 2))  # columns 0-5: x_idx * 8 + y_idx < 48
    pts[5] = (2.25, 3.25)
    g, o = _pair(grid, pts)
    qs = np.array([(2.25, 3.25), (0.0, 1.0), (6.9, 6.4), (-5.0, 2.0), (3.0, 40.0)])
    radii = [NAN, 0.0, -0.0, -1.0, -math.inf, 5e-324, 1.5, 24.0]
    seen = {}
    for r in radii:
        off, ids = g.query_radius(qs, np.full(len(qs), r))
        for k, q in enumerate(qs):
            want = list(o.query_radius(r, q))
            assert [int(v) for v in ids[int(off[k]):int(off[k + 1])]] == want, (r, q)
            seen[(r if r == r else "nan", k)] = want
    assert seen[(5e-324, 0)] == [5]
    assert all(seen[(r, k)] == [] for r in ("nan", 0.0, -1.0, -math.inf) for k in range(len(qs)))
    multi = seen[(24.0, 0)]
    assert len(multi) > len(set(multi)) and set(multi) == set(range(60))
