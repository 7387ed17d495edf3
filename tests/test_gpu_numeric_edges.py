"""GPU: the step kernels where their exactness arguments (DESIGN.md section 4) live -- time_to_collision's early
exits and the division-free probe, the radius threshold T(R), div_floor's 8-ulp fallback, the weight-0 proof, the
reference's width-stride aliasing and degenerate eyesights.  Isolated pairs and small clusters of many edge classes
share one handle; every step is checked against the oracle at the bar of tests/parity.py (neighbour lists and t_i
bit-exact, forces and velocities within 1e-9 with identical NaN / inf patterns), and the three forms of the step kernel
against each other bit for bit."""
import math

import numpy as np
import pytest

import oracle_ffi as O
import parity as P
import rmf_crowdsim_b200 as R
from rmf_crowdsim_b200 import _native as N
from rmf_crowdsim_b200 import scenes as SC
from rmf_crowdsim_b200.strips import LocalStripGroup
from parity import _nx, _same, threshold_points

pytestmark = pytest.mark.gpu

INF, NAN = float("inf"), float("nan")
ZA = (0.05, 1.0, 0.0, 0.5, 1.0, 0.2)
HEAVY = (0.05, 1.0, 0.0, 0.5, 50.0, 0.05)  # heavy, small agents: a crowd that stays sane for a few steps
DT = (0, 16_666_667)


class Layout:
    """Planner groups of one handle (ids sequential in group order), built identically in the oracle and on the GPU;
    velocities are injected with set_state on both."""

    def __init__(self, w, h, cell, off=(0.0, 0.0)):
        self.grid = (float(w), float(h), float(cell), (float(off[0]), float(off[1])))
        self.groups = []

    def add(self, xy, vxy, eyesight, lp=ZA, pref=(1.3, 0.0)):
        xy = np.asarray(xy, dtype=np.float64).reshape(-1, 2)
        vxy = np.asarray(vxy, dtype=np.float64).reshape(-1, 2)
        assert xy.shape == vxy.shape
        first = self.n
        self.groups.append((xy, vxy, float(eyesight), tuple(float(v) for v in lp), pref))
        return np.arange(first, first + len(xy))

    @property
    def n(self):
        return sum(len(g[0]) for g in self.groups)

    def state(self):
        return np.concatenate([g[0] for g in self.groups]), np.concatenate([g[1] for g in self.groups])

    def oracle(self, index_mode=O.DEFERRED):
        w, h, cell, off = self.grid
        o = O.OracleSim(w, h, cell, off, index_mode=index_mode)
        for xy, _, eye, lp, pref in self.groups:
            o.add_agents(xy, o.hl_parity(pref), o.lp_zanlungo(*lp), eye)
        xy, v = self.state()
        o.set_state(np.arange(self.n, dtype=np.uint64), xy[:, 0], xy[:, 1], v[:, 0], v[:, 1])
        o.enable_trace(True)
        return o

    def sim(self, kernel=0):
        w, h, cell, off = self.grid
        g = R.Simulation(R.LocationHash2D(w, h, cell, off, capacity=max(self.n, 64)))
        g._keep = []
        for xy, _, eye, lp, pref in self.groups:
            planners = (R.ParityVelocityPlan(pref), R.Zanlungo(*lp))
            g._keep.append(planners)
            g.add_agents(xy, *planners, eye)
        xy, v = self.state()
        g.set_state(None, xy[:, 0], xy[:, 1], v[:, 0], v[:, 1])
        g.set_option(N.RCS_OPT_STEP_KERNEL, kernel)
        g.set_trace(True)
        return g


def _check_forms(lay, steps=1, in_loop=False):
    """Steps the layout on the three forms of the step kernel (thread per agent, warp-cooperative, staged tile) and,
    with in_loop, through step_in_loop, each step from the oracle's state.  Returns the oracle's traces."""
    o = lay.oracle()
    sims = [lay.sim(k) for k in (1, 2, 3)]
    lo = lay.oracle(O.IN_LOOP) if in_loop else None
    gl = lay.sim() if in_loop else None
    traces = []
    for _ in range(steps):
        for g in sims:
            P.resync(g, o)
        o.step(*DT)
        for g in sims:
            g.step(R.Duration(*DT))
        to, so = o.read_trace(), o.read_state()
        for g in sims:
            r = P.compare_traces(g.read_trace(), to)
            assert r["force_rel_err"] <= P.REL_TOL, r
            s = P.compare_states(g.read_state(), so)
            assert s["vel_rel_err"] <= P.REL_TOL and s["pos_rel_err"] <= P.REL_TOL, s
        t1, s1 = sims[0].read_trace(), sims[0].read_state()
        for g in sims[1:]:
            _same(t1, g.read_trace(), ("id", "nb_offsets", "nb_ids", "t_i", "fx", "fy"))
            _same(s1, g.read_state(), ("id", "x", "y", "vx", "vy"))
        if in_loop:
            P.resync(gl, lo)
            lo.step(*DT)
            gl.step_in_loop(R.Duration(*DT))
            r = P.compare_traces(gl.read_trace(), lo.read_trace())
            assert r["force_rel_err"] <= P.REL_TOL, r
            s = P.compare_states(gl.read_state(), lo.read_state())
            assert s["vel_rel_err"] <= P.REL_TOL and s["pos_rel_err"] <= P.REL_TOL, s
        traces.append(to)
    st = [g.stats() for g in sims]
    assert len({(s.candidate_total, s.neighbour_total, s.finite_tti_count) for s in st}) == 1
    return traces


def _sites(n, spacing, origin=(0.0, 0.0), per_row=None):
    """n lattice sites `spacing` apart, row by row."""
    per_row = per_row or int(math.ceil(math.sqrt(n)))
    k = np.arange(n)
    return np.stack([origin[0] + (k % per_row) * spacing, origin[1] + (k // per_row) * spacing], axis=1)


def _ordinary_pairs(sites, rng):
    """Two agents 0.6-1.2 m apart per site on roughly converging courses: finite t_i, ordinary forces."""
    xy, v = [], []
    for s in sites:
        ang = rng.uniform(0, 2 * math.pi)
        d = rng.uniform(0.6, 1.2)
        e = np.array([math.cos(ang), math.sin(ang)])
        xy += [s, s + d * e]
        v += [0.8 * e + rng.uniform(-0.2, 0.2, 2), -0.8 * e + rng.uniform(-0.2, 0.2, 2)]
    return np.array(xy), np.array(v)


# ---- 1. time_to_collision edges as agent states --------------------------------------------------------------------
# (agent_radius, rel_vel, rel_pos): the neighbour sits at base + rel_pos with velocity v + rel_vel.  Positions cannot
# be non-finite (the index rejects them), velocities can.
TTC_PAIRS = [
    (0.2, (1.4e-162, 0.0), (1.0, 0.0)),       # a underflows to 0, b*b subnormal, b > 0: t_i = 0, force NaN
    (0.2, (-1.4e-162, 0.0), (1.0, 0.0)),      # the same with b < 0
    (0.2, (0.0, 1.4e-162), (0.0, 1.0)),       # along y
    (0.2, (7e-163, 7e-163), (0.75, 0.875)),   # a == 0, sqrt(fl(b*b)) < b
    (0.2, (-7e-163, -7e-163), (0.75, 0.875)),
    (0.2, (1e-163, 0.0), (-1.0, 0.0)),        # a == 0, b*b == 0
    (0.2, (0.0, 0.0), (1.0, 0.0)),            # a == 0, b == 0
    (0.2, (1e-160, 0.0), (-1.0, 0.0)),        # a subnormal > 0: t ~ 1e160
    (0.2, (1e-160, 0.0), (1.0, 0.0)),
    (0.5, (-1.0, 0.0), (1.5, 0.5)),           # grazing: disc == 0, t = 1.5
    (0.5, (-1.0, 0.0), (1.5, 0.5 - 2.0 ** -40)),  # disc just above 0
    (0.5, (-1.0, 0.0), (1.5, 0.5 + 2.0 ** -40)),  # disc just below 0
    (0.5, (-1.0, 0.0), (0.5, 0.0)),           # touching: c == 0
    (0.5, (1.0, 0.0), (0.5, 0.0)),            # touching, receding
    (0.5, (-1.0, 0.0), (0.375, 0.0)),         # overlap: t_i = 0
    (0.2, (1e200, 0.0), (-1.0, 0.0)),         # a overflows
    (0.2, (INF, 0.0), (-1.0, 0.0)),           # non-finite neighbour velocity: literal magnitude branch
    (0.2, (NAN, 0.0), (-1.0, 0.0)),
    (0.2, (0.0, -INF), (0.0, 1.0)),
]


def ttc_layout(seed=0):
    """Every TTC_PAIRS class twice (both id orders of the pair) on a 12 m lattice, ordinary pairs on the sites between
    them (tile path), a second copy of the near-grazing classes with eyesight 4 (wider than the 2 m cells: the aside
    lists) and a crowded cell whose agents move at +-7e-163 m/s (the sequential routine)."""
    rng = np.random.default_rng(seed)
    lay = Layout(192.0, 192.0, 2.0)
    sites = _sites(4 * len(TTC_PAIRS) + 16, 12.0, origin=(8.0, 8.0), per_row=14)
    k = 0
    by_radius = {}
    for rep in range(2):
        for r, rv, rp in TTC_PAIRS:
            b = sites[k] + 0.0
            k += 1
            tiny = all(abs(c) < 1e-100 for c in rv)  # v0 + rv must keep the tiny relative speed exactly
            v0 = np.zeros(2) if tiny else np.array([0.3, -0.2])
            a, o = (b, b + rp), (v0, v0 + np.array(rv))
            if rep == 1:  # the other agent gets the lower id
                a, o = a[::-1], o[::-1]
            xy, v = by_radius.setdefault(r, ([], []))
            xy += list(a)
            v += list(o)
            k += 1  # an ordinary pair in between
    for r, (xy, v) in by_radius.items():
        lay.add(xy, v, 2.0, lp=ZA[:5] + (r,))
    oxy, ov = _ordinary_pairs(sites[1:2 * len(TTC_PAIRS) * 2:2], rng)
    lay.add(oxy, ov, 2.0)
    wide = [p for p in TTC_PAIRS if p[0] == 0.5]
    xy, v = [], []
    for j, (r, rv, rp) in enumerate(wide):
        b = sites[k + j]
        xy += [b, b + rp]
        v += [np.zeros(2), np.array(rv)]
    lay.add(xy, v, 4.0, lp=ZA[:5] + (0.5,))
    crowd = sites[k + len(wide) + 1] + _sites(36, 0.3)
    lay.add(crowd, [(7e-163 * (-1) ** i, 0.0) for i in range(len(crowd))], 2.0, lp=ZA[:5] + (0.1,),
            pref=(7e-163, 0.0))
    return lay


def test_ttc_edge_classes_match_the_oracle_on_every_kernel_form():
    lay = ttc_layout()
    (t,) = _check_forms(lay)
    # the classes are really hit: t_i = 0 from an underflowing relative speed (with its NaN force), finite t_i, inf
    assert (t["t_i"] == 0.0).sum() >= 8 and np.isnan(t["fx"]).sum() >= 8
    assert np.isfinite(t["t_i"]).sum() > 40 and np.isinf(t["t_i"]).sum() > 20


# ---- 2. radius threshold -------------------------------------------------------------------------------------------
EYESIGHTS = [1.1, 0.3, 1.7, 2.7, 4.1, 0.5, 2.0]  # R*R inexact, then exact


def threshold_layout(rng):
    """Per eyesight: probe agents with a neighbour at T-1ulp (a neighbour), T and T+1ulp (not), along an axis and a
    diagonal, each pair isolated, in one row along y = 0; plus ordinary pairs.  Returns the layout and
    (probe position, radius, id)."""
    lay = Layout(704.0, 704.0, 2.0, (0.0, -352.0))
    xs = iter(5.0 + 11.0 * np.arange(64))
    probes = []
    for r in EYESIGHTS:
        xy, v = [], []
        for diagonal in (False, True):
            for which in range(3):
                p, qs = threshold_points(r, next(xs), diagonal)
                xy += [p, qs[which]]
                v += [rng.uniform(-0.3, 0.3, 2), rng.uniform(-0.3, 0.3, 2)]
        first = lay.n
        lay.add(xy, v, r)
        probes += [(np.array(xy[i]), r, first + i) for i in range(0, len(xy), 2)]
    oxy, ov = _ordinary_pairs([(next(xs), 8.0) for _ in range(20)], rng)
    lay.add(oxy, ov, 2.0)
    return lay, probes


def test_radius_threshold_neighbours_match_the_oracle():
    lay, probes = threshold_layout(np.random.default_rng(5))
    (t,) = _check_forms(lay)
    off = t["nb_offsets"].astype(np.int64)
    got = [list(t["nb_ids"][off[i]:off[i + 1]]) for _, _, i in probes]
    # the classification is the one the threshold argument claims: only T - 1 ulp is inside
    assert got == [[i + 1] if k % 3 == 0 else [] for k, (_, _, i) in enumerate(probes)]


def test_radius_threshold_through_query_radius():
    lay, probes = threshold_layout(np.random.default_rng(6))
    w, h, cell, off = lay.grid
    xy, _ = lay.state()
    ids = np.arange(len(xy), dtype=np.uint64)
    o = O.OracleSim(w, h, cell, off)
    for i, p in zip(ids, xy):
        o.index_add_or_update(int(i), p)
    g = R.LocationHash2D(w, h, cell, off, capacity=len(xy))
    g.add_or_update_many(ids, xy)
    q = np.array([p for p, _, _ in probes])
    radius = np.array([r for _, r, _ in probes])
    offs, got = g.query_radius(q, radius)
    for k, (p, r, i) in enumerate(probes):
        want = list(o.query_radius(r, p))
        assert list(got[int(offs[k]):int(offs[k + 1])]) == want, k
        assert want == ([i, i + 1] if k % 3 == 0 else [i])


# ---- 3. cell edges with non-power-of-two cells ----------------------------------------------------------------------
ULPS = [0, 1, -1, 2, -2, 4, -4, 7, -7, 8, -8, 9, -9, 12, -12, 16, -16]
CELLS = [(0.3, (0.0, 0.0)), (0.7, (-7.7, 13.1)), (1.1, (0.0, 0.0)), (2.6, (-7.7, 13.1))]


def edge_scene(cell, off, rng, ncol=48):
    """Agents at k*cell + off and 1-16 ulp either side of it in x and in y, with eyesight == cell so that p +- eyesight
    also lands next to an edge (stencils of 2, 3 or 4 columns), each with a partner 0.4-0.9 cells away."""
    xy, v = [], []
    edges = [(3 * a + 2, 3 * b + 2) for a in range(ncol // 3 - 1) for b in range(ncol // 3 - 1)]
    rng.shuffle(edges)
    for n, (kx, ky) in enumerate(edges[:120]):
        ex, ey = kx * cell + off[0], ky * cell + off[1]
        ux, uy = ULPS[n % len(ULPS)], ULPS[(n // len(ULPS) + n) % len(ULPS)]
        p = np.array([_nx(ex, ux), _nx(ey, uy)])
        ang = rng.uniform(0, 2 * math.pi)
        xy += [p, p + rng.uniform(0.4, 0.9) * cell * np.array([math.cos(ang), math.sin(ang)])]
        v += [rng.uniform(-0.5, 0.5, 2) * cell, rng.uniform(-0.5, 0.5, 2) * cell]
    lp = ("zanlungo",) + HEAVY[:5] + (0.05 * cell,)
    return SC.Scene(name="edges", width=ncol * cell, height=ncol * cell, cell=cell, offset=off, xy=np.array(xy),
                    vxy=np.array(v), eyesight=cell, lp=lp)


def _layout_of(scene):
    lay = Layout(scene.width, scene.height, scene.cell, scene.offset)
    lay.add(scene.xy, scene.vxy, scene.eyesight, lp=scene.lp[1:], pref=scene.hl[1])
    return lay


@pytest.mark.parametrize("cell,off", CELLS)
def test_cell_edges_match_the_oracle_and_commit_to_the_right_cells(cell, off):
    scene = edge_scene(cell, off, np.random.default_rng(int(cell * 10)))
    lay = _layout_of(scene)
    _check_forms(lay, steps=2)
    g = lay.sim(3)
    idx = g.spatial_index
    o = lay.oracle()
    xy0 = scene.xy
    assert np.array_equal(idx.cell_of(xy0), o.cell_of(xy0))
    g.step(R.Duration(*DT))
    g.step(R.Duration(0, 0))  # sorts by the committed positions and leaves them where they are
    st = g.read_state(order=N.RCS_ORDER_STORAGE)
    pts = np.stack([st["x"], st["y"]], axis=1)
    cells = idx.cell_of(pts)
    assert np.array_equal(cells, o.cell_of(pts)) and (cells >= 0).all()
    key = cells.astype(np.uint64) * np.uint64(1 << 32) + st["id"]
    assert np.all(key[1:] > key[:-1])  # storage order: (committed cell, ascending id)


# ---- strips: families 2 and 3 against one handle -------------------------------------------------------------------
def _strip_vs_single(scene, world, boundaries, steps=3):
    single = SC.build_simulation(scene)
    grp = LocalStripGroup(scene, world, boundaries=boundaries, halo_capacity=4096)
    single.set_trace(True)
    grp.set_trace(True)
    for _ in range(steps):
        single.step(R.Duration(*DT))
        grp.step(R.Duration(*DT))
        _same(single.read_trace(), grp.read_trace(), ("id", "nb_offsets", "nb_ids", "t_i", "fx", "fy"))
        _same(single.read_state(), grp.read_state(), ("id", "x", "y", "vx", "vy", "next_waypoint"))
    assert sum(grp.agent_counts()) == scene.n


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("cell,off", CELLS[1:3])
def test_cell_edges_on_strips_match_one_handle(world, cell, off):
    scene = edge_scene(cell, off, np.random.default_rng(int(cell * 10) + world))
    # boundaries at columns that hold edge agents (column 3a + 2)
    ncol = int(scene.width / scene.cell)  # (width / resolution) as usize: 47 for 48 * 0.7 / 0.7
    bounds = [0, 17, 32, ncol] if world == 3 else [0, 23, ncol]
    _strip_vs_single(scene, world, bounds)


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("r", [1.1, 2.7])
def test_radius_threshold_on_strips_match_one_handle(world, r):
    rng = np.random.default_rng(world)
    xy, v = [], []
    for n in range(8):
        p, qs = threshold_points(r, 4.25 + 9.0 * n, diagonal=n % 2 == 1)
        xy += [p, qs[n % 3]]
        v += [rng.uniform(-0.3, 0.3, 2), rng.uniform(-0.3, 0.3, 2)]
    oxy, ov = _ordinary_pairs(_sites(24, 9.0, origin=(4.25, 6.0), per_row=8), rng)
    xy, v = np.concatenate([np.array(xy), oxy]), np.concatenate([np.array(v), ov])
    # pairs straddle the boundaries: probes sit at x = 4.25 + 9 k (columns 2, 6, 11, 15, ...), their partners r to the
    # right, in columns 7 and 16
    scene = SC.Scene(name="thr", width=80.0, height=80.0, cell=2.0, offset=(0.0, -40.0), xy=xy, vxy=v,
                     eyesight=r, lp=("zanlungo",) + ZA)
    bounds = [0, 7, 16, 40] if world == 3 else [0, 16, 40]
    _strip_vs_single(scene, world, bounds)


# ---- 4. non-square grids through the step ---------------------------------------------------------------------------
@pytest.mark.parametrize("w,h,eyesight", [(24.0, 8.0, 1.5), (8.0, 24.0, 4.5)])
def test_non_square_grids_through_the_step(w, h, eyesight):
    """n_x > n_y: agents above the rectangle are accepted into the gap cells of the width stride.  n_y > n_x: rows
    alias into the next column, and with a stencil of 10 rows (eyesight 4.5 cells, 8 rows per column) two stencil
    columns reach the same cells, so the
    reference lists a neighbour twice.  Three kernel forms and step_in_loop against the oracle."""
    rng = np.random.default_rng(int(w))
    o = O.OracleSim(w, h, 1.0, (0.0, 0.0))
    pts = rng.uniform([0.0, 0.0], [max(w, h)] * 2, size=(4000, 2))
    inside = o.cell_of(pts) >= 0
    for d in ((0.05, 0.05), (-0.05, 0.05), (0.05, -0.05), (-0.05, -0.05)):  # and stays so for a couple of steps
        inside &= o.cell_of(pts + d) >= 0
    pts = pts[inside]
    keep = [pts[0]]
    for p in pts[1:]:  # no two agents closer than 0.5 m
        if len(keep) < 120 and min(np.hypot(*(p - q)) for q in keep) > 0.5:
            keep.append(p)
    xy = np.array(keep)
    lay = Layout(w, h, 1.0)
    lay.add(xy, rng.uniform(-0.4, 0.4, size=xy.shape), eyesight, lp=HEAVY[:5] + (0.1,))
    if w > h:
        assert (xy[:, 1] > h).sum() > 10  # above the rectangle, inside the grid's index range
    traces = _check_forms(lay, steps=2, in_loop=True)
    t = traces[0]
    off = t["nb_offsets"].astype(np.int64)
    dup = sum(len(set(t["nb_ids"][off[i]:off[i + 1]])) < off[i + 1] - off[i] for i in range(len(off) - 1))
    assert w > h or dup > 0


# ---- 5. planners outside the weight-0 proof ------------------------------------------------------------------------
def planner_layout(rng):
    """Groups with w0_fast = 0 (two_r / force_distance at 700 -+ a few ulp, force_distance 0 and negative,
    agent_scale inf and NaN, agent_radius 0) next to proof-eligible groups; clusters of three with converging,
    overlapping and non-finite (inf, NaN, 1e200) neighbour velocities."""
    r = 0.35
    params = [
        ZA,
        HEAVY,
        (0.05, 1.0, 0.0, 2 * r / _nx(700.0, -2), 1.0, r),  # two_r / force_distance just below 700: proof-eligible
        (0.05, 1.0, 0.0, 2 * r / _nx(700.0, 2), 1.0, r),   # just above 700
        (0.05, 1.0, 0.0, 2 * r / 700.0, 1.0, r),
        (0.05, 1.0, 0.0, 0.0, 1.0, 0.2),
        (0.05, 1.0, 0.0, -0.5, 1.0, 0.2),
        (INF, 1.0, 0.0, 0.5, 1.0, 0.2),
        (NAN, 1.0, 0.0, 0.5, 1.0, 0.2),
        (0.05, 1.0, 0.0, 0.5, 1.0, 0.0),
    ]
    lay = Layout(256.0, 256.0, 2.0)
    sites = iter(_sites(400, 10.0, origin=(5.0, 5.0), per_row=24))
    other_v = [(0.0, 0.0), (INF, 0.0), (NAN, 0.5), (1e200, -1e200), (-0.7, 0.1)]
    for lp in params:
        # capped forces times exp((2r - dist) / force_distance) must not throw anybody out of the grid: with an infinite
        # mass the new velocity is the preferred one (finite force) or NaN (non-finite force, the agent goes to cell 0)
        lp = lp[:4] + (INF, lp[5])
        s = 3.0 if lp[5] > 0.3 or lp[3] == 0.0 else 1.0
        xy, v = [], []
        for k in range(10):
            b = next(sites)
            gap = [0.3, 0.6, 0.9, 0.25, 0.71][k % 5]
            xy += [b, b + (s * gap, 0.0), b + (0.2 * s, 0.55 * s)]
            v += [(0.6, 0.05), other_v[k % 5], rng.uniform(-0.5, 0.5, 2)]
        lay.add(xy, v, 2.0, lp=lp)
    return lay


def test_planners_outside_the_weight_zero_proof():
    (t,) = _check_forms(planner_layout(np.random.default_rng(8)))
    assert np.isfinite(t["t_i"]).sum() > 50 and np.isnan(t["fx"]).sum() > 10


# ---- 6. degenerate eyesights ---------------------------------------------------------------------------------------
def test_degenerate_eyesights():
    """Eyesight 0, negative, NaN, 1e-300 and exactly the cell: the agents see nobody (or their cell-sized stencil) but
    are seen by their neighbours.  (An infinite eyesight would make the reference's scan loop walk ~2^64 cells.)"""
    rng = np.random.default_rng(12)
    lay = Layout(128.0, 128.0, 2.0)
    sites = iter(_sites(200, 9.0, origin=(4.5, 4.5), per_row=14))
    for eye in (0.0, -1.0, -0.0, NAN, 1e-300, 2.0, 1.0):
        xy, v = [], []
        for _ in range(6):
            b = next(sites)
            xy += [b, b + rng.uniform(-0.9, 0.9, 2)]
            v += [rng.uniform(-0.5, 0.5, 2), rng.uniform(-0.5, 0.5, 2)]
        lay.add(xy, v, eye, lp=ZA[:4] + (INF, 0.2))  # infinite mass: overlapping pairs stay in the grid
    (t,) = _check_forms(lay)
    off = t["nb_offsets"].astype(np.int64)
    assert off[60] == 0 and off[-1] > 0  # eyesight 0, -1, -0, NaN and 1e-300 see nobody
