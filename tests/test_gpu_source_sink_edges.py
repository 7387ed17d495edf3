"""GPU: the SourceSink stream at its exactness edges -- the spawn probe `norm(agent - source) < 0.4` against its
stencil (ss_probe_kernel, lib.rs:212-214), the chunked spawn numbering (ss_spawn_kernel), MonotonicCrowd's rounding and
degenerate parameters, the sink / waypoint test on the old position (integrate_and_store, lib.rs:305-336), the device
route follower (HL_ROUTE, rmf/mod.rs:197-215), asynchronous streams under the coarse launch bound and strips.  Every
configuration is built identically in the oracle and on the device; ids, next_waypoint, events and state are compared
bit for bit where only IEEE + - * / sqrt are involved, within 1e-9 with Zanlungo.  Each family also asserts that its
edge classes are really hit."""
import math

import numpy as np
import pytest

import oracle_ffi as O
import parity as P
import rmf_crowdsim_b200 as R
from rmf_crowdsim_b200 import _native as N
from rmf_crowdsim_b200 import scenes as SC
from rmf_crowdsim_b200.strips import LocalStripGroup, strip_columns
from parity import _same

pytestmark = pytest.mark.gpu

INF, NAN = float("inf"), float("nan")
ZA = (0.05, 1.0, 0.0, 0.5, 1.0, 0.2)
HEAVY = (0.05, 1.0, 0.0, 0.5, 50.0, 0.1)
STILL = (0.0, 0.0)
STATE = ("id", "x", "y", "vx", "vy")


class Recorder(R.EventListener):
    def __init__(self):
        self.added, self.removed = [], []

    def agent_spawned(self, position, agent):
        self.added.append((agent, position))

    def agent_destroyed(self, agent):
        self.removed.append(agent)


def _pbits(p):
    return tuple(P._bits(np.array(p, dtype=np.float64)).tolist())


class Pair:
    """One configuration in the oracle and on the device, built with the same calls.  Planners are named by kind:
    ("constant", v), ("route", points), ("zanlungo", params) or ("none",)."""

    def __init__(self, w, h, cell, off=(0.0, 0.0), capacity=4096):
        self.o = O.OracleSim(w, h, cell, off)
        self.g = R.Simulation(R.LocationHash2D(w, h, cell, off, capacity=capacity))
        self.rec = Recorder()
        self.g.add_event_listener(self.rec)
        self.keep = []
        self.spawned, self.destroyed = [], []  # the oracle's events, destroyed in canonical order per step
        self.ohl = {}

    def _planners(self, hl, lp):
        if hl[0] == "constant":
            ohl, ghl = self.o.hl_constant(hl[1]), R.ConstantVelocityPlan(hl[1])
        else:
            ohl, ghl = self.o.hl_route(hl[1]), R.RouteFollowPlan(hl[1])
        if lp[0] == "none":
            olp, glp = self.o.lp_none(), R.NoLocalPlan()
        else:
            olp, glp = self.o.lp_zanlungo(*lp[1]), R.Zanlungo(*lp[1])
        self.keep.append((ghl, glp))
        self.ohl[id(ghl)] = ohl
        return ohl, olp, ghl, glp

    def agents(self, xy, hl=("constant", STILL), lp=("none",), eyesight=1.0, vxy=None):
        ohl, olp, ghl, glp = self._planners(hl, lp)
        xy = np.asarray(xy, dtype=np.float64).reshape(-1, 2)
        ids = self.o.add_agents(xy, ohl, olp, eyesight)
        assert list(self.g.add_agents(xy, ghl, glp, eyesight)) == ids.tolist()
        s, sxy, _ = self.o.poll_events()  # add_agents reports its agents as spawned too (lib.rs:119-156)
        self.spawned += [(int(i), (float(p[0]), float(p[1]))) for i, p in zip(s, sxy)]
        if vxy is not None:
            self.set_state(ids, xy, vxy)
        return ids, ohl, ghl

    def source(self, src, wps, hl=("constant", STILL), lp=("none",), radius_sink=0.5, rate=1.0, loop=False,
               eyesight=1.0):
        ohl, olp, ghl, glp = self._planners(hl, lp)
        a = self.o.add_source_sink(src, radius_sink, rate, ohl, olp, wps, loop, eyesight)
        b = self.g.add_source_sink(R.SourceSink(tuple(src), radius_sink, R.MonotonicCrowd(rate), ghl, glp,
                                                [tuple(p) for p in wps], loop, eyesight))
        assert a == b
        return a

    def set_state(self, ids, xy, vxy):
        xy, vxy = np.asarray(xy, dtype=np.float64).reshape(-1, 2), np.asarray(vxy, dtype=np.float64).reshape(-1, 2)
        self.o.set_state(ids, xy[:, 0], xy[:, 1], vxy[:, 0], vxy[:, 1])
        self.g.set_state(ids, xy[:, 0], xy[:, 1], vxy[:, 0], vxy[:, 1])

    def oracle_step(self, dt):
        self.o.step(*dt)
        s, sxy, d = self.o.poll_events()
        self.spawned += [(int(i), (float(p[0]), float(p[1]))) for i, p in zip(s, sxy)]
        self.destroyed += sorted(int(i) for i in d)
        return s, sxy, d

    def step(self, dt, exact=True):
        """One synchronous step on both; returns the oracle's (spawned ids, spawn positions, destroyed ids)."""
        ev = self.oracle_step(dt)
        self.g.step(R.Duration(*dt))
        self.check(exact)
        return ev

    def check(self, exact=True):
        so, sg = self.o.read_state(), self.g.read_state()
        r = P.compare_states(sg, so)  # ids and next_waypoint
        if exact:
            _same(sg, so, STATE)
        else:
            assert r["vel_rel_err"] <= P.REL_TOL and r["pos_rel_err"] <= P.REL_TOL, r
        # ids, positions (as bits: NaN sources spawn at NaN) and order
        assert [(a, _pbits(p)) for a, p in self.rec.added] == [(a, _pbits(p)) for a, p in self.spawned]
        assert self.rec.removed == self.destroyed
        return so


def _spawned_sources(pair, s, sxy, sources):
    """Indices into `sources` (distinct points) of the spawns (ids s at positions sxy) of one step."""
    at = {(float(q[0]), float(q[1])): k for k, q in enumerate(sources)}
    return sorted(at[(float(p[0]), float(p[1]))] for p in sxy)


# ---- 1. the spawn probe at its threshold and its stencil edges --------------------------------------------------
def test_spawn_probe_threshold():
    """Agents at T(0.4) - 1 ulp (blocks), T and T + 1 ulp (do not) from a source, along an axis and a diagonal."""
    cfg = P.probe_threshold_configs()
    pair = Pair(80.0, 80.0, 2.0, (0.0, -40.0))
    pair.agents([a for _, a, _ in cfg])
    srcs = [s for s, _, _ in cfg]
    for s in srcs:
        pair.source(s, [(s[0], 30.0)])
    s, sxy, _ = pair.step((1, 0))
    got = _spawned_sources(pair, s, sxy, srcs)
    assert got == [k for k, (_, _, blocked) in enumerate(cfg) if not blocked] and len(got) == 4
    s, _, _ = pair.step((1, 0))  # the spawned agents stand on their sources
    assert len(s) == 0


@pytest.mark.parametrize("cell,off", P.CELLS)
def test_spawn_probe_stencil_edges(cell, off):
    """Sources whose +-0.4 lands within a few ulps of a cell edge, agents within a few ulps of that edge: inside and
    outside the 0.4 m, in the stencil's edge column and the next.  The class "within 0.4 m but inserted outside the
    probe stencil" cannot be built: the stencil floors fl(fl(source +- 0.4) - offset) / cell, the insert truncates
    fl(agent - offset) / cell, both agree on non-negative values, and norm < 0.4 puts the agent on the near side of
    fl(source +- 0.4) (rounding is monotone).  tests/test_oracle_independent.py checks that claim on these pairs."""
    cfg = P.probe_edge_configs(cell, off)
    w = 400 * cell
    pair = Pair(w, w, cell, off)
    pair.agents([a for _, a in cfg])
    srcs = [s for s, _ in cfg]
    for s in srcs:
        pair.source(s, [(s[0] + 2 * cell, s[1] + 2 * cell)])
    s, sxy, _ = pair.step((1, 0))
    near = [math.sqrt((a[0] - q[0]) ** 2 + (a[1] - q[1]) ** 2) < P.PROBE_RADIUS for q, a in cfg]
    assert _spawned_sources(pair, s, sxy, srcs) == [k for k in range(len(cfg)) if not near[k]]
    assert sum(near) > 10 and len(cfg) - sum(near) > 10


def test_spawn_probe_grid_origin_and_aliased_rows():
    """Agents left of / below the grid origin (insert cell saturates to 0, the stencil floors to -1) and, on a grid with
    more rows than columns, a source in the top rows whose stencil rows alias into the next column: an agent above the
    grid's top within 0.4 m blocks it, an agent in an aliased stencil cell farther away blocks nothing."""
    pair = Pair(8.0, 24.0, 1.0, (0.0, 0.0))
    blockers = [(-0.1, 5.0), (3.0, -0.15), (-0.2, -0.2), (3.5, 24.1), (6.5, 0.2), (4.5, 24.3)]
    srcs = [(0.2, 5.0), (3.0, 0.2), (0.05, 0.05), (3.5, 23.8), (6.5, 0.5), (7.5, 0.5)]
    ids, _, _ = pair.agents(blockers)
    for s in srcs:
        pair.source(s, [(s[0], s[1] + 3.0)])
    # saturated insert cells; (3.5, 24.1) and (4.5, 24.3) sit in the cells of (6, 0) and (7, 0) by aliasing
    assert pair.o.cell_of(np.array(blockers)).tolist() == [5, 24, 0, 48, 48, 56]
    s, sxy, _ = pair.step((1, 0))
    assert _spawned_sources(pair, s, sxy, srcs) == [5]
    pair.set_state(ids, [(7.5, 10.0 + k) for k in range(6)], np.zeros((6, 2)))
    s, sxy, _ = pair.step((1, 0))
    assert _spawned_sources(pair, s, sxy, srcs) == [0, 1, 2, 3, 4]


def test_close_coincident_and_non_finite_sources():
    """Two sources 0.3 m apart and two at the same point spawn together in the first step (every probe runs before any
    insertion), then stay blocked while their agents are near; sources at NaN and -inf are accepted and never
    blocked (the lookup grid skips them); a despawned agent next to a source does not block it in the next step."""
    pair = Pair(64.0, 64.0, 2.0)
    slow = ("constant", (0.0, 0.1))
    pair.source((10.0, 10.0), [(10.0, 40.0)], hl=slow)
    pair.source((10.3, 10.0), [(10.3, 40.0)], hl=slow)
    pair.source((20.0, 10.0), [(20.0, 40.0)], hl=slow)
    pair.source((20.0, 10.0), [(20.0, 41.0)], hl=slow)
    pair.source((NAN, 5.0), [(5.0, 5.0)], hl=("constant", (1.0, 0.0)))
    pair.source((-INF, 5.0), [(5.0, 5.0)], hl=("constant", (1.0, 0.0)))
    # A walks onto its sink at x = 40 and is removed there with its new position 0.2 m from B's source
    pair.source((30.0, 30.0), [(40.0, 30.0)], hl=("constant", (1.0, 0.0)), radius_sink=0.5)
    pair.source((41.2, 30.0), [(41.2, 60.0)], hl=("constant", (0.0, 1.0)))
    counts = []
    for step in range(16):
        s, sxy, d = pair.step((1, 0))
        counts.append(len(s))
    assert counts[0] == 8 and all(c == 4 for c in counts[1:4])  # close / coincident sources blocked
    assert pair.g.stats().nonfinite_count > 0
    assert len(pair.destroyed) >= 5  # B spawned in every step although A's removed agents ended next to it
    assert sum(1 for _, p in pair.spawned if p == (41.2, 30.0)) == 16


# ---- 2. many sources -----------------------------------------------------------------------------------------
def test_many_sources_over_a_wide_grid():
    """640 sources (three 256-source chunks of ss_spawn_kernel), spread over 1300 m (lookup cells > 1 m) with 36 of
    them 0.2 m apart inside one lookup cell; a seeded-random subset is blocked every step by agents parked 0.39 m
    away, a different subset each step.  Spawned ids, positions and the event order equal the oracle's."""
    rng = np.random.default_rng(3)
    pair = Pair(1400.0, 1400.0, 2.0, capacity=16384)
    srcs = [tuple(p) for p in rng.uniform(10.0, 1310.0, size=(604, 2))]
    srcs[300:300] = [(700.0 + 0.2 * (k % 6), 700.0 + 0.2 * (k // 6)) for k in range(36)]
    parked = 120
    park = np.stack([5.0 + 10.0 * np.arange(parked), np.full(parked, 1395.0)], axis=1)
    ids, _, _ = pair.agents(park)
    for p in srcs:
        pair.source(p, [(p[0], p[1] + 3.0)], hl=("constant", (0.0, 1.0)))
    srcs = np.array(srcs)
    hit_chunks = 0
    for step in range(6):
        pick = rng.choice(len(srcs), parked, replace=False)
        ang = rng.uniform(0, 2 * math.pi, parked)
        xy = srcs[pick] + 0.39 * np.stack([np.cos(ang), np.sin(ang)], axis=1)
        pair.set_state(ids, xy, np.zeros((parked, 2)))
        s, sxy, d = pair.step((1, 0))
        got = set(_spawned_sources(pair, s, sxy, list(srcs)))
        assert not got & set(pick.tolist())
        hit_chunks += min(k // 256 for k in pick) == 0 and max(got) >= 512
    assert hit_chunks == 6 and len(pair.destroyed) > 0


# ---- 3. generator rounding and degenerate parameters ------------------------------------------------------------
def test_generator_rounding_and_degenerate_rates():
    rates = [0.0, -1.0, NAN, INF, 1e308, 1.0, math.nextafter(1.0, 0.0), 5.0]
    pair = Pair(128.0, 128.0, 2.0)
    for k, rate in enumerate(rates):
        pair.source((5.0 + 10.0 * k, 5.0), [(5.0 + 10.0 * k, 100.0)], hl=("constant", (0.0, 1.0)), rate=rate)
    for dt in ((0, 500_000_000), (0, 500_000_000), (0, 0), (0, 500_000_000)):
        s, sxy, _ = pair.step(dt)
        # round(dt * rate) > 0: inf and 1e308 saturate, 0.5 rounds to 1, 0.5 - 2^-54 to 0, 2.5 to 3 (still one agent)
        assert [int((p[0] - 5.0) / 10.0) for p in sxy] == ([] if dt == (0, 0) else [3, 4, 5, 7])


def test_degenerate_sink_radii_sink_on_source_and_loops():
    """radius_sink 0, -0.5 and NaN never remove, inf and 1e300 remove in the spawn step; a sink on the source: every
    agent lives exactly one step; loop_forever with one waypoint and with three (the wrap 2 -> 0)."""
    pair = Pair(128.0, 128.0, 2.0)
    for k, r in enumerate([0.0, -0.5, NAN, INF, 1e300]):
        pair.source((5.0 + 10.0 * k, 5.0), [(5.0 + 10.0 * k, 7.0)], hl=("constant", (0.0, 1.0)), radius_sink=r)
    pair.source((5.0, 20.0), [(5.0, 20.0)], hl=("constant", (1.0, 0.0)))
    pair.source((5.0, 40.0), [(8.0, 40.0)], hl=("constant", (1.0, 0.0)), loop=True)
    pair.source((5.0, 60.0), [(7.0, 60.0), (9.0, 60.0), (11.0, 60.0)], hl=("constant", (1.0, 0.0)), loop=True,
                radius_sink=0.6)
    history = {}
    for step in range(12):
        s, sxy, d = pair.step((1, 0))
        assert len(s) == 8 and sorted(d.tolist()) == sorted(s[[3, 4, 5]].tolist())
        st = pair.o.read_state()
        for i, w in zip(st["id"].tolist(), st["next_waypoint"].tolist()):
            history.setdefault(i, []).append(w)
    assert any(2 in h and 0 in h[h.index(2):] for h in history.values())  # the three-waypoint loop wraps


# ---- 4. the sink / waypoint threshold --------------------------------------------------------------------------
def _sink_pair(cfg, make_pair):
    """Three source sinks per configuration, spawning their agent at the threshold point: waypoints [wp, far]
    (advance), [wp] (removal) and, looping, [spawn point, wp] (the agent advances to 1 in its spawn step, then wraps
    or not)."""
    pair = make_pair()
    for kind in ("advance", "remove", "wrap"):
        for r, wp, a, _ in cfg:
            wps = {"advance": [wp, (wp[0], 25.0)], "remove": [wp], "wrap": [a, wp]}[kind]
            pair.source(a, wps, radius_sink=r, loop=kind == "wrap")
    return pair


def test_sink_threshold():
    cfg = P.sink_threshold_configs()
    n = len(cfg)
    pair = _sink_pair(cfg, lambda: Pair(400.0, 400.0, 2.0, (0.0, -200.0)))
    _, _, d1 = pair.step((1, 0))
    pair.step((1, 0))
    wp = dict(zip(*[pair.o.read_state()[k].tolist() for k in ("id", "next_waypoint")]))
    inside = [c[3] for c in cfg]
    assert [wp[i] for i in range(n)] == [1 if v else 0 for v in inside] and sum(inside) == 10
    assert sorted(d1.tolist()) == [n + i for i in range(n) if inside[i]]
    assert [wp[2 * n + i] for i in range(n)] == [0 if v else 1 for v in inside]


# ---- 5. the route follower -------------------------------------------------------------------------------------
def test_route_follower_threshold_and_degenerate_routes():
    """Agents at T(0.1) - 1 ulp (advance), T and T + 1 ulp from their route point 0, along an axis and a diagonal;
    an agent exactly on the point of a one-point route (0 / 0: NaN, cell 0, counted as non-finite); consecutive
    duplicate route points."""
    pair = Pair(256.0, 256.0, 2.0, (0.0, -128.0))
    advanced = []
    for k in range(6):
        p, qs = P.threshold_points(0.1, 5.0 + 11.0 * k, k >= 3)
        ids, ohl, ghl = pair.agents([qs[k % 3]], hl=("route", [tuple(p), (p[0] + 3.0, p[1] + 4.0)]))
        pair.o.hl_set_target(ohl, ids)
        pair.g.route_set_target(ids)
        advanced.append(k % 3 == 0)
    one = (80.0, 10.0)
    dup = [(90.0, 10.0), (90.0, 10.0), (95.0, 10.0)]
    for xy, route in [(one, [one]), (dup[0], dup), ((90.05, 20.0), [(90.0, 20.0), (90.0, 20.0), (95.0, 20.0)])]:
        ids, ohl, ghl = pair.agents([xy], hl=("route", route))
        pair.o.hl_set_target(ohl, ids)
        pair.g.route_set_target(ids)
    pair.step((0, 250_000_000))
    st = pair.o.read_state()
    heading_on = [st["vy"][k] > 0.5 for k in range(6)]  # towards route point 1: (3, 4) / 5
    assert heading_on == advanced
    assert np.isnan(st["x"][6]) and np.isnan(st["x"][7]) and not np.isnan(st["x"][8])
    assert pair.g.stats().nonfinite_count >= 2
    for _ in range(4):
        pair.step((0, 250_000_000))


def test_route_longer_than_256_points_with_set_target_mid_stream():
    """A 300-point route walked one point per step (0.05 m apart, unit speed, dt = 0.05 s): the route index passes
    255.  Plain agents enter the planner with route_set_target after a few steps of standing still."""
    route = [(2.0 + 0.05 * k, 10.0 + 0.001 * (k % 3)) for k in range(300)]
    pair = Pair(64.0, 64.0, 2.0)
    ids, ohl, ghl = pair.agents([(2.0, 10.0), (1.9, 10.02), (2.5, 9.0)], hl=("route", route))
    dt = (0, 50_000_000)
    for _ in range(3):
        pair.step(dt)
    pair.o.hl_set_target(ohl, ids[:2])
    pair.g.route_set_target(ids[:2])
    for step in range(5):
        pair.step(dt)
    pair.o.hl_set_target(ohl, ids[2:])
    pair.g.route_set_target(ids[2:])
    for step in range(290):
        pair.step(dt)
    st = pair.o.read_state()
    assert st["x"][0] > route[270][0] and st["x"][1] > route[260][0]


@pytest.mark.parametrize("wiggle", [0.1, 0.05])
def test_route_followers_with_zanlungo_on_every_kernel_form(wiggle):
    """Route-following source sinks under the Zanlungo planner, in lanes of two 0.5 m apart: one lane straight, the
    other zigzagging +-`wiggle` around its line, so that neighbours move relative to each other (finite t_i, forces);
    plain route followers that enter the planner with route_set_target.  The three forms of the step kernel bit for
    bit with each other, within 1e-9 of the oracle, every step from the oracle's state."""
    pairs = [Pair(64.0, 64.0, 2.0, capacity=512) for _ in range(3)]
    for form, pair in zip((1, 2, 3), pairs):
        pair.g.set_option(N.RCS_OPT_STEP_KERNEL, form)
        pair.g.set_trace(True)
        pair.o.enable_trace(True)
        for k in range(3):
            y = 10.0 + 12.0 * k
            zig = [(5.0 + 1.5 * j, y + 0.5 + wiggle * (-1) ** j) for j in range(8)] + [(18.0, y + 0.5)]
            for yy, route in ((y, [(18.0, y)]), (y + 0.5, zig)):
                pair.source((4.0, yy), [(18.0, yy)], hl=("route", route), lp=("zanlungo", ZA), radius_sink=0.6,
                            rate=2.0, eyesight=2.0)
        xy = np.stack([10.0 + 3.0 * np.arange(8), 44.0 + 2.0 * np.arange(8)], axis=1)  # one row each
        ids, ohl, ghl = pair.agents(xy, hl=("route", [(60.0, 50.0)]), lp=("zanlungo", ZA), eyesight=2.0)
        pair.o.hl_set_target(ohl, ids[::2])
        pair.g.route_set_target(ids[::2])
    finite = 0
    for step in range(36):
        for pair in pairs:
            P.resync(pair.g, pair.o)
            pair.step((0, 500_000_000), exact=False)
            t = P.compare_traces(pair.g.read_trace(), pair.o.read_trace())
            assert t["force_rel_err"] <= P.REL_TOL
        finite += t["finite_tti"]
        t1, s1 = pairs[0].g.read_trace(), pairs[0].g.read_state()
        for pair in pairs[1:]:
            _same(t1, pair.g.read_trace(), ("id", "nb_offsets", "nb_ids", "t_i", "fx", "fy"))
            _same(s1, pair.g.read_state(), STATE + ("next_waypoint",))
    st = pairs[0].o.read_state()
    assert finite > 1000 and len(pairs[0].destroyed) > 40 and np.isfinite(st["x"]).all()


# ---- 6. asynchronous streams against the oracle ----------------------------------------------------------------
@pytest.mark.parametrize("graphs", [1, 0])
def test_async_stream_under_the_coarse_launch_bound(graphs):
    """60 committed step_async calls, synced every 10 steps and compared with the oracle there.  4060 parked agents and
    8 sources (constant and route planners, NoLocalPlan): the live count crosses 4096, a multiple of the launch bound's
    granule max(32 x sources, 4096), between the first two syncs, at a capacity of 20000.  A source sink whose agents are
    removed 0.2 m from another source checks that agents flagged for removal do not block the next step's probe."""
    pair = Pair(256.0, 256.0, 2.0, capacity=20000)
    pair.g.set_option(N.RCS_OPT_GRAPHS, graphs)
    park = np.stack([2.0 + 0.5 * (np.arange(4060) % 500), 200.0 + 0.5 * (np.arange(4060) // 500)], axis=1)
    pair.agents(park)
    for k in range(3):
        y = 10.0 + 10.0 * k
        pair.source((5.0, y), [(20.0, y)], hl=("constant", (1.0, 0.0)), radius_sink=0.6)
        pair.source((5.0, y + 100.0), [(20.0, y + 100.0)], hl=("route", [(12.0, y + 101.0), (20.0, y + 100.0)]))
    pair.source((30.0, 60.0), [(40.0, 60.0)], hl=("constant", (1.0, 0.0)), radius_sink=0.5)
    pair.source((40.7, 60.0), [(40.7, 90.0)], hl=("constant", (0.0, 1.0)))
    dt = (0, 500_000_000)
    counts = [pair.g.agent_count()]
    for rounds in range(6):
        for _ in range(10):
            pair.oracle_step(dt)
            pair.g.step_async(R.Duration(*dt))
        pair.g.sync()
        pair.g._dispatch_events()
        pair.check()
        counts.append(pair.g.agent_count())
    assert counts[0] < 4096 < counts[1] and max(counts) * 4 <= 20000
    assert len(pair.destroyed) > 20
    assert sum(1 for _, p in pair.spawned if p == (40.7, 60.0)) == 60  # never blocked by removed agents
    assert (pair.g.graph_stats()[0] > 0) == bool(graphs)


# ---- 7. strips ------------------------------------------------------------------------------------------------
def _strip_scene(xy):
    xy = np.asarray(xy, dtype=np.float64).reshape(-1, 2)
    return SC.Scene(name="ss-edges", width=400.0, height=400.0, cell=2.0, offset=(0.0, -200.0), xy=xy,
                    vxy=np.zeros_like(xy), eyesight=1.0, hl=("constant", STILL), lp=("none",))


def _strips_vs_single(scene, makers, world, bounds, steps=3):
    single = SC.build_simulation(scene, capacity=1024)
    grp = LocalStripGroup(scene, world, capacity=1024, halo_capacity=256, boundaries=bounds)
    rs, rg = Recorder(), Recorder()
    single.add_event_listener(rs)
    grp.add_event_listener(rg)
    keep = []
    for make in makers:
        ss = make()
        keep.append(ss)
        single.add_source_sink(ss)
        grp.add_source_sink(make)
    for _ in range(steps):
        single.step(R.Duration(1, 0))
        grp.step(R.Duration(1, 0))
        grp.dispatch_events()
        _same(single.read_state(), grp.read_state(), STATE + ("next_waypoint",))
    assert sorted(rg.added) == sorted(rs.added) and sorted(rg.removed) == sorted(rs.removed)
    return single, rs


def _ss(src, wps, radius_sink=0.5, loop=False):
    return lambda: R.SourceSink(tuple(src), radius_sink, R.MonotonicCrowd(1.0), R.ConstantVelocityPlan(STILL),
                                R.NoLocalPlan(), [tuple(p) for p in wps], loop, 1.0)


# boundaries between the threshold configurations (sources 11 m apart from x = 5: columns 2, 8, 13, 19, ...)
STRIP_BOUNDS = {2: [0, 40, 200], 3: [0, 25, 90, 200]}


@pytest.mark.parametrize("world", [2, 3])
def test_probe_and_sink_thresholds_on_strips(world):
    probe = P.probe_threshold_configs()
    sink = P.sink_threshold_configs(x0=71.0)
    scene = _strip_scene([a for _, a, _ in probe])
    makers = [_ss(s, [(s[0], 30.0)]) for s, _, _ in probe]
    for kind in ("advance", "remove", "wrap"):
        for r, wp, a, _ in sink:
            wps = {"advance": [wp, (wp[0], 25.0)], "remove": [wp], "wrap": [a, wp]}[kind]
            makers.append(_ss(a, wps, radius_sink=r, loop=kind == "wrap"))
    single, rs = _strips_vs_single(scene, makers, world, STRIP_BOUNDS[world])
    assert len(rs.removed) >= 10 and sum(1 for _, p in rs.added if p[1] < 1.0 and p[0] < 70.0) > 0


@pytest.mark.parametrize("cell,off", P.CELLS[1:3])
def test_probe_stencil_edges_on_strips(cell, off):
    cfg = P.probe_edge_configs(cell, off)
    w = 400 * cell
    xy = np.array([a for _, a in cfg])
    scene = SC.Scene(name="ss-stencil", width=w, height=w, cell=cell, offset=off, xy=xy, vxy=np.zeros_like(xy),
                     eyesight=1.0, hl=("constant", STILL), lp=("none",))
    cols = sorted({int(math.floor((s[0] - off[0]) / cell)) for s, _ in cfg})
    mid = next(c for c in range(cols[len(cols) // 2], 400) if all(abs(c - q) > 2 for q in cols))
    makers = [_ss(s, [(s[0] + 2 * cell, s[1] + 2 * cell)]) for s, _ in cfg]
    _strips_vs_single(scene, makers, 2, [0, mid, 400], steps=2)


def test_strip_probe_refusal_edge():
    """A source whose probe stencil starts exactly at the strip's first column is accepted, one ulp further left (the
    stencil reaches the previous column) it is refused -- on every rank alike -- and the refused call changes nothing."""
    scene = _strip_scene([(10.0, 10.0), (150.0, -20.0)])
    bounds = [0, 30, 200]
    x = 60.4  # column 30 starts at x = 60
    while math.floor((x - 0.4) / 2.0) >= 30:
        x = math.nextafter(x, -INF)
    bad, good = x, math.nextafter(x, INF)
    assert math.floor((good - 0.4) / 2.0) == 30 and math.floor((bad - 0.4) / 2.0) == 29

    def build(refused):
        grp = LocalStripGroup(scene, 2, capacity=256, halo_capacity=64, boundaries=bounds)
        if refused:
            for sm in grp.sims:  # every rank says no
                assert strip_columns(sm, 1, 2) == (30, 200)
                with pytest.raises(R.CrowdsimError):
                    sm.add_source_sink(_ss((bad, 0.0), [(bad + 5.0, 0.0)])())
        grp.add_source_sink(_ss((good, 0.0), [(good + 5.0, 0.0)]))
        grp.add_source_sink(_ss((good, 8.0), [(good, 12.0)]))
        return grp

    a, b = build(True), build(False)
    for _ in range(4):
        a.step(R.Duration(1, 0))
        b.step(R.Duration(1, 0))
        _same(a.read_state(), b.read_state(), STATE + ("next_waypoint",))
    assert a.read_state()["id"].tolist() == [0, 1, 2, 3]


# ---- 8. host-evaluated planners get set_target at every waypoint ------------------------------------------------
def test_host_planner_gets_set_target_at_each_waypoint():
    """lib.rs:326-333: an agent advancing from waypoint k to k + 1 gets set_target(agent, waypoints[k + 1],
    (radius_sink, radius_sink)) with its state from before the step; not at the loop wrap, not when it is removed."""

    class Towards(R.HighLevelPlanner):
        def __init__(self):
            self.target, self.calls = {}, []

        def set_target(self, agent, point, tolerance):
            self.target[agent.agent_id] = point
            self.calls.append((agent.agent_id, agent.position, agent.next_waypoint, point, tolerance))

        def get_desired_velocity(self, agent, time):
            t = self.target.get(agent.agent_id)
            if t is None:
                return None
            dx, dy = t[0] - agent.position[0], t[1] - agent.position[1]
            n = math.hypot(dx, dy)
            return (dx / n, dy / n) if n > 0 else (0.0, 0.0)

    wps = [(10.0, 10.0), (15.0, 12.0), (20.0, 10.0)]
    runs = []
    for loop in (False, True):
        hl = Towards()
        g = R.Simulation(R.LocationHash2D(64.0, 64.0, 2.0, (0.0, 0.0), capacity=256))
        g.add_source_sink(R.SourceSink((5.0, 10.0), 0.6, R.MonotonicCrowd(1.0), hl, R.NoLocalPlan(), wps, loop, 2.0))
        want = []
        for step in range(60):
            before = g.read_state()
            g.step(R.Duration(0, 500_000_000))
            after = g.read_state()
            pre = {int(i): k for k, i in enumerate(before["id"])}
            for k, i in enumerate(after["id"].tolist()):
                j = pre.get(i)
                w0 = int(before["next_waypoint"][j]) if j is not None else 0
                if int(after["next_waypoint"][k]) == w0 + 1:
                    pos = (float(before["x"][j]), float(before["y"][j])) if j is not None else (5.0, 10.0)
                    want.append((i, pos, w0, wps[w0 + 1], (0.6, 0.6)))
        got = [c for c in hl.calls if not (c[2] == 0 and c[3] == wps[0] and c[1] == (5.0, 10.0))]
        assert got == want and len(want) > 10
        runs.append(want)
    assert any(w[2] == 1 for w in runs[1])  # the loop runs reach the second advance too
