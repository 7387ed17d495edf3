"""GPU: the route-table planner (RouteTablePlan, rcs_hl_route_table) -- RMFPlanner with a caller-filled route cache
driving source sinks through every waypoint on the device.  Compared with the oracle's RouteTablePlan
(tests/oracle_route_table.cpp) bit for bit under NoLocalPlan (only IEEE + - * / sqrt) and within 1e-9 under
Zanlungo; across the step-kernel forms, CUDA graphs, asynchronous streams and strips bit for bit."""
import ctypes as C

import numpy as np
import pytest

import oracle_ffi as O
import oracle_route_table as RT
import parity as P
import rmf_crowdsim_b200 as R
from rmf_crowdsim_b200 import _native as N
from rmf_crowdsim_b200 import scenes as SC
from rmf_crowdsim_b200.strips import LocalStripGroup
from parity import _same

pytestmark = pytest.mark.gpu

ZA = (0.05, 1.0, 0.0, 0.5, 1.0, 0.2)
ZS = (0.05, 1.0, 0.0, 0.5, 1.0, 0.05)  # agent radius 0.05 m: the sinks spawn agents in single file 0.4 m apart
STATE = ("id", "x", "y", "vx", "vy", "next_waypoint")
DT = (0, 100_000_000)


class Recorder(R.EventListener):
    def __init__(self):
        self.added, self.removed = [], []

    def agent_spawned(self, position, agent):
        self.added.append((agent, position))

    def agent_destroyed(self, agent):
        self.removed.append(agent)


def _approach(w, u, n=3, step=0.5):
    """A leg that reaches w along direction u: n points before it, `step` apart, then w."""
    return [(w[0] - step * k * u[0], w[1] - step * k * u[1]) for k in range(n, 0, -1)] + [tuple(w)]


def stream_sinks():
    """Source sinks of the multi-waypoint stream: (source, waypoints, routes, radius_sink, loop, shared-planner key).
    Sinks with the same key share one planner (one table)."""
    out = []
    # 1. A -> B -> A: the leg of A serves waypoints 0 and 2
    A, B = (14.013, 10.021), (14.037, 14.011)
    out.append(((10.0, 10.0), [A, B, A], {A: [(12.01, 10.0), A], B: [(14.0, 12.03), B]}, 0.5, False, None))
    # 2. one-point legs in a cycle; the last leg runs on to the first waypoint, so after the loop wrap (no set_target)
    #    the agent follows it there and the cycle goes on
    P1, P2, P3 = (34.011, 10.017), (34.023, 14.031), (30.019, 14.007)
    out.append(((30.0, 10.0), [P1, P2, P3], {P1: [P1], P2: [P2], P3: [P3, (30.5, 10.9), P1]}, 0.5, True, None))
    # 3. a 300-point leg (a 0.05 m zigzag: the follower advances one point per step and lags behind), then a short one
    zz = [(50.0 + 0.05 * j, 10.0 + 0.02 * (-1) ** j) for j in range(300)]
    Q2 = (65.013, 14.029)
    out.append(((49.0, 10.0), [zz[-1], Q2], {zz[-1]: zz, Q2: [(64.9, 12.0), Q2]}, 0.5, False, None))
    # 4. radius_sink (1.2 m) reached while the follower still heads for an earlier point of the leg
    R1, R2, R3 = (74.3, 10.1), (74.3, 15.2), (70.1, 15.2)
    out.append(((70.0, 10.1), [R1, R2, R3], {R1: _approach(R1, (1, 0)), R2: _approach(R2, (0, 1)),
                                              R3: _approach(R3, (-1, 0))}, 1.2, False, None))
    # 5. six waypoints around a rectangle, loop_forever, mid-leg switches everywhere
    c = [(94.0, 10.2), (98.1, 10.2), (98.1, 13.3), (98.1, 16.4), (94.0, 16.4), (90.3, 13.3)]
    dirs = [(1, 0), (1, 0), (0, 1), (0, 1), (-1, 0), (-1, -1)]
    out.append(((90.0, 10.2), c, {w: _approach(w, (d[0] / np.hypot(*d), d[1] / np.hypot(*d)))
                                  for w, d in zip(c, dirs)}, 1.2, True, None))
    # 6 + 7. two sinks on one table, walking against each other (Zanlungo forces)
    X1, X2 = (16.2, 39.4), (10.2, 42.6)
    table = {X1: [(13.1, 39.4), X1], X2: [(13.1, 42.6), X2]}
    out.append(((10.0, 40.0), [X1, X2], table, 0.5, False, "xx"))
    out.append(((16.0, 40.0), [X2, X1], table, 0.5, False, "xx"))
    # 8. loop wrap onto a one-point leg: the agent keeps that leg and stays at its target
    Y1, Y2 = (30.5, 43.2), (36.3, 43.7)
    out.append(((30.0, 40.0), [Y1, Y2], {Y1: [(33.0, 40.5), (33.0, 43.0), Y1], Y2: [Y2]}, 0.5, True, None))
    # 9. a leg whose last point is beyond its waypoint, and a repeated one-point leg
    Z1, Z2 = (52.2, 40.3), (56.1, 40.3)
    out.append(((50.0, 40.3), [Z1, Z2, Z1, Z2], {Z1: [Z1, (53.0, 40.3)], Z2: [Z2]}, 0.4, False, None))
    return out


class TPair:
    """The same configuration in the oracle (with RouteTablePlan) and on the device."""

    def __init__(self, w=120.0, h=120.0, cell=2.0, capacity=4096, lp=("none",), oracle=True):
        self.o = RT.RouteTableOracle(w, h, cell, (0.0, 0.0)) if oracle else None
        self.g = R.Simulation(R.LocationHash2D(w, h, cell, (0.0, 0.0), capacity=capacity))
        self.rec = Recorder()
        self.g.add_event_listener(self.rec)
        self.lp = lp
        self.glp = R.NoLocalPlan() if lp[0] == "none" else R.Zanlungo(*lp[1])
        self.olp = None if not oracle else (self.o.lp_none() if lp[0] == "none" else self.o.lp_zanlungo(*lp[1]))
        self.tables = {}
        self.sinks = []  # (source, waypoints, radius, loop, routes)
        self.spawned, self.destroyed = [], []

    def table(self, routes, key=None):
        k = key if key is not None else len(self.tables)
        if k not in self.tables:
            self.tables[k] = (self.o.hl_route_table(routes) if self.o else None, R.RouteTablePlan(routes))
        return self.tables[k]

    def source(self, src, wps, routes, radius, loop, key=None, rate=10.0, eyesight=2.0):
        ohl, ghl = self.table(routes, key)
        if self.o:
            self.o.add_source_sink(src, radius, rate, ohl, self.olp, wps, loop, eyesight)
        self.g.add_source_sink(R.SourceSink(tuple(src), radius, R.MonotonicCrowd(rate), ghl, self.glp,
                                            [tuple(p) for p in wps], loop, eyesight))
        self.sinks.append((tuple(src), [tuple(p) for p in wps], radius, loop, routes))

    def oracle_step(self):
        self.o.step(*DT)
        s, sxy, d = self.o.poll_events()
        self.spawned += [(int(i), (float(p[0]), float(p[1]))) for i, p in zip(s, sxy)]
        self.destroyed += sorted(int(i) for i in d)

    def check(self, exact):
        so, sg = self.o.read_state(), self.g.read_state()
        r = P.compare_states(sg, so)
        if exact:
            _same(sg, so, STATE[:5])
        else:
            assert r["vel_rel_err"] <= P.REL_TOL and r["pos_rel_err"] <= P.REL_TOL, r
        assert self.rec.added == self.spawned and self.rec.removed == self.destroyed
        return so


def build_stream(pair):
    """Under Zanlungo without the six-waypoint loop and the two sinks whose agents crowd at a leg's end: agents that
    meet there leave the grid within 300 steps, in the reference as in the oracle."""
    for k, (src, wps, routes, radius, loop, key) in enumerate(stream_sinks()):
        if pair.lp[0] == "none" or k not in (4, 7, 8):
            pair.source(src, wps, routes, radius, loop, key)
    return pair


def classify(pair, before, after):
    """Counts of the event classes between two oracle (or device) states: advances, advances while the agent was
    still farther from the waypoint than the leg's second-to-last point is (the follower was mid-leg), loop wraps."""
    sink_of = {a: pair.sinks[[s[0] for s in pair.sinks].index(p)] for a, p in pair.rec.added}
    pre = {int(a): k for k, a in enumerate(before["id"])}
    adv = mid = wrap = 0
    for k, a in enumerate(after["id"]):
        j = pre.get(int(a))
        if j is None:
            continue
        w0, w1 = int(before["next_waypoint"][j]), int(after["next_waypoint"][k])
        src, wps, radius, loop, routes = sink_of[int(a)]
        if w1 == w0 + 1:
            adv += 1
            leg = routes[wps[w0]]
            if len(leg) > 1:
                d = np.hypot(before["x"][j] - wps[w0][0], before["y"][j] - wps[w0][1])
                mid += d > np.hypot(leg[-2][0] - wps[w0][0], leg[-2][1] - wps[w0][1])
        elif w1 == 0 and w0 == len(wps) - 1 and loop:
            wrap += 1
    return adv, mid, wrap


# ---- 1. the multi-waypoint stream against the oracle ------------------------------------------------------------
@pytest.mark.parametrize("lp", [("none",), ("zanlungo", ZS)], ids=["nolocalplan", "zanlungo"])
def test_multi_waypoint_stream_against_the_oracle(lp):
    """Nine source sinks (six under Zanlungo) with 2 to 6 waypoints (a repeated waypoint, one-point legs, a 300-point
    leg, loop_forever, sink radii reached mid-leg, two sinks on one table), 320 steps, read_state() compared after
    every step."""
    exact = lp[0] == "none"
    pair = build_stream(TPair(lp=lp))
    adv = mid = wrap = 0
    before = pair.o.read_state()
    for step in range(320):
        if not exact:
            P.resync(pair.g, pair.o)
        pair.oracle_step()
        pair.g.step(R.Duration(*DT))
        after = pair.check(exact)
        a, m, w = classify(pair, before, after)
        adv, mid, wrap = adv + a, mid + m, wrap + w
        before = after
    assert adv > 100 and mid > 20 and wrap > 5 and len(pair.destroyed) > 10, (adv, mid, wrap, len(pair.destroyed))
    assert np.isfinite(before["x"]).all()


# ---- 2. kernel forms, graphs and asynchronous streams agree bit for bit ----------------------------------------------
def test_kernel_forms_graphs_and_async_streams_agree():
    """The Zanlungo stream under RCS_OPT_STEP_KERNEL 1, 2 and 3, with CUDA graphs on and off, stepped with 60 step_async
    calls between syncs, and once synchronously: every run bit-identical at every sync."""
    runs = [(None, None, False)] + [(form, graphs, True) for form in (1, 2, 3) for graphs in (1, 0)]
    states = []
    for form, graphs, asy in runs:
        pair = TPair(lp=("zanlungo", ZS), oracle=False)
        if form is not None:
            pair.g.set_option(N.RCS_OPT_STEP_KERNEL, form)
            pair.g.set_option(N.RCS_OPT_GRAPHS, graphs)
        build_stream(pair)
        snaps = []
        for rounds in range(5):
            for _ in range(60):
                if asy:
                    pair.g.step_async(R.Duration(*DT))
                else:
                    pair.g.step(R.Duration(*DT))
            pair.g.sync()
            pair.g._dispatch_events()
            snaps.append(pair.g.read_state())
        states.append((snaps, list(pair.rec.added), list(pair.rec.removed)))
        if form is not None and graphs:
            assert pair.g.graph_stats()[0] > 0
    ref = states[0]
    assert len(ref[2]) > 10
    for snaps, added, removed in states[1:]:
        for a, b in zip(ref[0], snaps):
            _same(a, b, STATE)
        assert added == ref[1] and removed == ref[2]


# ---- 3. strips ------------------------------------------------------------------------------------------------
def strip_makers():
    """Sources 0.05 m off the 0.1 m lattice of their walk, so that an agent crosses x = 32 (column 16) in the very step
    in which it reaches a waypoint 0.5 m beyond (advance on the old position, ownership by the new one); others cross x =
    32 and x = 80 in the middle of a leg."""
    specs = []  # (source, waypoints, routes, radius_sink, loop, Zanlungo)
    for k in range(3):
        y = 10.0 + 6.0 * k
        W1, W2 = (32.4, y), (35.0 + k, y + 3.0)
        specs.append(((30.05, y), [W1, W2], {W1: [(31.0, y), W1], W2: [(34.0, y + 1.0), W2]}, 0.5, False, False))
        V1, V2 = (83.0, y + 0.3), (84.1, y + 3.0)
        specs.append(((78.05, y), [V1, V2], {V1: [(79.0, y + 0.1), V1], V2: [V2]}, 0.5, False, True))
    specs.append(((26.05, 40.0), [(36.0, 40.2), (26.5, 40.7)],
                  {(36.0, 40.2): [(36.0, 40.2)], (26.5, 40.7): [(31.0, 40.9), (26.5, 40.7)]}, 0.5, True, False))
    return [(lambda s=s: R.SourceSink(s[0], s[3], R.MonotonicCrowd(10.0), R.RouteTablePlan(s[2]),
                                      R.Zanlungo(*ZS) if s[5] else R.NoLocalPlan(), list(s[1]), s[4], 2.0))
            for s in specs]


STRIP_BOUNDS = {2: [0, 16, 60], 3: [0, 16, 40, 60]}


@pytest.mark.parametrize("world", [2, 3])
def test_strips_match_one_handle(world):
    xy = np.array([[110.0, 70.0]])
    scene = SC.Scene(name="route-table-strips", width=120.0, height=120.0, cell=2.0, offset=(0.0, 0.0), xy=xy,
                     vxy=np.zeros_like(xy), eyesight=1.0, hl=("constant", (0.0, 0.0)), lp=("none",))
    single = SC.build_simulation(scene, capacity=2048)
    grp = LocalStripGroup(scene, world, capacity=2048, halo_capacity=512, boundaries=STRIP_BOUNDS[world])
    rs, rg = Recorder(), Recorder()
    single.add_event_listener(rs)
    grp.add_event_listener(rg)
    keep = []
    for make in strip_makers():
        ss = make()
        keep.append(ss)
        single.add_source_sink(ss)
        grp.add_source_sink(make)
    bounds_x = [2.0 * b for b in STRIP_BOUNDS[world][1:-1]]
    rank = lambda x: np.searchsorted(bounds_x, x, side="right")  # noqa: E731
    at_switch = mid_leg = 0
    before = single.read_state()
    for _ in range(160):
        single.step(R.Duration(*DT))
        grp.step(R.Duration(*DT))
        grp.dispatch_events()
        after = single.read_state()
        _same(after, grp.read_state(), STATE)
        pre = {int(a): k for k, a in enumerate(before["id"])}
        for k, a in enumerate(after["id"]):
            j = pre.get(int(a))
            if j is not None and rank(before["x"][j]) != rank(after["x"][k]):
                if after["next_waypoint"][k] != before["next_waypoint"][j]:
                    at_switch += 1
                else:
                    mid_leg += 1
        before = after
    assert sorted(rg.added) == sorted(rs.added) and sorted(rg.removed) == sorted(rs.removed)
    assert at_switch >= 3 and mid_leg >= 10 and len(rs.removed) > 5, (at_switch, mid_leg, len(rs.removed))


# ---- 4. a one-leg table is RouteFollowPlan ---------------------------------------------------------------------
@pytest.mark.parametrize("lp", [("none",), ("zanlungo", ZS)], ids=["nolocalplan", "zanlungo"])
def test_one_leg_table_is_route_follow_plan(lp):
    sims = []
    for kind in ("route", "table"):
        g = R.Simulation(R.LocationHash2D(64.0, 64.0, 2.0, (0.0, 0.0), capacity=1024))
        glp = R.NoLocalPlan() if lp[0] == "none" else R.Zanlungo(*lp[1])
        keep = []
        for k in range(4):
            y = 6.0 + 9.0 * k
            sink = (30.0 + k, y + 1.0)
            route = [(10.0, y + 0.3), (10.0 + 0.07 * k, y + 0.3)] + [(12.0 + 0.6 * j, y + 0.1 * (-1) ** j)
                                                                    for j in range(20)] + [sink]
            hl = R.RouteFollowPlan(route) if kind == "route" else R.RouteTablePlan({sink: route})
            keep.append(hl)
            # the loop wrap keeps agents at the sink: only without local forces
            loop = k == 3 and lp[0] == "none"
            g.add_source_sink(R.SourceSink((5.0, y), 0.6, R.MonotonicCrowd(10.0), hl, glp, [sink], loop, 2.0))
        g._keep = keep
        sims.append(g)
    for _ in range(300):
        for g in sims:
            g.step(R.Duration(*DT))
        _same(sims[0].read_state(), sims[1].read_state(), STATE)
    assert sims[0].agent_count() > 50


# ---- 5. plain agents and route_table_set_target ------------------------------------------------------------------
def test_set_target_on_plain_agents_against_the_oracle():
    pair = TPair(64.0, 64.0, 2.0, capacity=512)
    T1, T2, T3 = (40.0, 10.0), (10.0, 40.0), (40.0, 40.0)
    routes = {T1: [(20.0, 12.0), T1], T2: [(12.0, 25.0), (11.0, 30.0), T2], T3: [T3]}
    ohl, ghl = pair.table(routes)
    xy = np.stack([10.0 + 0.9 * np.arange(12), 10.0 + 0.7 * np.arange(12)], axis=1)
    ids = pair.o.add_agents(xy, ohl, pair.olp, 1.0)
    assert list(pair.g.add_agents(xy, ghl, pair.glp, 1.0)) == ids.tolist()
    ohl2, ghl2 = pair.table({T1: [T1]})
    other = pair.o.add_agents([(50.0, 50.0)], ohl2, pair.olp, 1.0)
    assert list(pair.g.add_agents([(50.0, 50.0)], ghl2, pair.glp, 1.0)) == other.tolist()
    pair.o.poll_events()
    pair.rec.added.clear()
    # an id listed twice takes its last target; ids[10:] stay outside the cache (velocity 0)
    sel = list(ids[:8]) + [ids[0]]
    tg = [T1, T2, T3, T1, T2, T3, T1, T2, T3]
    pair.o.hl_route_table_set_target(ohl, sel, tg)
    pair.g.route_table_set_target(ghl, sel, tg)
    pair.o.hl_route_table_set_target(ohl2, other, [T1])
    pair.g.route_table_set_target(ghl2, other, [T1])
    refusals = [(ghl, [ids[0], 10**9], [T1, T1]),          # unknown id
                (ghl, [ids[1], other[0]], [T1, T1]),       # an agent of another planner
                (ghl, [ids[1], ids[2]], [T1, (40.0, 10.5)]),  # a point without a leg
                (ghl, [ids[1]], [(float("nan"), 10.0)]),
                (ghl2, [other[0]], [T2])]
    for step in range(80):
        if step == 30:
            pair.o.hl_route_table_set_target(ohl, [ids[3], ids[10]], [T2, T1])
            pair.g.route_table_set_target(ghl, [ids[3], ids[10]], [T2, T1])
        if step == 40:
            before = pair.g.read_state()
            for hl, sel, tg in refusals:
                with pytest.raises(R.CrowdsimError):
                    pair.g.route_table_set_target(hl, sel, tg)
            _same(before, pair.g.read_state(), STATE)
        pair.oracle_step()
        pair.g.step(R.Duration(*DT))
        st = pair.check(True)
    moved = np.hypot(st["vx"], st["vy"]) != 0.0
    assert moved[:8].all() and moved[10] and not moved[11]


# ---- 6. refusals ------------------------------------------------------------------------------------------------
def _table(sim, legs):
    t = np.ascontiguousarray([p for p, _ in legs], dtype=np.float64).reshape(-1)
    n = np.ascontiguousarray([len(r) for _, r in legs], dtype=np.uint64)
    xy = np.ascontiguousarray([q for _, r in legs for q in r] or [0.0], dtype=np.float64).reshape(-1)
    out = C.c_uint32(0xFFFFFFFF)
    rc = sim._lib.rcs_hl_route_table(sim._h, len(legs), t.ctypes.data_as(N.c_f64p), n.ctypes.data_as(N.c_u64p),
                                     xy.ctypes.data_as(N.c_f64p), C.byref(out))
    return rc, out.value


def test_refusals_change_nothing():
    g = R.Simulation(R.LocationHash2D(64.0, 64.0, 2.0, (0.0, 0.0), capacity=512))
    lp = R.NoLocalPlan()
    keep = R.RouteTablePlan({(20.0, 20.0): [(10.0, 12.0), (20.0, 20.0)]})
    g.add_source_sink(R.SourceSink((5.0, 5.0), 0.5, R.MonotonicCrowd(10.0), keep, lp, [(20.0, 20.0)], False, 1.0))
    for _ in range(20):
        g.step(R.Duration(*DT))
    before = g.read_state()
    rc, first = _table(g, [((1.0, 1.0), [(1.0, 1.0)])])
    assert rc == N.RCS_OK
    bad = [[],                                                             # no legs
           [((1.0, 1.0), [(1.0, 1.0)]), ((2.0, 2.0), [])],                 # a leg without points
           [((1.0, 1.0), [(1.0, 1.0)]), ((1.0, 1.0), [(3.0, 3.0)])],       # equal targets
           [((0.0, 1.0), [(1.0, 1.0)]), ((-0.0, 1.0), [(3.0, 3.0)])],      # equal under IEEE ==
           [((1.0, 1.0), [(1.0, 1.0)] * 40000), ((2.0, 2.0), [(2.0, 2.0)] * 25535)]]  # 65535 points
    for legs in bad:
        rc, out = _table(g, legs)
        assert rc == N.RCS_ERR_ARG and out == 0xFFFFFFFF
    rc, nxt = _table(g, [((1.0, 1.0), [(1.0, 1.0)] * 40000), ((2.0, 2.0), [(2.0, 2.0)] * 25534)])  # 65534: accepted
    assert rc == N.RCS_OK and nxt == first + 1
    W = (30.0, 30.0)
    table = R.RouteTablePlan({W: [W], (40.0, 30.0): [(40.0, 30.0)]})
    for wps in ([W, (40.0, 31.0)], [(float("nan"), 30.0)], [(40.0, 30.0), W, (30.0, 30.5)]):
        with pytest.raises(R.CrowdsimError, match="has no leg"):
            g.add_source_sink(R.SourceSink((8.0, 40.0), 0.5, R.MonotonicCrowd(10.0), table, lp, wps, False, 1.0))
    _same(before, g.read_state(), STATE)
    assert g.add_source_sink(R.SourceSink((8.0, 40.0), 0.5, R.MonotonicCrowd(10.0), table, lp,
                                          [(40.0, 30.0), W], False, 1.0)) == 1
    # the refused calls added no source sink: the next step spawns for ids 0 and 1 only
    g.step(R.Duration(*DT))
    assert g.agent_count() == len(before["id"]) + 2
    # the route follower's refusal: study mode refuses handles with a route-table planner
    h = R.Simulation(R.LocationHash2D(64.0, 64.0, 2.0, (0.0, 0.0), capacity=64))
    h.add_agents([(3.0, 3.0)], R.RouteTablePlan({(9.0, 9.0): [(9.0, 9.0)]}), lp, 1.0)
    with pytest.raises(R.CrowdsimError, match="without strips, source sinks or route followers"):
        h.step_in_loop(R.Duration(*DT))
