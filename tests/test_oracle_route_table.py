"""CPU: the oracle's RouteTablePlan (tests/oracle_route_table.cpp) on a hand-checkable scene -- axis-aligned legs at
unit speed and dt = 0.5 s, so that every position is exact -- and a one-leg table against the oracle's RouteFollowPlan."""
import numpy as np
import pytest

import oracle_ffi as O
import oracle_route_table as RT

DT = (0, 500_000_000)
W0, W1, W2 = (8.0, 6.0), (8.0, 8.0), (6.0, 8.0)
# the leg to W0 turns at (7, 6); the leg to W2 runs on past it to (2, 8)
ROUTES = {W0: [(7.0, 6.0), W0], W1: [(8.0, 7.0), W1], W2: [W2, (2.0, 8.0)]}
# agent 0 after steps 1..11 (spawned at (6, 6) in step 1): the sink test (radius 0.6, on the old position) advances
# it in steps 4 and 8, each time 0.5 m before the leg's last point, i.e. while the follower still heads for it
PATH = [((6.5, 6.0), 0), ((7.0, 6.0), 0), ((7.5, 6.0), 0), ((8.0, 6.0), 1), ((8.0, 6.5), 1), ((8.0, 7.0), 1),
        ((8.0, 7.5), 1), ((8.0, 8.0), 2), ((7.5, 8.0), 2), ((7.0, 8.0), 2), ((6.5, 8.0), 2)]


def _scene(loop):
    o = RT.RouteTableOracle(20.0, 20.0, 1.0, (0.0, 0.0))
    hl = o.hl_route_table(ROUTES)
    o.add_source_sink((6.0, 6.0), 0.6, 2.0, hl, o.lp_none(), [W0, W1, W2], loop, 1.0)
    return o


def _agent0(o):
    st = o.read_state()
    k = int(np.searchsorted(st["id"], 0))
    if k == len(st["id"]) or st["id"][k] != 0:
        return None
    return (float(st["x"][k]), float(st["y"][k])), int(st["next_waypoint"][k]), (float(st["vx"][k]),
                                                                                 float(st["vy"][k]))


@pytest.mark.parametrize("loop", [False, True])
def test_route_table_through_three_waypoints(loop):
    o = _scene(loop)
    for pos, wp in PATH:
        o.step(*DT)
        assert _agent0(o)[:2] == (pos, wp)
    o.step(*DT)  # step 12: the old position (6.5, 8) is within 0.6 of the sink W2
    if not loop:
        assert _agent0(o) is None
        assert 0 in o.poll_events()[2].tolist()
        return
    # loop_forever: next_waypoint wraps to 0 WITHOUT set_target, so the agent keeps the leg to W2 and walks on to (2, 8)
    assert _agent0(o)[:2] == ((6.0, 8.0), 0)
    for x in (5.5, 5.0, 4.5):
        o.step(*DT)
        assert _agent0(o) == ((x, 8.0), 0, (-1.0, 0.0))


def test_every_agent_walks_the_same_path():
    """One spawn per step (MonotonicCrowd 2/s at dt 0.5 s; the previous agent is 0.5 m away): agent k is agent 0
    delayed by k steps."""
    o = _scene(False)
    hist = []
    for _ in range(11):
        o.step(*DT)
        st = o.read_state()
        hist.append({int(a): ((float(x), float(y)), int(w)) for a, x, y, w in
                     zip(st["id"], st["x"], st["y"], st["next_waypoint"])})
    for step, h in enumerate(hist):
        for a, v in h.items():
            assert v == PATH[step - a]


def test_set_target_selects_the_leg_by_point():
    o = RT.RouteTableOracle(20.0, 20.0, 1.0, (0.0, 0.0))
    hl = o.hl_route_table(ROUTES)
    ids = o.add_agents([(6.0, 6.0), (6.0, 9.0), (2.0, 2.0)], hl, o.lp_none(), 1.0)
    o.hl_route_table_set_target(hl, ids[:2], [W1, W2])
    with pytest.raises(O.OracleError, match="no route to this point"):
        o.hl_route_table_set_target(hl, ids[2:], [(8.0, 8.5)])
    with pytest.raises(O.OracleError, match="no route to this point"):
        o.hl_route_table_set_target(hl, ids[2:], [(float("nan"), 8.0)])
    o.step(*DT)
    st = o.read_state()
    # agent 0 heads for (8, 7) (leg of W1), agent 1 for W2 = (6, 8) itself, agent 2 is in no cache: None -> (0, 0)
    assert np.hypot(st["vx"][0] - 2.0 / 5 ** 0.5, st["vy"][0] - 1.0 / 5 ** 0.5) < 1e-15
    assert (st["vx"][1], st["vy"][1]) == (0.0, -1.0) and (st["vx"][2], st["vy"][2]) == (0.0, 0.0)


def test_one_leg_table_equals_route_follow_plan():
    route = [(5.0, 5.3), (9.0, 5.1)] + [(10.0 + 0.6 * j, 5.0 + 0.1 * (-1) ** j) for j in range(12)] + [(19.0, 6.0)]
    sims = []
    for kind in ("route", "table"):
        o = RT.RouteTableOracle(24.0, 24.0, 1.0, (0.0, 0.0))
        hl = o.hl_route(route) if kind == "route" else o.hl_route_table({(19.0, 6.0): route})
        lp = o.lp_zanlungo(0.05, 1.0, 0.0, 0.5, 1.0, 0.2)
        o.add_source_sink((2.0, 5.0), 0.6, 10.0, hl, lp, [(19.0, 6.0)], False, 2.0)
        sims.append(o)
    for _ in range(250):
        for o in sims:
            o.step(0, 100_000_000)
        a, b = (o.read_state() for o in sims)
        for k in a:
            assert np.array_equal(a[k].view(np.uint64), b[k].view(np.uint64)), k
    assert sims[0].agent_count() > 20
