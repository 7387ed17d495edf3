"""Route-table planner on the C5 geometry (rmf_crowdsim_b200/stream_bench.py): each source's three-segment route becomes
three waypoints with one leg per waypoint, so the source sinks go through every waypoint as RMF scenes do
(set_target at the spawn and at each advance).  Times committed steps of

  (a) the route-table planner on the device (RouteTablePlan),
  (b) the same scene with a host-evaluated Python planner of identical semantics (read back, one Python call per agent,
      upload, every step), and
  (c) the single-leg C5 scene (RouteFollowPlan, one waypoint: bench.py's C5 line),

and prints one JSON line with the card's name and power limit.  (a) and (c) run on the full C5 lattice (8192 sources,
~2.5 M agents after the fill); the host planner cannot fill that in useful time, so (b) runs on a small lattice and is
compared with (a) on the same small lattice.  Usage: python tools/route_table_bench.py [--steps K] [--small-steps k]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rmf_crowdsim_b200 import _native as N  # noqa: E402
from rmf_crowdsim_b200 import sim as S  # noqa: E402
from rmf_crowdsim_b200 import stream_bench  # noqa: E402

DT = S.Duration(0, 100_000_000)


class HostRouteTable(S.HighLevelPlanner):
    """RouteTablePlan's semantics evaluated in Python (the host path)."""

    def __init__(self, routes):
        self.routes = {tuple(t): [tuple(p) for p in r] for t, r in routes.items()}
        self.cache = {}

    def set_target(self, agent, point, tolerance):
        self.cache[agent.agent_id] = [self.routes[(float(point[0]), float(point[1]))], 0]

    def remove_agent_id(self, agent):
        self.cache.pop(agent, None)

    def get_desired_velocity(self, agent, time):
        e = self.cache.get(agent.agent_id)
        if e is None:
            return None
        leg, k = e
        px, py = agent.position
        dx, dy = px - leg[k][0], py - leg[k][1]
        if math.sqrt(dx * dx + dy * dy) < 1e-1 and len(leg) > k + 1:
            k += 1
            e[1] = k
        dx, dy = leg[k][0] - px, leg[k][1] - py
        n = math.sqrt(dx * dx + dy * dy)
        return (dx / n, dy / n)


def build_table(cols, rows, host=False):
    """stream_bench.build's lattice with three waypoints per source and one single-point leg per waypoint."""
    margin, cell = 32.0, 2.0
    pitch_x, pitch_y = 130.0, 16.25
    dom = float(math.ceil((cols * pitch_x + 2 * margin) / cell) * cell)
    cap = int(cols * rows * 330 * 1.1)
    sim = S.Simulation(S.LocationHash2D(dom, dom, cell, (-margin, -margin), capacity=cap))
    lp = S.NoLocalPlan()
    keep = [lp]
    for c in range(cols):
        for r in range(rows):
            x0, y0 = c * pitch_x + 2.0, r * pitch_y + 8.0
            route = [(x0 + 40.03, y0 + 3.0), (x0 + 80.07, y0 - 3.0), (x0 + 125.01, y0)]
            legs = {p: [p] for p in route}
            hl = HostRouteTable(legs) if host else S.RouteTablePlan(legs)
            keep.append(hl)
            sim.add_source_sink(S.SourceSink((x0, y0), 0.6, S.MonotonicCrowd(10.0), hl, lp, route, False, 2.0))
    sim._keep = keep
    return sim


def fill(sim, n, device_only=True):
    done = 0
    while done < n:
        k = min(100, n - done)
        if device_only:
            for _ in range(k):
                N.check(sim._h, sim._lib.rcs_step_async(sim._h, DT.secs, DT.nanos, N.RCS_STEP_DEFAULT))
            sim.sync()
            sim._dispatch_events()
        else:
            for _ in range(k):
                sim.step(DT)
        done += k


def time_device(sim, K):
    """K committed asynchronous steps between two device events (as bench.py's C5 line)."""
    fill(sim, 1400)
    for _ in range(4):
        N.check(sim._h, sim._lib.rcs_step_async(sim._h, DT.secs, DT.nanos, N.RCS_STEP_DEFAULT))
    sim.sync()
    sim._dispatch_events()
    n0 = sim.agent_count()
    sim.event_record(0)
    for _ in range(K):
        N.check(sim._h, sim._lib.rcs_step_async(sim._h, DT.secs, DT.nanos, N.RCS_STEP_DEFAULT))
    sim.event_record(1)
    sim.sync()
    ms = sim.event_elapsed_ms(0, 1)
    n1 = sim.agent_count()
    sim._dispatch_events()
    return {"ms_per_step": ms / K, "agents": n1, "agent_steps_per_s": 0.5 * (n0 + n1) * K / (ms * 1e-3), "steps": K}


def time_stepped(sim, K, fill_steps):
    """Simulation.step (step + events + host planners) K times, wall clock: the path a host planner needs."""
    fill(sim, fill_steps, device_only=False)
    n0 = sim.agent_count()
    t0 = time.perf_counter()
    for _ in range(K):
        sim.step(DT)
    wall = time.perf_counter() - t0
    n1 = sim.agent_count()
    return {"ms_per_step": wall * 1e3 / K, "agents": n1, "agent_steps_per_s": 0.5 * (n0 + n1) * K / wall, "steps": K}


def card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:  # the number is still reported, without its power limit
        pl = f"unknown ({exc})"
    return name, pl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--small-steps", type=int, default=20)
    ap.add_argument("--small", default="2x16", help="cols x rows of the lattice for (b) and its (a) counterpart")
    args = ap.parse_args()
    cols, rows = (int(v) for v in args.small.split("x"))
    name, pl = card()
    out = {"gpu": name, "power_limit": pl, "dt_s": DT.as_secs_f64(), "local_planner": "NoLocalPlan"}
    sim = build_table(32, 256)
    out["a_route_table_device"] = time_device(sim, args.steps)
    sim.spatial_index.close()
    sim, _, _ = stream_bench.build(True)
    out["c_single_leg_c5"] = time_device(sim, args.steps)
    sim.spatial_index.close()
    small_fill = 400
    sim = build_table(cols, rows)
    out["a_route_table_device_small"] = dict(time_stepped(sim, args.small_steps, small_fill), lattice=args.small)
    sim.spatial_index.close()
    sim = build_table(cols, rows, host=True)
    out["b_host_planner_small"] = dict(time_stepped(sim, args.small_steps, small_fill), lattice=args.small)
    sim.spatial_index.close()
    out["a_over_c_ms"] = out["a_route_table_device"]["ms_per_step"] / out["c_single_leg_c5"]["ms_per_step"]
    out["b_over_a_small_ms"] = out["b_host_planner_small"]["ms_per_step"] / out["a_route_table_device_small"]["ms_per_step"]
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
