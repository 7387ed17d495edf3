"""PoissonCrowd on the C5 geometry (rmf_crowdsim_b200/stream_bench.py): 8192 source sinks, device-side route
followers, NoLocalPlan.  Times committed asynchronous steps of

  (m) the C5 building with MonotonicCrowd(10/s) (bench.py --workload c5),
  (p) the same building with PoissonCrowd(10/s) (lambda = 1 at dt = 0.1 s: a source wants to spawn in ~63 % of the
      steps, so the live count is lower than (m)'s), and
  (a) (p) with dt alternating between 0.1 s and 0.09 s every step: the per-source thresholds are recomputed and
      uploaded every step, without a stream synchronisation,

in alternating rounds after a fill of 1400 steps each, and prints one JSON line with ms/step, agent-steps/s, live agents
and spawns per step of each, and the card's name and power limit.
Usage: python tools/poisson_stream_bench.py [--steps K] [--rounds R]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rmf_crowdsim_b200 import _native as N  # noqa: E402
from rmf_crowdsim_b200 import sim as S  # noqa: E402
from rmf_crowdsim_b200 import stream_bench  # noqa: E402

DT = S.Duration(0, 100_000_000)
DT_ALT = S.Duration(0, 90_000_000)


def steps(sim, dts):
    for dt in dts:
        N.check(sim._h, sim._lib.rcs_step_async(sim._h, dt.secs, dt.nanos, N.RCS_STEP_DEFAULT))


def fill(sim, n=1400):
    for _ in range(n // 100):  # one route takes ~1256 steps; events are drained so the buffers never overflow
        steps(sim, [DT] * 100)
        sim.sync()
        sim._dispatch_events()


def timed(sim, dts):
    """len(dts) committed steps between two device events, after 4 untimed steps (new counts after the sync: the
    steps are captured as graphs again)."""
    steps(sim, dts[:4])
    sim.sync()
    sim._dispatch_events()
    n0 = sim.agent_count()
    sim.event_record(0)
    steps(sim, dts)
    sim.event_record(1)
    sim.sync()
    ms = sim.event_elapsed_ms(0, 1)
    n1 = sim.agent_count()
    ns, nd = C.c_uint64(), C.c_uint64()
    N.check(sim._h, sim._lib.rcs_poll_events(sim._h, 0, None, None, C.byref(ns), 0, None, C.byref(nd)))
    sim._dispatch_events()
    k = len(dts)
    return {"ms_per_step": ms / k, "agent_steps_per_s": 0.5 * (n0 + n1) * k / (ms * 1e-3), "agents": n1,
            "spawns_per_step": ns.value / k, "despawns_per_step": nd.value / k}


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
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    name, pl = card()
    runs = {"monotonic": (S.MonotonicCrowd(10.0), [DT] * args.steps),
            "poisson": (S.PoissonCrowd(10.0, seed=1), [DT] * args.steps),
            "poisson_dt_alternating": (S.PoissonCrowd(10.0, seed=1),
                                       [DT if k % 2 == 0 else DT_ALT for k in range(args.steps)])}
    sims = {}
    for key, (gen, _) in runs.items():
        sims[key], n_src, _ = stream_bench.build(True, generator=gen)
        fill(sims[key])
    res = {key: [] for key in runs}
    for _ in range(args.rounds):
        for key, (_, dts) in runs.items():
            res[key].append(timed(sims[key], dts))
    out = {"gpu": name, "power_limit": pl, "sources": n_src, "local_planner": "NoLocalPlan", "steps": args.steps,
           "rounds": args.rounds, "dt_s": [DT.as_secs_f64(), DT_ALT.as_secs_f64()]}
    for key, rs in res.items():
        ms = [r["ms_per_step"] for r in rs]
        out[key] = {"ms_per_step_median": statistics.median(ms), "ms_per_step_min": min(ms), "ms_per_step_max": max(ms),
                    "agent_steps_per_s_median": statistics.median(r["agent_steps_per_s"] for r in rs),
                    "agents": rs[-1]["agents"],
                    "spawns_per_step": statistics.mean(r["spawns_per_step"] for r in rs),
                    "despawns_per_step": statistics.mean(r["despawns_per_step"] for r in rs),
                    "graph_launches": sims[key].graph_stats()[0]}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
