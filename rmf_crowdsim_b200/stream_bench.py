"""bench.py --workload c5: the SourceSink spawn / despawn stream (BASELINE.json config 5; SURVEY.md 8d C5).

8192 source sinks on a 32 x 256 lattice inside a 4224 m square hash domain (cell 2 m).  Every source spawns with
MonotonicCrowd(10/s) at dt = 0.1 s (round(dt * rate) = 1 per step, and only while nobody stands within 0.4 m of the
source, lib.rs:208-217), its agents follow a three-segment route of ~125.6 m at unit speed through the device-side
route follower (the per-step half of RMFPlanner, rmf/mod.rs:197-215; routes are supplied as polylines because route
planning is host-side `mapf`) and are removed at the sink.  Steady state: ~2.5 M live agents, ~2048 spawns and
despawns per step, all handled on the device (spawn kernel, keep flags dropped by the next counting sort).
Steps are COMMITTED: this crowd stays finite (agents of one source walk in single file, lanes are 16 m apart).
"""
from __future__ import annotations

import ctypes as C
import json
import time

import numpy as np


def build(lp_none: bool, device: int = 0, cols: int = 32, rows: int = 256, strip=None, generator=None):
    """strip = (rank, world, nccl_id[, peer_gather]): this rank of a strip-partitioned stream.  Every rank holds all source sinks;
    the rank that owns a source's cell column spawns for it (source columns are 65 c + 17 of 2112: never next to a
    boundary of 2, 4 or 8 equal strips).  generator: the CrowdGenerator of every source (None: MonotonicCrowd(10/s))."""
    from . import sim as S

    margin, cell = 32.0, 2.0
    pitch_x, pitch_y = 130.0, 16.25
    dom = float(np.ceil((cols * pitch_x + 2 * margin) / cell) * cell)
    n_src = cols * rows
    cap = int(n_src * 330 * 1.1)  # ~314 agents per source in steady state
    if strip is None:
        idx = S.LocationHash2D(dom, dom, cell, (-margin, -margin), capacity=cap, device=device)
        sim = S.Simulation(idx)
    else:
        from .strips import StripSimulation

        rank, world, nccl_id = strip[:3]
        gather = strip[3] if len(strip) > 3 else None
        halo_cap = int(3 * rows * 2.5 * 1.5) + 4096  # three columns per side, ~2 agents per lane and column
        cap = int(cap / world * 1.3) + 2 * halo_cap + 8192
        idx = S.LocationHash2D(dom, dom, cell, (-margin, -margin), capacity=cap, device=device)
        sim = StripSimulation(idx, rank, world, nccl_id, halo_capacity=halo_cap, peer_gather=gather)
    lp = S.NoLocalPlan() if lp_none else S.Zanlungo(0.05, 1.0, 0.0, 0.5, 1.0, 0.2)
    keep = [lp]
    for c in range(cols):
        for r in range(rows):
            x0, y0 = c * pitch_x + 2.0, r * pitch_y + 8.0
            route = [(x0 + 40.03, y0 + 3.0), (x0 + 80.07, y0 - 3.0), (x0 + 125.01, y0)]
            hl = S.RouteFollowPlan(route)
            keep.append(hl)
            gen = S.MonotonicCrowd(10.0) if generator is None else generator
            sim.add_source_sink(S.SourceSink((x0, y0), 0.6, gen, hl, lp, [route[-1]], False, 2.0))
    sim._keep = keep
    return sim, n_src, dom


def measure(lp_none: bool, K: int, W: int, peaks: dict) -> dict:
    """Short form for bench.py's `secondary` table: fill the building, W warm-up steps, K timed committed steps."""
    from . import _native as N
    from .sim import Duration
    from bench import ALGO_BYTES_NOLOCALPLAN, ALGO_BYTES_ZANLUNGO

    sim, n_src, dom = build(lp_none)
    lib, h = sim._lib, sim._h
    dt = Duration(0, 100_000_000)

    def steps(k):
        for _ in range(k):
            N.check(h, lib.rcs_step_async(h, dt.secs, dt.nanos, N.RCS_STEP_DEFAULT))

    done = 0
    while done < 1400:  # one route takes ~1256 steps; events are drained so the buffers never overflow
        steps(100)
        sim.sync()
        sim._dispatch_events()
        done += 100
    steps(W)
    sim.sync()
    sim._dispatch_events()
    n_before = sim.agent_count()
    steps(4)  # after the sync: new counts, new buffer roles -- the steps are captured as a graph again
    launches0 = sim.launch_count()
    sim.event_record(0)
    steps(K)
    sim.event_record(1)
    sim.sync()
    total_ms = sim.event_elapsed_ms(0, 1)
    launches = sim.launch_count() - launches0
    st = sim.stats()
    n_after = sim.agent_count()
    sim._dispatch_events()
    N.check(h, lib.rcs_kernel_timing(h, 1))  # the dominant kernel, second short pass (kernel by kernel)
    steps(min(K, 8))
    sim.sync()
    kt_ms, kt_n = C.c_double(), C.c_uint64()
    N.check(h, lib.rcs_kernel_time_ms(h, C.byref(kt_ms), C.byref(kt_n)))
    N.check(h, lib.rcs_kernel_timing(h, 0))
    sim._dispatch_events()
    n_mean = 0.5 * (n_before + n_after)
    k_ms = kt_ms.value / max(kt_n.value, 1)
    algo = ALGO_BYTES_NOLOCALPLAN if lp_none else ALGO_BYTES_ZANLUNGO
    sim.spatial_index.close()
    return {"workload": f"C5: SourceSink stream, {n_src} sources, device-side route follower, "
                        f"{'NoLocalPlan' if lp_none else 'Zanlungo'}",
            "agents": n_after, "mode": "committed steps (spawn + despawn every step)",
            "value": n_mean * K / (total_ms * 1e-3), "ms_per_step": total_ms / K, "kernel_ms": k_ms,
            "frac": algo * n_mean / (k_ms * 1e-3) / 1e9 / peaks["hbm_gbs"] if k_ms > 0 else None,
            "frac_whole_step": algo * n_mean * K / (total_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
            "nonfinite": int(st.nonfinite_count), "launches_per_step": launches / K, "steps": K}


def run(args) -> None:
    from . import _native as N
    from .sim import Duration
    from bench import ALGO_BYTES_NOLOCALPLAN, ALGO_BYTES_ZANLUNGO, ClockSampler, measured_peaks

    lp_none = not args.c5_zanlungo
    sim, n_src, dom = build(lp_none)
    lib, h = sim._lib, sim._h
    dt = Duration(0, 100_000_000)

    def steps(k):
        for _ in range(k):
            N.check(h, lib.rcs_step_async(h, dt.secs, dt.nanos, N.RCS_STEP_DEFAULT))

    # fill the building: one route takes ~1256 steps; events are drained so the buffers never overflow
    t0 = time.time()
    done = 0
    while done < 1400:
        steps(100)
        sim.sync()
        sim._dispatch_events()
        done += 100
    fill_s = time.time() - t0
    clocks = ClockSampler(0)
    clocks.start()
    for _ in range(max(args.warmup, 3)):
        steps(1)
    sim.sync()
    sim._dispatch_events()
    n_before = sim.agent_count()
    launches0 = sim.launch_count()
    N.check(h, lib.rcs_kernel_timing(h, 1))
    K = args.steps
    sim.sync()
    wall0 = time.perf_counter()
    sim.event_record(0)
    steps(K)
    sim.event_record(1)
    sim.sync()
    wall1 = time.perf_counter()
    total_ms = sim.event_elapsed_ms(0, 1)
    kt_ms, kt_n = C.c_double(), C.c_uint64()
    N.check(h, lib.rcs_kernel_time_ms(h, C.byref(kt_ms), C.byref(kt_n)))
    N.check(h, lib.rcs_kernel_timing(h, 0))
    launches = sim.launch_count() - launches0
    st = sim.stats()
    n_after = sim.agent_count()
    ns, nd = C.c_uint64(), C.c_uint64()
    N.check(h, lib.rcs_poll_events(h, 0, None, None, C.byref(ns), 0, None, C.byref(nd)))  # counts of the timed steps
    sim._dispatch_events()
    clk = clocks.stop()
    n_mean = 0.5 * (n_before + n_after)
    value = n_mean * K / (total_ms * 1e-3)

    # end to end: every step the host drains the spawn / destroy events and reads the positions (pinned)
    e2e = None
    if not args.skip_e2e:
        cap = sim.spatial_index.capacity
        bufs, ptrs = [], []
        for _ in range(2):
            p = C.c_void_p()
            N.check(None, lib.rcs_host_alloc(cap * 8, C.byref(p)))
            ptrs.append(p)
            bufs.append(C.cast(p, N.c_f64p))
        out_n = C.c_uint64()
        moved = 0
        ke = min(K, 10)
        t0 = time.perf_counter()
        for _ in range(ke):
            sim.step(dt)  # rcs_step + rcs_poll_events -> EventListener callbacks (none registered)
            N.check(h, lib.rcs_read_agents(h, N.RCS_ORDER_STORAGE, cap, None, bufs[0], bufs[1], None, None, None,
                                           C.byref(out_n)))
            moved += out_n.value
        t1 = time.perf_counter()
        for p in ptrs:
            lib.rcs_host_free(p)
        e2e = {"value": moved / (t1 - t0), "unit": "agent-steps/s", "h2d_bytes_per_step": 0,
               "d2h_bytes_per_step": int(16 * moved / ke) + 24 * 2 * 2048, "steps": ke,
               "path": "Simulation.step (rcs_step + rcs_poll_events) + rcs_read_agents(x, y -> pinned host); the "
                       "stream's inputs (source sinks, routes) are resident, the per-step host traffic is events + positions"}

    peaks, how = measured_peaks()
    algo = ALGO_BYTES_NOLOCALPLAN if lp_none else ALGO_BYTES_ZANLUNGO
    k_ms = kt_ms.value / max(kt_n.value, 1)
    achieved = algo * n_mean / (k_ms * 1e-3) / 1e9 if k_ms > 0 else None
    line = {
        "metric": "agent-steps/sec (query+Zanlungo+integrate)", "value": value, "unit": "agent-steps/s", "n_gpus": 1,
        "steps": K, "warmup": args.warmup, "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {
            "workload": f"C5: SourceSink stream, {n_src} sources (MonotonicCrowd 10/s, dt 0.1 s), device-side route "
                        f"follower on 3-segment routes, {'NoLocalPlan' if lp_none else 'Zanlungo'}, committed steps",
            "agents_live": n_after, "domain_m": dom, "spawned_in_timed_steps": int(ns.value),
            "destroyed_in_timed_steps": int(nd.value), "fill_steps": 1400, "fill_wall_s": fill_s,
            "l2": "inputs larger than L2", "mean_neighbours": st.neighbour_total / max(n_after, 1),
            "nonfinite": int(st.nonfinite_count), "oob": int(st.oob_count),
        },
        "e2e": e2e, "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "step_warp_kernel + step_aside_kernel", "achieved": achieved,
                     "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": (achieved / peaks["hbm_gbs"]) if achieved else None,
                     "peak_source": how, "traffic": None, "algorithmic_bytes_per_agent_step": algo, "kernel_ms": k_ms,
                     "kernel_share_of_step": k_ms * K / total_ms},
        "cpu_baseline": None, "clocks": clk, "wall_s_timed_region": wall1 - wall0,
    }
    print(json.dumps(line), flush=True)
