#!/usr/bin/env python
"""bench.py -- agent-steps/sec of the per-timestep agent update (query + Zanlungo + integrate).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload c3|c4|c2] [--variant ...]
                    [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" is one pass of the whole hot path (LocationHash2D rebuild,
radius query, Zanlungo force, Euler integration) over the synthetic crowd.

Workloads (SURVEY.md section 8d; BASELINE.json configs):
  default, every N : C4 -- 2^24 agents, 4096 m x 4096 m, density 1/m^2 (jittered lattice), Zanlungo, shuffled
                     ids, bidirectional +-x flow by id parity.  N > 1: spatial strips over the N GPUs with
                     an NCCL halo exchange (strong scaling: the crowd is the same for every N).
  --workload c3    : 2^20 agents (single-GPU roofline study), --workload c2: 10^4 agents.
The shuffled crowd is timed in frozen-snapshot mode (RCS_STEP_NO_COMMIT): the reference model itself drives
a dense mixed bidirectional crowd non-finite within 3-23 steps (SURVEY.md section 0.4), so every timed step
runs the full pipeline on the same physical snapshot and discards the result.  `--variant lane` times the
lane-ordered crowd with committed steps instead (force pass idle).

--dump-outputs DIR (one GPU): after the timed steps, the agent state the last timed step produced -- ids, x, y, vx, vy
in ascending id order, what rcs_read_agents returns to a caller -- goes to DIR/<name>.npy as float64, a fixed
seeded sample of DUMP_MAX_AGENTS agents for larger crowds.  The inputs are the same in every run with the same
arguments, so two builds can be compared array for array.

The reference arm (--impl reference) and the cpu_baseline leg time the CPU oracle in its literal
data-structure form (hash maps, in-loop index update, map iteration order), single-threaded like the
reference, on a bounded sub-crowd of the same density and planner.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from untouched (it may be read-only)

ALGO_BYTES_ZANLUNGO = 88  # SURVEY.md 8(d): read x,y,vx,vy,pvx,pvy + id, write x,y,vx,vy
ALGO_BYTES_NOLOCALPLAN = 64
L2_FLUSH_BYTES = 512 << 20
DUMP_MAX_AGENTS = 1 << 20  # --dump-outputs: five float64 arrays of at most 2^20 agents, 40 MiB
DUMP_SEED = 0


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the GPU is under load."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.lines: list[str] = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax.append(float(f[1]))
                power.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def make_scene(workload: str, variant: str, lp_none: bool = False):
    from rmf_crowdsim_b200 import scenes as SC

    lp = ("none",) if lp_none else None
    if workload == "c2":
        sc = SC.config_c2(variant)
        if lp_none:
            sc.lp = ("none",)
        return sc
    if workload == "c3":
        return SC.config_c3(variant, lp=lp)
    if workload == "c4":
        sc = SC.config_c4(variant)
        if lp_none:
            sc.lp = ("none",)
        return sc
    if workload.startswith("side"):  # sideN[:cell]: N x N agents, optional hash cell size (default 2 m = eyesight)
        side, _, cell = workload[4:].partition(":")
        return SC.uniform_crowd(int(side), variant, margin=64.0, lp=lp, cell=float(cell) if cell else 2.0)
    raise SystemExit(f"unknown workload {workload}")


# --------------------------------------------------------------------------------------------------
# CPU oracle legs (cpu_baseline and --impl reference).  The only places bench.py executes oracle/.
# --------------------------------------------------------------------------------------------------
def oracle_run(scene, steps: int, warmup: int):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_ffi as O

    o = O.OracleSim(scene.width, scene.height, scene.cell, scene.offset, index_mode=O.IN_LOOP,
                    iter_order=O.MAP_ORDER, canonical=False)
    hl = o.hl_parity(scene.hl[1])
    lp = o.lp_none() if scene.lp[0] == "none" else o.lp_zanlungo(*scene.lp[1:])
    ids = o.add_agents(scene.xy, hl, lp, scene.eyesight)

    def inject():
        o.set_state(ids, scene.xy[:, 0], scene.xy[:, 1], scene.vxy[:, 0], scene.vxy[:, 1])

    total = 0.0
    for k in range(warmup + steps):
        inject()  # frozen snapshot: every step sees the same crowd (not timed)
        t0 = time.perf_counter()
        o.step(*scene.dt)
        t1 = time.perf_counter()
        if k >= warmup:
            total += t1 - t0
    return scene.n * steps / total, total


def flat_port_run(variant: str, steps: int = 12):
    """oracle/flat_parallel.cpp on all host cores: NOT the reference (which is single-threaded and HashMap-based) but a
    strong multi-threaded CPU implementation of the same deferred step (flat arrays, counting-sort grid, the oracle's
    Zanlungo arithmetic, bit-identical results) -- reported so that the GPU number can also be read against the best
    the host could do.  Frozen snapshot of a 262,144-agent sub-crowd of the same density."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_ffi as O
    from rmf_crowdsim_b200 import scenes as SC

    scene = SC.uniform_crowd(512, variant, margin=64.0)
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cols = [np.ascontiguousarray(a) for a in (scene.xy[:, 0], scene.xy[:, 1], scene.vxy[:, 0], scene.vxy[:, 1])]
    total = 0.0
    for k in range(steps + 1):
        work = [c.copy() for c in cols]  # frozen snapshot: every step sees the same crowd (not timed)
        t0 = time.perf_counter()
        O.flat_step(scene, *work, scene.dt, threads)
        t1 = time.perf_counter()
        if k >= 1:
            total += t1 - t0
    return {"value": scene.n * steps / total, "unit": "agent-steps/s", "cores": threads,
            "kind": "flat-array multi-threaded port, NOT the reference (oracle/flat_parallel.cpp)",
            "sample": f"{scene.n}-agent sub-crowd (same density 1/m^2, R=2 m, Zanlungo params), frozen snapshot, "
                      f"{steps} steps"}


def cpu_sample_scene(workload: str, variant: str, budget_steps: int):
    """Bounded sample of the workload for the CPU legs: a sub-crowd of the same density, spacing and
    planner, sized for ~0.35 s/step on one host core of the GPU box at the default step counts (the literal data
    structures cost 3-4 us per agent-step there, ~20 us in the build container), i.e. 10-20 s of CPU work per run."""
    from rmf_crowdsim_b200 import scenes as SC

    side = 320 if budget_steps <= 40 else (224 if budget_steps <= 120 else 128)
    sc = SC.uniform_crowd(side, variant, margin=64.0)
    return sc, f"{side * side}-agent sub-crowd of {workload} (same density 1/m^2, R=2 m, Zanlungo params), frozen snapshot"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    workload = args.workload or "c4"
    scene, sample = cpu_sample_scene(workload, args.variant, args.steps + args.warmup)
    value, total = oracle_run(scene, args.steps, max(args.warmup, 1))
    cores = os.cpu_count()
    line = {
        "impl": "reference", "metric": "agent-steps/sec (query+Zanlungo+integrate)", "value": value,
        "unit": "agent-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(workload, args.variant), "sample": sample},
        "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": 1, "kind": "port", "sample": sample,
                         "host_cores_available": cores,
                         "note": "C++ restatement of the reference CPU path (the Rust reference cannot be built "
                                 "here: no rustc/cargo); single-threaded like the reference"},
        "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        # for context only (the line's value is the reference-style run above): the best this host does on the same step
        "cpu_parallel_port": flat_port_run(args.variant, 6),
    }
    print(json.dumps(line), flush=True)


def workload_name(workload: str, variant: str) -> str:
    names = {
        "c2": "C2: 10,000 agents, 100x100 m, density 1/m^2, Zanlungo",
        "c3": "C3: 2^20 agents, 1024x1024 m, density 1/m^2 (jittered lattice), Zanlungo, R=cell=2 m",
        "c4": "C4: 2^24 agents, 4096x4096 m bidirectional +-x flow by id parity, spatial strips",
    }
    return names.get(workload, workload) + f", ids {variant}"


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def run_gpu_single(args):
    import ctypes as C

    from rmf_crowdsim_b200 import Duration, _native as N
    from rmf_crowdsim_b200 import scenes as SC

    workload = args.workload or "c4"
    scene = make_scene(workload, args.variant, lp_none=args.no_local_plan)
    # committed steps only for the lane-ordered Zanlungo crowd (stays finite); everything else is timed on a
    # frozen snapshot so that agents cannot walk out of the hash domain during a long run
    frozen = not (args.variant == "lane" and not args.no_local_plan)
    dt = Duration(*scene.dt)
    sim = SC.build_simulation(scene, device=0)
    lib, h = sim._lib, sim._h
    if args.kernel:
        sim.set_option(N.RCS_OPT_STEP_KERNEL, args.kernel)
    n = scene.n
    state_bytes = n * 48 * 2
    flush = state_bytes < (1 << 30)

    clocks = ClockSampler(0)
    m = timed_steps(sim, n, dt, frozen, args.steps, max(args.warmup, 3), flush, heat_s=0.4, clocks=clocks,
                    keep_state=bool(args.dump_outputs) and not frozen)
    total_ms, K, kt_ms, kt_n, launches, st = m["total_ms"], args.steps, m["kt_ms"], m["kt_n"], m["launches"], m["stats"]
    wall0, wall1 = m["wall0"], m["wall1"]
    value = n * K / (total_ms * 1e-3)

    # end to end through the C ABI with HOST buffers: every step uploads the preferred velocities of a host
    # HighLevelPlanner (pinned), runs the step, and reads back x,y,vx,vy of every agent (pinned).
    e2e = None if args.skip_e2e else run_e2e(scene, frozen, min(K, 10), max(3, min(args.warmup, 5)))
    clk = clocks.stop()

    peaks, how = measured_peaks()
    algo = ALGO_BYTES_NOLOCALPLAN if args.no_local_plan else ALGO_BYTES_ZANLUNGO
    k_ms = kt_ms / max(kt_n, 1)
    achieved = algo * n / (k_ms * 1e-3) / 1e9 if k_ms > 0 else None
    traffic = None
    counts0 = kernel_counts(f"{workload}_{args.variant}" + ("_nolp" if args.no_local_plan else ""))
    if counts0:
        traffic = counts0.get("kernel_dram_bytes")
    roofline = {
        "bound": "hbm", "kernel": "step_warp_kernel + step_aside_kernel (radius query + Zanlungo + Euler, fused)",
        "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
        "frac": (achieved / peaks["hbm_gbs"]) if achieved else None, "peak_source": how, "traffic": traffic,
        "algorithmic_bytes_per_agent_step": algo, "kernel_ms": k_ms, "kernel_share_of_step": k_ms * K / total_ms,
        "note": "the Zanlungo kernel is FP64-pipe-bound, not HBM-bound (SURVEY.md 8d); see fp64 keys",
    }
    fp64 = fp64_info(args)
    if fp64:
        roofline["fp64_peak_tflops_measured"] = fp64
        counts = kernel_counts(f"{workload}_{args.variant}" + ("_nolp" if args.no_local_plan else ""))
        if counts and k_ms > 0:
            # FP64 pipe: double-precision thread instructions per agent (ncu capture of this kernel on this workload,
            # profiles/kernel_counts.json) x agents / kernel time, against the measured DFMA issue rate
            peak_inst = fp64["dfma_tflops"] * 1e12 / 2.0
            dp = counts["dp_inst_per_agent"]
            roofline["fp64"] = {"dp_inst_per_agent": dp, "peak_dp_inst_per_s": peak_inst,
                                "achieved_dp_inst_per_s": dp * n / (k_ms * 1e-3),
                                "frac": dp * n / (k_ms * 1e-3) / peak_inst, "source": counts.get("source")}
            roofline["step_dram_bytes"] = counts.get("step_dram_bytes")
            roofline["step_algorithmic_bytes"] = algo * n

    if args.dump_outputs:
        state = m["state"]
        if frozen:
            # the timed steps discarded their result (RCS_STEP_NO_COMMIT) and left the snapshot as it was: one
            # committed step from that snapshot computes the same step and makes its result readable
            sim.step(dt)
            state = sim.read_state()
        dump_outputs(args.dump_outputs, state)
    sim.spatial_index.close()
    secondary = None if args.skip_secondary else secondary_lines(args, scene, peaks)
    sample_scene, sample = cpu_sample_scene(workload, args.variant, 6)
    if args.no_local_plan:
        sample_scene.lp = ("none",)
    cpu_v = None if args.skip_cpu else oracle_run(sample_scene, 30, 2)[0]  # ~10 s of CPU work on one core
    cpu_par = None if (args.skip_cpu or args.no_local_plan) else flat_port_run(args.variant)
    line = {
        "metric": "agent-steps/sec (query+Zanlungo+integrate)", "value": value, "unit": "agent-steps/s",
        "n_gpus": 1, "steps": K, "warmup": args.warmup, "ms_per_step": total_ms / K, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {
            "workload": workload_name(workload, args.variant) + (", NoLocalPlan" if args.no_local_plan else ""),
            "agents": n, "mode": "frozen snapshot (RCS_STEP_NO_COMMIT)" if frozen else "committed steps",
            "l2": "flushed between timed steps (512 MiB write)" if flush else "inputs larger than L2",
            "seed": scene.seed, "dt_ns": scene.dt[1],
            "mean_neighbours": st.neighbour_total / max(n, 1), "candidates_per_agent": st.candidate_total / max(n, 1),
            "finite_tti_fraction": st.finite_tti_count / max(n, 1), "nonfinite": int(st.nonfinite_count),
            "oob": int(st.oob_count),
        },
        "e2e": e2e, "gpu_launches": int(launches), "graph_steps_so_far": m["graph_steps"],
        "roofline": roofline, "cpu_parallel_port": cpu_par,
        "dist_verified": None, "secondary": secondary,
        "cpu_baseline": {"value": cpu_v, "unit": "agent-steps/s", "cores": 1, "kind": "port", "sample": sample,
                         "host_cores_available": os.cpu_count()},
        "clocks": clk, "wall_s_timed_region": wall1 - wall0,
    }
    print(json.dumps(line), flush=True)


def timed_steps(sim, n, dt, frozen, K, warmup, flush, heat_s=0.0, clocks=None, keep_state=False):
    """W untimed steps (+ optional extra load for the clock samples), then K steps, each bracketed by events on the
    launching stream with L2 flushed in between when the state is small.  Returns times and counters, and with
    keep_state the agent state right after the K steps."""
    import ctypes as C

    from rmf_crowdsim_b200 import _native as N

    lib, h = sim._lib, sim._h

    def one_step(commit=not frozen):
        N.check(h, lib.rcs_step_async(h, dt.secs, dt.nanos, N.RCS_STEP_DEFAULT if commit else N.RCS_STEP_NO_COMMIT))

    for _ in range(warmup):
        one_step()
    sim.sync()
    if clocks is not None:
        clocks.start()
    if heat_s > 0:  # keep stepping so that the clock samples are taken under load
        t_end = time.time() + heat_s
        heat = 0
        # The number of these steps depends on the clock: they never commit, so that the timed steps start from the
        # same state in every run.  An even number of them leaves the handle's buffers as the warm-up left them.
        while time.time() < t_end and heat < 600:
            for _ in range(8):
                one_step(commit=False)
            heat += 8
            sim.sync()
    launches0 = sim.launch_count()
    sim.sync()
    wall0 = time.perf_counter()
    total_ms = 0.0
    done = 0
    while done < K:
        batch = min(K - done, N.RCS_NUM_EVENTS // 2)
        for b in range(batch):
            if flush:
                sim.flush_l2(L2_FLUSH_BYTES)
            sim.event_record(2 * b)
            one_step()
            sim.event_record(2 * b + 1)
        sim.sync()
        for b in range(batch):
            total_ms += sim.event_elapsed_ms(2 * b, 2 * b + 1)
        done += batch
    wall1 = time.perf_counter()
    launches = sim.launch_count() - launches0 - (K if flush else 0)
    stats = sim.stats()
    state = sim.read_state() if keep_state else None  # before the kernel-timing steps below move the crowd on
    g0 = sim.graph_stats()
    # The dominant kernel, bracketed by its own event pair on the launching stream: a second short pass, because a
    # step with kernel timing on is launched kernel by kernel while the steps above replay as CUDA graphs.
    N.check(h, lib.rcs_kernel_timing(h, 1))
    for _ in range(min(K, 10)):
        if flush:
            sim.flush_l2(L2_FLUSH_BYTES)
        one_step()
    sim.sync()
    kt_ms, kt_n = C.c_double(), C.c_uint64()
    N.check(h, lib.rcs_kernel_time_ms(h, C.byref(kt_ms), C.byref(kt_n)))
    N.check(h, lib.rcs_kernel_timing(h, 0))
    return {"total_ms": total_ms, "kt_ms": kt_ms.value, "kt_n": kt_n.value, "launches": launches, "stats": stats,
            "wall0": wall0, "wall1": wall1, "graph_steps": g0[0], "graphs_captured": g0[1], "state": state}


def dump_outputs(out_dir: str, state: dict) -> None:
    """ids, x, y, vx, vy (ascending id) as DIR/<name>.npy, float64.  A crowd of more than DUMP_MAX_AGENTS agents is
    sampled: DUMP_MAX_AGENTS of them drawn with DUMP_SEED, kept in id order, the same agents in every run."""
    n = len(state["id"])
    pick = slice(None)
    if n > DUMP_MAX_AGENTS:
        pick = np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_MAX_AGENTS, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name in ("id", "x", "y", "vx", "vy"):
        np.save(os.path.join(out_dir, f"{name}.npy"), state[name][pick].astype(np.float64))


def secondary_lines(args, main_scene, peaks) -> list:
    """The rest of BASELINE.md's table in the same run: every entry is a short measurement (3 warm-up + 8 timed
    steps, CUDA events on the launching stream) of another configuration of BASELINE.json on this GPU."""
    from rmf_crowdsim_b200 import Duration, _native as N
    from rmf_crowdsim_b200 import scenes as SC

    out = []
    K, W = 8, 3

    def entry(name, scene, frozen, lp_none=False):
        t0 = time.time()
        e = {"workload": name, "agents": scene.n,
             "mode": "frozen snapshot (RCS_STEP_NO_COMMIT)" if frozen else "committed steps"}
        try:
            sim = SC.build_simulation(scene, device=0)
            flush = scene.n * 96 < (1 << 30)
            m = timed_steps(sim, scene.n, Duration(*scene.dt), frozen, K, W, flush)
            k_ms = m["kt_ms"] / max(m["kt_n"], 1)
            algo = ALGO_BYTES_NOLOCALPLAN if lp_none else ALGO_BYTES_ZANLUNGO
            st = m["stats"]
            e.update({"value": scene.n * K / (m["total_ms"] * 1e-3), "ms_per_step": m["total_ms"] / K, "kernel_ms": k_ms,
                      "frac": algo * scene.n / (k_ms * 1e-3) / 1e9 / peaks["hbm_gbs"] if k_ms > 0 else None,
                      "frac_whole_step": algo * scene.n * K / (m["total_ms"] * 1e-3) / 1e9 / peaks["hbm_gbs"],
                      "finite_tti_fraction": st.finite_tti_count / max(scene.n, 1), "nonfinite": int(st.nonfinite_count),
                      "launches_per_step": m["launches"] / K, "steps": K, "graph_steps": m["graph_steps"]})
            sim.spatial_index.close()
        except Exception as ex:  # a crowd the model drives out of bounds fails its step: say so, keep going
            e["error"] = str(ex)
        e["wall_s"] = round(time.time() - t0, 2)
        out.append(e)

    entry("C2: 10,000 agents, Zanlungo, ids shuffled", SC.config_c2("shuffled"), True)
    entry("C3: 2^20 agents, Zanlungo, ids shuffled", SC.config_c3("shuffled"), True)
    entry("C3: 2^20 agents, NoLocalPlan", SC.config_c3("shuffled", lp=("none",)), True, lp_none=True)
    if main_scene is not None and main_scene.n == 1 << 24 and main_scene.lp[0] != "none":
        nolp = main_scene
        keep_lp = nolp.lp
        nolp.lp = ("none",)
        entry("C4: 2^24 agents, NoLocalPlan", nolp, True, lp_none=True)
        nolp.lp = keep_lp
    entry("C4: 2^24 agents, Zanlungo, lane-ordered ids (force pass idle)", SC.config_c4("lane"), False)
    sparse = SC.uniform_crowd(4096, "shuffled", s=5.0, cell=5.0, eyesight=5.0, margin=40.0, seed=1,
                              lp=("zanlungo", 0.1, 1.0, 0.0, 0.4, 1.0, 0.2), name="sparse_16m")
    entry("C2-sparse parameters at 2^24 agents (5 m spacing, R = cell = 5 m), Zanlungo, force pass busy", sparse, False)
    del sparse
    # C5: SourceSink stream (rmf_crowdsim_b200/stream_bench.py), NoLocalPlan and Zanlungo
    from rmf_crowdsim_b200 import stream_bench

    for lp_none in (True, False):
        t0 = time.time()
        try:
            out.append(stream_bench.measure(lp_none, K, W, peaks))
        except Exception as ex:
            out.append({"workload": "C5 SourceSink stream", "error": str(ex)})
        out[-1]["wall_s"] = round(time.time() - t0, 2)
    return out


def kernel_counts(key: str):
    """Per-workload counters taken from the committed ncu captures (profiles/kernel_counts.json, written by
    tools/ncu_summary.py): DRAM bytes of the dominant kernel and of the whole step, FP64 instructions per agent."""
    tp = os.path.join(ROOT, "profiles", "kernel_counts.json")
    try:
        with open(tp) as f:
            return json.load(f).get(key)
    except Exception:
        return None


def fp64_info(args):
    import ctypes as C

    from rmf_crowdsim_b200 import _native as N

    try:
        a, b = C.c_double(), C.c_double()
        if N.load().rcs_fp64_peak(0, C.byref(a), C.byref(b)) == 0:
            return {"dfma_tflops": a.value, "dadd_tops": b.value}
    except Exception:
        pass
    return None


def run_e2e(scene, frozen: bool, steps: int, warmup: int) -> dict:
    """Host-buffer path: rcs_set_preferred_velocity (H2D from pinned) + rcs_step_async + rcs_read_agents
    (D2H to pinned), all inside the timed region."""
    import ctypes as C

    from rmf_crowdsim_b200 import Duration, _native as N
    from rmf_crowdsim_b200 import sim as S

    n = scene.n
    lib = N.load()
    idx = S.LocationHash2D(scene.width, scene.height, scene.cell, scene.offset, capacity=n, device=0)
    sim = S.Simulation(idx)
    h = sim._h

    class HostPlan(S.HighLevelPlanner):  # evaluated by the caller, uploaded every step
        pass

    hl = HostPlan()
    lp = S.NoLocalPlan() if scene.lp[0] == "none" else S.Zanlungo(*scene.lp[1:])
    from rmf_crowdsim_b200.scenes import add_agents_bulk

    add_agents_bulk(sim, scene.xy, hl, lp, scene.eyesight)
    sim._host_hl.clear()  # the bulk path below replaces the per-agent Python callbacks
    sim.set_state(None, vx=scene.vxy[:, 0].copy(), vy=scene.vxy[:, 1].copy())

    def pinned(count, dtype):
        p = C.c_void_p()
        nbytes = count * np.dtype(dtype).itemsize
        N.check(None, lib.rcs_host_alloc(nbytes, C.byref(p)))
        buf = (C.c_char * nbytes).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype, count=count), p

    pref, pref_p = pinned(2 * n, np.float64)
    outs2 = [[pinned(n, np.float64) for _ in range(4)] for _ in range(2)]  # double-buffered results
    outs = outs2[0] + outs2[1]
    speed = scene.hl[1]
    par = (np.arange(n) % 2 == 0)
    pref[0::2] = np.where(par, -speed[0], speed[0])
    pref[1::2] = np.where(par, -speed[1], speed[1])
    dt = Duration(*scene.dt)
    out_n = C.c_uint64()
    flags = N.RCS_STEP_NO_COMMIT if frozen else 0

    def one_sync(k):
        N.check(h, lib.rcs_set_preferred_velocity(h, n, None, pref.ctypes.data_as(N.c_f64p)))
        N.check(h, lib.rcs_step_async(h, dt.secs, dt.nanos, flags))
        N.check(h, lib.rcs_read_agents(h, N.RCS_ORDER_ID, n, None, *[o[0].ctypes.data_as(N.c_f64p) for o in outs2[0]],
                                       None, C.byref(out_n)))

    def one_async(k):
        # the read-back of step k (device -> pinned host, second stream) overlaps the upload and the compute of step
        # k + 1; every step still uploads its inputs and downloads its results
        N.check(h, lib.rcs_set_preferred_velocity(h, n, None, pref.ctypes.data_as(N.c_f64p)))
        N.check(h, lib.rcs_step_async(h, dt.secs, dt.nanos, flags))
        N.check(h, lib.rcs_read_agents_async(h, N.RCS_ORDER_ID, n, None,
                                             *[o[0].ctypes.data_as(N.c_f64p) for o in outs2[k & 1]], C.byref(out_n)))

    def timed(one):
        for k in range(warmup):
            one(k)
        N.check(h, lib.rcs_read_wait(h))
        N.check(h, lib.rcs_sync(h))
        t0 = time.perf_counter()
        for k in range(steps):
            one(k)
        N.check(h, lib.rcs_read_wait(h))  # the last step's results are on the host
        N.check(h, lib.rcs_sync(h))
        return time.perf_counter() - t0

    t_sync = timed(one_sync)
    t_async = timed(one_async)
    # both buffer sets hold results of the same frozen snapshot step: the pipelined read returns the same bits
    same = all(np.array_equal(a[0], b[0]) for a, b in zip(outs2[0], outs2[1])) if frozen else None
    res = {"value": n * steps / t_async, "unit": "agent-steps/s", "h2d_bytes_per_step": 16 * n,
           "d2h_bytes_per_step": 32 * n, "steps": steps,
           "path": "rcs_set_preferred_velocity(pinned host) + rcs_step_async + rcs_read_agents_async(ORDER_ID, pinned "
                   "host, double-buffered): the download of step k overlaps the upload and compute of step k+1",
           "synchronous_value": n * steps / t_sync,
           "synchronous_path": "same with the blocking rcs_read_agents", "buffers_identical": same}
    for _, p in [(pref, pref_p)] + outs:
        lib.rcs_host_free(p)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None)
    ap.add_argument("--variant", default="shuffled", choices=["shuffled", "lane"])
    ap.add_argument("--no-local-plan", action="store_true")
    ap.add_argument("--kernel", type=int, default=0, help="RCS_OPT_STEP_KERNEL: 0 default, 1 thread/agent, 2 warp")
    ap.add_argument("--c5-zanlungo", action="store_true", help="--workload c5 with the Zanlungo planner")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-secondary", action="store_true", help="skip the other BASELINE configurations")
    ap.add_argument("--skip-verify", action="store_true", help="--gpus N: skip the pre-timing NCCL correctness check")
    ap.add_argument("--verify-dist", action="store_true",
                    help="with --gpus N: committed steps over the NCCL transport compared bit for bit with one handle")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the agent state the last timed step produced to DIR/<name>.npy (one GPU)")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl == "reference" or args.workload == "c5" or args.gpus != 1 or world != 1):
        ap.error("--dump-outputs is implemented for the one-GPU arm only (not --impl reference, --workload c5, --gpus N)")
    if args.impl == "reference":
        run_reference(args)
        return
    if args.workload == "c5" and args.gpus == 1 and world == 1:
        from rmf_crowdsim_b200 import stream_bench

        stream_bench.run(args)
        return
    if args.gpus == 1 and world == 1:
        run_gpu_single(args)
    elif world == 1:
        # `python bench.py --gpus N` without a launcher: start one rank per GPU ourselves (the driver uses torchrun)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29517"),
               os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    else:
        from rmf_crowdsim_b200 import dist_bench

        if args.verify_dist:
            dist_bench.verify(args)
        elif args.workload == "c5":
            dist_bench.run_stream(args)
        else:
            dist_bench.run(args)


if __name__ == "__main__":
    main()
