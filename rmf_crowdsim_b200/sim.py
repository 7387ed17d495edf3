"""Host-side mirror of the reference's public interface for the hot path, over the C ABI.

Same type and method names, argument meaning and error behaviour as the Rust crate
(/root/reference/rmf_crowdsim/src): `Simulation` (lib.rs:69-384), `LocationHash2D`
(spatial_index/location_hash_2d.rs), `NoLocalPlan` / `Zanlungo` (local_planners/), `HighLevelPlanner`
(highlevel_planners/highlevel_planners.rs:8-16), `SourceSink` / `MonotonicCrowd`
(source_sink/source_sink.rs), `EventListener` (lib.rs:22-33).  `Result<_, String>` errors become
`CrowdsimError` carrying the reference's literal message.

All arithmetic happens on the GPU through librcs.so; this module only marshals.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Mapping, Optional, Sequence, Tuple

import numpy as np

from . import _native as N
from ._native import RcsError as CrowdsimError

Vec2f = Tuple[float, float]
Point = Vec2f
AgentId = int


def _f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def _u64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint64)


def _p(a: Optional[np.ndarray], ty):
    return a.ctypes.data_as(ty) if a is not None else None


@dataclass(frozen=True)
class Duration:
    """std::time::Duration: whole seconds + nanoseconds (dt = secs + nanos / 1e9, lib.rs:295)."""

    secs: int = 0
    nanos: int = 0

    def as_secs_f64(self) -> float:
        return float(self.secs) + float(self.nanos) / 1e9


@dataclass
class Agent:
    """lib.rs:46-65.  orientation / angular_vel are never written by the reference and stay 0."""

    agent_id: int
    position: Vec2f
    velocity: Vec2f
    next_waypoint: int
    eyesight_range: float = 0.0
    orientation: float = 0.0
    angular_vel: float = 0.0


# ---- local planners (descriptors; evaluated on the device) -----------------------------------
class LocalPlanner:
    def _register(self, lib, handle) -> int:  # pragma: no cover - interface
        raise NotImplementedError


class NoLocalPlan(LocalPlanner):
    """local_planners/no_local_plan.rs:7-18"""

    def _register(self, lib, handle) -> int:
        out = C.c_uint32()
        N.check(handle, lib.rcs_lp_none(handle, C.byref(out)))
        return out.value


class Zanlungo(LocalPlanner):
    """local_planners/zanlungo.rs:31-48, same argument order as Zanlungo::new."""

    def __init__(self, agent_scale, obstacle_scale, reaction_time, force_distance, agent_mass, agent_radius):
        self.params = (
            float(agent_scale),
            float(obstacle_scale),
            float(reaction_time),
            float(force_distance),
            float(agent_mass),
            float(agent_radius),
        )

    def _register(self, lib, handle) -> int:
        out = C.c_uint32()
        N.check(handle, lib.rcs_lp_zanlungo(handle, *self.params, C.byref(out)))
        return out.value


# ---- high-level planners ---------------------------------------------------------------------
class HighLevelPlanner:
    """highlevel_planners/highlevel_planners.rs:8-16.  Subclass and override to run a planner on the
    host (slow path: positions are read back, get_desired_velocity is called per agent, the
    results are uploaded before each step)."""

    device_kind: Optional[str] = None

    def get_desired_velocity(self, agent: Agent, time: Duration) -> Optional[Vec2f]:
        raise NotImplementedError

    def set_target(self, agent: Agent, point: Vec2f, tolerance: Vec2f) -> None:
        pass

    def remove_agent_id(self, agent: AgentId) -> None:
        pass


class ConstantVelocityPlan(HighLevelPlanner):
    """The fixture planner of lib.rs:391-420 (always Some(default_vel)), evaluated on the device."""

    device_kind = "constant"

    def __init__(self, default_vel: Vec2f):
        self.default_vel = (float(default_vel[0]), float(default_vel[1]))

    def get_desired_velocity(self, agent, time):
        return self.default_vel


class ParityVelocityPlan(HighLevelPlanner):
    """The fixture planner of rmf_crowdsim_viz/src/main.rs:20-30 (even id -> -v, odd -> +v)."""

    device_kind = "parity"

    def __init__(self, default_vel: Vec2f):
        self.default_vel = (float(default_vel[0]), float(default_vel[1]))

    def get_desired_velocity(self, agent, time):
        v = self.default_vel
        return (-v[0], -v[1]) if agent.agent_id % 2 == 0 else v


class RouteFollowPlan(HighLevelPlanner):
    """The per-step half of rmf::RMFPlanner (rmf/mod.rs:197-215) on a caller-supplied route, evaluated on the
    device: head for route[k], advance once within 0.1 m, return the UNIT vector towards it.  Agents enter the
    planner's cache (at route point 0) when a SourceSink spawns them or sends them to its next waypoint, or
    through Simulation.route_set_target.  Route planning itself (`mapf` A*) is not part of this library."""

    device_kind = "route"

    def __init__(self, route: Sequence[Vec2f]):
        self.route = [(float(p[0]), float(p[1])) for p in route]


class RouteTablePlan(HighLevelPlanner):
    """rmf::RMFPlanner (rmf/mod.rs:86-241) with a route cache the caller has filled, evaluated on the device.
    `routes` maps each target point to the route (leg) that set_target(agent, target, ..) selects.  set_target makes the
    leg whose target equals the point (IEEE == on both coordinates) the agent's current leg, at its route point 0;
    get_desired_velocity is RouteFollowPlan's follower on that leg.  A SourceSink calls set_target with waypoints[0] at
    the spawn and with waypoints[k + 1] at every advance (not at a loop_forever wrap), so a SourceSink with this planner
    may have any number of waypoints, each of which must have a leg.  Route planning itself (`mapf`) stays outside."""

    device_kind = "route_table"

    def __init__(self, routes: Mapping[Vec2f, Sequence[Vec2f]]):
        self.routes = {(float(t[0]), float(t[1])): [(float(p[0]), float(p[1])) for p in r] for t, r in routes.items()}


class NoHighLevelPlan(HighLevelPlanner):
    """Always None: velocity (0,0) (lib.rs:263-273)."""

    device_kind = "none"

    def get_desired_velocity(self, agent, time):
        return None


# ---- source sinks ----------------------------------------------------------------------------
class CrowdGenerator:
    """source_sink.rs:63-66.  Subclass and override get_number_to_spawn to run a generator on the host: the simulation
    calls it once per step for every alive source sink that has it (in ascending source-sink id) and uploads the counts
    before the step.  Only "at least one" matters: a source spawns at most one agent per step (lib.rs:207-219)."""

    def get_number_to_spawn(self, time_elapsed: Duration) -> int:
        raise NotImplementedError


class MonotonicCrowd(CrowdGenerator):
    """source_sink.rs:85-100: round(dt * rate) agents per step, no fractional carry."""

    def __init__(self, rate: float):
        self.rate = float(rate)

    def get_number_to_spawn(self, time_elapsed: Duration) -> int:
        x = time_elapsed.as_secs_f64() * self.rate
        if not x > 0:  # f64::round (half away from zero) then the saturating `as usize`
            return 0
        r = np.floor(x)
        return int(r + 1) if x - r >= 0.5 else int(r)


class PoissonCrowd(CrowdGenerator):
    """source_sink.rs:63-82, drawn on the device with a keyed generator instead of thread_rng, so that runs are
    reproducible.  `seed` is an addition to the reference's constructor.  Source sink `sid` wants to spawn in the step
    that starts with stats().steps == k iff (word 0 of Philox4x64-10, counter (k + 1, sid, 0, 0), key (seed, 0)) >> 11
    >= ceil(exp(-dt * rate) * 2^53): probability 1 - exp(-dt * rate) = P(Poisson(dt * rate) >= 1).  rate must be finite
    and > 0, and a step with dt * rate <= 0 is refused (Poisson::new fails in the reference)."""

    def __init__(self, rate: float, seed: int = 0):
        self.rate = float(rate)
        self.seed = int(seed)

    def get_number_to_spawn(self, time_elapsed: Duration) -> int:
        raise NotImplementedError("PoissonCrowd is drawn on the device inside Simulation.step")


@dataclass
class SourceSink:
    """source_sink.rs:36-60"""

    source: Vec2f
    radius_sink: float
    crowd_generator: CrowdGenerator
    high_level_planner: HighLevelPlanner
    local_planner: LocalPlanner
    waypoints: List[Vec2f]
    loop_forever: bool
    agent_eyesight_range: float


class EventListener:
    """lib.rs:22-33"""

    def agent_spawned(self, position: Vec2f, agent: AgentId) -> None:
        pass

    def agent_destroyed(self, agent: AgentId) -> None:
        pass

    def waypoint_reached(self, position: Vec2f, agent: AgentId) -> None:  # never invoked by the reference
        pass


# ---- spatial index ---------------------------------------------------------------------------
class LocationHash2D:
    """spatial_index/location_hash_2d.rs: LocationHash2D::new(width, height, cell_size, offset).

    Owns the device handle.  Usable on its own through the SpatialIndex trait methods
    (add_or_update / get_neighbours_in_radius / get_nearest_neighbours / remove_agent) or handed to
    `Simulation(spatial_index)`.  `capacity` and `device` are the only additions to the reference's
    constructor (device memory is sized up front)."""

    def __init__(self, width, height, cell_size, offset: Point, capacity: int = 1 << 16, device: int = 0):
        self._lib = N.load()
        desc = N.SimDesc(float(width), float(height), float(cell_size), float(offset[0]), float(offset[1]),
                         int(capacity), int(device), 0)
        h = C.c_void_p()
        rc = self._lib.rcs_sim_create(C.byref(desc), C.byref(h))
        if rc != N.RCS_OK:
            raise CrowdsimError(rc, (self._lib.rcs_last_error(None) or b"").decode())
        self._h = h
        self.capacity = int(capacity)

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.rcs_sim_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # SpatialIndex trait (spatial_index.rs:4-14)
    def add_or_update(self, index: AgentId, position: Point) -> None:
        ids = _u64([index])
        xy = _f64([position[0], position[1]])
        N.check(self._h, self._lib.rcs_index_add_or_update(self._h, 1, _p(ids, N.c_u64p), _p(xy, N.c_f64p)))

    def add_or_update_many(self, ids, xy) -> None:
        ids = _u64(ids)
        xy = _f64(xy).reshape(-1)
        N.check(self._h, self._lib.rcs_index_add_or_update(self._h, len(ids), _p(ids, N.c_u64p), _p(xy, N.c_f64p)))

    def remove_agent(self, agent: AgentId) -> None:
        ids = _u64([agent])
        N.check(self._h, self._lib.rcs_index_remove(self._h, 1, _p(ids, N.c_u64p)))

    def get_neighbours_in_radius(self, radius: float, position: Point) -> List[AgentId]:
        off, ids = self.query_radius(_f64([[position[0], position[1]]]), _f64([radius]))
        return [int(v) for v in ids]

    def query_radius(self, qxy: np.ndarray, radius: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        """Batched get_neighbours_in_radius: CSR (offsets[nq+1], ids)."""
        qxy = _f64(qxy).reshape(-1, 2)
        nq = qxy.shape[0]
        radius = np.broadcast_to(_f64(radius), (nq,)).copy()
        offsets = np.zeros(nq + 1, dtype=np.uint64)
        cap = max(64, 64 * nq)
        while True:
            ids = np.zeros(cap, dtype=np.uint64)
            rc = self._lib.rcs_query_radius(self._h, nq, _p(qxy, N.c_f64p), _p(radius, N.c_f64p),
                                            _p(offsets, N.c_u64p), _p(ids, N.c_u64p), cap)
            if rc == N.RCS_ERR_CAPACITY:
                cap = int(offsets[nq]) + 1
                continue
            N.check(self._h, rc)
            return offsets, ids[: int(offsets[nq])]

    def get_nearest_neighbours(self, n: int, position: Point) -> List[AgentId]:
        ids, counts = self.query_knn(_f64([[position[0], position[1]]]), n)
        return [int(v) for v in ids[0, : int(counts[0])]]

    def query_knn(self, qxy: np.ndarray, k: int) -> Tuple[np.ndarray, np.ndarray]:
        """Batched get_nearest_neighbours: ids[nq, max(k, 1)] and counts[nq].  Raises CrowdsimError where the
        reference's sort panics: a query with >= 2 candidates of which one is at a NaN distance."""
        qxy = _f64(qxy).reshape(-1, 2)
        nq = qxy.shape[0]
        ids = np.zeros((nq, max(k, 1)), dtype=np.uint64)
        counts = np.zeros(nq, dtype=np.uint64)
        N.check(self._h, self._lib.rcs_query_knn(self._h, nq, _p(qxy, N.c_f64p), int(k), _p(ids, N.c_u64p),
                                                 _p(counts, N.c_u64p)))
        return ids, counts

    def cell_of(self, xy: np.ndarray) -> np.ndarray:
        """location_to_index for many points: data index, or -1 for "Index out of bounds"."""
        xy = _f64(xy).reshape(-1, 2)
        out = np.zeros(xy.shape[0], dtype=np.int64)
        N.check(self._h, self._lib.rcs_cell_of(self._h, xy.shape[0], _p(xy, N.c_f64p), _p(out, N.c_i64p)))
        return out


# ---- the simulation --------------------------------------------------------------------------
class Simulation:
    """lib.rs:69-384.  `Simulation(spatial_index)` = Simulation::new; `step(dur)` runs the whole
    per-timestep update on the GPU."""

    def __init__(self, spatial_index: LocationHash2D):
        self.spatial_index = spatial_index
        self._lib = spatial_index._lib
        self._h = spatial_index._h
        self._lp_handles: Dict[int, Tuple[LocalPlanner, int]] = {}
        self._hl_handles: Dict[int, Tuple[HighLevelPlanner, int]] = {}
        self._host_hl: Dict[int, HighLevelPlanner] = {}  # agent id -> host-evaluated planner
        self._host_hl_handle: Optional[int] = None
        self._host_ss: Dict[Tuple[float, float], SourceSink] = {}  # source position -> sink with a host planner
        self._host_ss_of: Dict[int, SourceSink] = {}  # agent id -> the sink that spawned it (host planners only)
        self._eyesight: Dict[int, float] = {}
        self._listeners: Dict[int, EventListener] = {}
        self._listener_counter = 0
        self._source_sinks: Dict[int, SourceSink] = {}
        self._host_gen: Dict[int, CrowdGenerator] = {}  # source-sink id -> generator evaluated on the host
        self.sim_time = Duration(0, 0)  # never advanced by the reference (lib.rs:81,110)

    # -- planner registration ------------------------------------------------------------------
    def _lp(self, lp: LocalPlanner) -> int:
        ent = self._lp_handles.get(id(lp))
        if ent is None:
            ent = (lp, lp._register(self._lib, self._h))
            self._lp_handles[id(lp)] = ent
        return ent[1]

    def _hl(self, hl: HighLevelPlanner) -> int:
        ent = self._hl_handles.get(id(hl))
        if ent is not None:
            return ent[1]
        out = C.c_uint32()
        kind = hl.device_kind
        if kind == "constant":
            N.check(self._h, self._lib.rcs_hl_constant(self._h, hl.default_vel[0], hl.default_vel[1], C.byref(out)))
        elif kind == "parity":
            N.check(self._h, self._lib.rcs_hl_parity(self._h, hl.default_vel[0], hl.default_vel[1], C.byref(out)))
        elif kind == "none":
            N.check(self._h, self._lib.rcs_hl_none(self._h, C.byref(out)))
        elif kind == "route":
            r = _f64(hl.route).reshape(-1)
            N.check(self._h, self._lib.rcs_hl_route(self._h, len(r) // 2, _p(r, N.c_f64p), C.byref(out)))
        elif kind == "route_table":
            legs = list(hl.routes.items())
            targets = _f64([t for t, _ in legs]).reshape(-1)
            counts = _u64([len(r) for _, r in legs])
            xy = _f64([p for _, r in legs for p in r]).reshape(-1)
            N.check(self._h, self._lib.rcs_hl_route_table(self._h, len(legs), _p(targets, N.c_f64p),
                                                          _p(counts, N.c_u64p), _p(xy, N.c_f64p), C.byref(out)))
        else:
            if self._host_hl_handle is None:
                N.check(self._h, self._lib.rcs_hl_host(self._h, C.byref(out)))
                self._host_hl_handle = out.value
            out = C.c_uint32(self._host_hl_handle)
        self._hl_handles[id(hl)] = (hl, out.value)
        return out.value

    # -- lib.rs:119-156 ------------------------------------------------------------------------
    def add_agents(self, spawn_positions: Sequence[Point], high_level_planner: HighLevelPlanner,
                   local_planner: LocalPlanner, agent_eyesight_range: float) -> List[AgentId]:
        xy = _f64(spawn_positions).reshape(-1, 2)
        n = xy.shape[0]
        ids = np.zeros(n, dtype=np.uint64)
        hl = self._hl(high_level_planner)
        lp = self._lp(local_planner)
        N.check(self._h, self._lib.rcs_add_agents(self._h, n, _p(xy, N.c_f64p), hl, lp,
                                                  float(agent_eyesight_range), _p(ids, N.c_u64p)))
        out = [int(v) for v in ids]
        if high_level_planner.device_kind is None:
            for a in out:
                self._host_hl[a] = high_level_planner
        if self._listeners:
            for k, a in enumerate(out):
                for key in sorted(self._listeners):
                    self._listeners[key].agent_spawned((float(xy[k, 0]), float(xy[k, 1])), a)
        return out

    # -- lib.rs:159-173 ------------------------------------------------------------------------
    def add_source_sink(self, source_sink: SourceSink) -> int:
        wp = _f64(source_sink.waypoints).reshape(-1, 2)
        gen = source_sink.crowd_generator
        if not isinstance(gen, CrowdGenerator):
            raise CrowdsimError(N.RCS_ERR_ARG, "the crowd generator must be a CrowdGenerator")
        if isinstance(gen, MonotonicCrowd):
            gdesc, rate = None, gen.rate
        elif isinstance(gen, PoissonCrowd):
            if not 0 <= gen.seed < 1 << 64:
                raise CrowdsimError(N.RCS_ERR_ARG, "PoissonCrowd: the seed must lie in [0, 2^64)")
            gdesc, rate = N.CrowdGeneratorDesc(N.RCS_CROWD_POISSON, 0, gen.rate, gen.seed), 0.0
        else:  # a user-implemented generator: evaluated on the host before every step (_run_host_generators)
            gdesc, rate = N.CrowdGeneratorDesc(N.RCS_CROWD_HOST, 0, 0.0, 0), 0.0
        desc = N.SourceSinkDesc(float(source_sink.source[0]), float(source_sink.source[1]),
                                float(source_sink.radius_sink), float(rate),
                                self._hl(source_sink.high_level_planner), self._lp(source_sink.local_planner),
                                wp.shape[0], _p(wp, N.c_f64p), 1 if source_sink.loop_forever else 0,
                                float(source_sink.agent_eyesight_range))
        host_key = None
        if source_sink.high_level_planner.device_kind is None:
            # A planner evaluated on the host: its spawned agents are recognised by their spawn position when the
            # spawn events are dispatched (_dispatch_events), so two such source sinks cannot share a source point.
            host_key = (float(source_sink.source[0]), float(source_sink.source[1]))
            if host_key in self._host_ss:
                raise CrowdsimError(N.RCS_ERR_ARG, "two source sinks with host-evaluated HighLevelPlanners share a "
                                                   "source position")
        out = C.c_uint64()
        if gdesc is None:
            N.check(self._h, self._lib.rcs_add_source_sink(self._h, C.byref(desc), C.byref(out)))
        else:
            N.check(self._h, self._lib.rcs_add_source_sink_gen(self._h, C.byref(desc), C.byref(gdesc), C.byref(out)))
        self._source_sinks[out.value] = source_sink
        if gdesc is not None and gdesc.kind == N.RCS_CROWD_HOST:
            self._host_gen[out.value] = gen
        if host_key is not None:
            self._host_ss[host_key] = source_sink
        return out.value

    def remove_source_sink(self, id: int) -> None:
        N.check(self._h, self._lib.rcs_remove_source_sink(self._h, int(id)))
        self._host_gen.pop(int(id), None)
        ss = self._source_sinks.pop(int(id), None)
        if ss is not None:
            self._host_ss.pop((float(ss.source[0]), float(ss.source[1])), None)

    def add_event_listener(self, event_listener: EventListener) -> int:
        k = self._listener_counter
        self._listeners[k] = event_listener
        self._listener_counter += 1
        return k

    # -- lib.rs:176-192 ------------------------------------------------------------------------
    def remove_agents(self, agent: AgentId) -> None:
        ids = _u64([agent])
        N.check(self._h, self._lib.rcs_remove_agents(self._h, 1, _p(ids, N.c_u64p)))
        self._host_ss_of.pop(int(agent), None)
        hl = self._host_hl.pop(int(agent), None)
        if hl is not None:
            hl.remove_agent_id(int(agent))
        for key in sorted(self._listeners):
            self._listeners[key].agent_destroyed(int(agent))

    # -- lib.rs:195-383 ------------------------------------------------------------------------
    def step(self, dur: Duration) -> None:
        """Err(String) of the reference becomes CrowdsimError with the same message."""
        before = self._run_host_planners() if self._host_hl else None
        self._run_host_generators(dur)
        N.check(self._h, self._lib.rcs_step(self._h, int(dur.secs), int(dur.nanos)))
        self._dispatch_events(before)

    def step_in_loop(self, dur: Duration, order=None, max_sweeps: int = 0) -> int:
        """One step under the reference's in-loop index semantic (lib.rs:299; SURVEY.md 8f-4) for the iteration order
        `order` (agent ids; None = ascending id).  Ids that are not live are ignored; live agents missing from `order`
        are visited after it in ascending id; an order that repeats an id raises CrowdsimError and changes nothing.
        max_sweeps = 0: no limit; otherwise a step without a fixed point within max_sweeps raises and commits nothing
        (max_sweeps = 1 always does: sweep 0 has nothing to agree with).  Returns the number of whole-crowd sweeps
        the fixed point took."""
        if self._host_hl:
            self._run_host_planners()
        sweeps = C.c_uint32()
        if order is None:
            rc = self._lib.rcs_step_in_loop(self._h, int(dur.secs), int(dur.nanos), None, 0, max_sweeps, C.byref(sweeps))
        else:
            order = _u64(order)
            rc = self._lib.rcs_step_in_loop(self._h, int(dur.secs), int(dur.nanos), _p(order, N.c_u64p), len(order),
                                            max_sweeps, C.byref(sweeps))
        N.check(self._h, rc)
        return int(sweeps.value)

    def step_async(self, dur: Duration, no_commit: bool = False) -> None:
        flags = N.RCS_STEP_NO_COMMIT if no_commit else N.RCS_STEP_DEFAULT
        self._run_host_generators(dur)
        N.check(self._h, self._lib.rcs_step_async(self._h, int(dur.secs), int(dur.nanos), flags))

    def sync(self) -> None:
        N.check(self._h, self._lib.rcs_sync(self._h))

    def _run_host_generators(self, dur: Duration) -> None:
        """get_number_to_spawn(dur) of every alive host-evaluated CrowdGenerator, in ascending source-sink id, uploaded
        as the counts of the next step (rcs_set_spawn_counts)."""
        if not self._host_gen:
            return
        ids = sorted(self._host_gen)
        counts = _u64([int(self._host_gen[i].get_number_to_spawn(dur)) for i in ids])
        ids = _u64(ids)
        N.check(self._h, self._lib.rcs_set_spawn_counts(self._h, len(ids), _p(ids, N.c_u64p), _p(counts, N.c_u64p)))

    def _run_host_planners(self) -> Dict[str, np.ndarray]:
        """Uploads the host planners' preferred velocities; returns the pre-step state it read."""
        st = self.read_state()
        ids = st["id"]
        sel, vxy = [], []
        nan = float("nan")
        for k in range(len(ids)):
            a = int(ids[k])
            hl = self._host_hl.get(a)
            if hl is None:
                continue
            agent = Agent(a, (float(st["x"][k]), float(st["y"][k])), (float(st["vx"][k]), float(st["vy"][k])),
                          int(st["next_waypoint"][k]))
            v = hl.get_desired_velocity(agent, self.sim_time)
            sel.append(a)
            vxy.append((nan, nan) if v is None else (float(v[0]), float(v[1])))
        if sel:
            self.set_preferred_velocity(np.array(sel, dtype=np.uint64), np.array(vxy, dtype=np.float64))
        return st

    def _dispatch_events(self, before: Optional[Dict[str, np.ndarray]] = None) -> None:
        """Spawn events, then set_target for the host-planned agents that reached an intermediate waypoint in the step
        (`before`: the state the step started from), then destroy events -- the reference's order (lib.rs:242-249,
        :326-333, :378-380)."""
        ns, nd = C.c_uint64(), C.c_uint64()
        N.check(self._h, self._lib.rcs_poll_events(self._h, 0, None, None, C.byref(ns), 0, None, C.byref(nd)))
        if ns.value == 0 and nd.value == 0:
            if before is not None and self._host_ss_of:
                self._host_waypoint_targets(before, {})
            return
        sid = np.zeros(max(ns.value, 1), dtype=np.uint64)
        sxy = np.zeros(2 * max(ns.value, 1), dtype=np.float64)
        did = np.zeros(max(nd.value, 1), dtype=np.uint64)
        N.check(self._h, self._lib.rcs_poll_events(self._h, len(sid), _p(sid, N.c_u64p), _p(sxy, N.c_f64p),
                                                   C.byref(ns), len(did), _p(did, N.c_u64p), C.byref(nd)))
        spawned: Dict[int, Point] = {}  # host-planned agents spawned in this step
        for k in range(ns.value):
            pos = (float(sxy[2 * k]), float(sxy[2 * k + 1]))
            ss = self._host_ss.get(pos) if self._host_ss else None
            if ss is not None:
                # lib.rs:242-249: set_target(agent, waypoints[0], (radius_sink, radius_sink)) right after the spawn.
                # The agent was spawned inside the device step with preferred velocity None, so it starts to move
                # with the NEXT step (the reference moves it in its spawn step already: one step of delay for
                # host-evaluated planners only, INTEGRATION.md).
                hl = ss.high_level_planner
                self._host_hl[int(sid[k])] = hl
                self._host_ss_of[int(sid[k])] = ss
                wp0 = ss.waypoints[0]
                hl.set_target(Agent(int(sid[k]), pos, (0.0, 0.0), 0), (float(wp0[0]), float(wp0[1])),
                              (float(ss.radius_sink), float(ss.radius_sink)))
                spawned[int(sid[k])] = pos
            for key in sorted(self._listeners):
                self._listeners[key].agent_spawned(pos, int(sid[k]))
        if before is not None and self._host_ss_of:
            self._host_waypoint_targets(before, spawned)
        for k in range(nd.value):
            self._host_ss_of.pop(int(did[k]), None)
            hl = self._host_hl.pop(int(did[k]), None)
            if hl is not None:
                hl.remove_agent_id(int(did[k]))
            for key in sorted(self._listeners):
                self._listeners[key].agent_destroyed(int(did[k]))

    def _host_waypoint_targets(self, before: Dict[str, np.ndarray], spawned: Dict[int, Point]) -> None:
        """lib.rs:326-333: an agent whose next_waypoint advanced k -> k + 1 in the step gets set_target(agent,
        waypoints[k + 1], (radius_sink, radius_sink)), with the agent as the step found it, in ascending id.  The loop
        wrap (last -> 0) calls nothing; agents removed in the step are no longer in the state and get no call."""
        after = self.read_state()
        pre = {int(a): k for k, a in enumerate(before["id"])}
        for k, a in enumerate(after["id"]):
            a = int(a)
            ss = self._host_ss_of.get(a)
            if ss is None:
                continue
            j = pre.get(a)
            if j is not None:
                agent = Agent(a, (float(before["x"][j]), float(before["y"][j])),
                              (float(before["vx"][j]), float(before["vy"][j])), int(before["next_waypoint"][j]))
            elif a in spawned:  # spawned in this step: it starts at the source, at rest, heading for waypoint 0
                agent = Agent(a, spawned[a], (0.0, 0.0), 0)
            else:
                continue
            wp = int(after["next_waypoint"][k])
            if wp == agent.next_waypoint + 1:
                p = ss.waypoints[wp]
                ss.high_level_planner.set_target(agent, (float(p[0]), float(p[1])),
                                                 (float(ss.radius_sink), float(ss.radius_sink)))

    # -- the pub `agents` field (lib.rs:71) ----------------------------------------------------
    def agent_count(self) -> int:
        out = C.c_uint64()
        N.check(self._h, self._lib.rcs_agent_count(self._h, C.byref(out)))
        return out.value

    def read_state(self, order: int = N.RCS_ORDER_ID) -> Dict[str, np.ndarray]:
        """Structure-of-arrays snapshot of `agents` (ascending id by default)."""
        n = self.agent_count()
        ids = np.zeros(n, dtype=np.uint64)
        x, y, vx, vy = (np.zeros(n, dtype=np.float64) for _ in range(4))
        wp = np.zeros(n, dtype=np.uint32)
        out_n = C.c_uint64()
        N.check(self._h, self._lib.rcs_read_agents(self._h, order, n, _p(ids, N.c_u64p), _p(x, N.c_f64p),
                                                   _p(y, N.c_f64p), _p(vx, N.c_f64p), _p(vy, N.c_f64p),
                                                   _p(wp, N.c_u32p), C.byref(out_n)))
        return {"id": ids, "x": x, "y": y, "vx": vx, "vy": vy, "next_waypoint": wp}

    @property
    def agents(self) -> Dict[AgentId, Agent]:
        st = self.read_state()
        return {
            int(i): Agent(int(i), (float(x), float(y)), (float(vx), float(vy)), int(w))
            for i, x, y, vx, vy, w in zip(st["id"], st["x"], st["y"], st["vx"], st["vy"], st["next_waypoint"])
        }

    def set_state(self, ids, x=None, y=None, vx=None, vy=None) -> None:
        """Write `agents[id].position / .velocity` (pub fields).  ids=None: all agents, ascending id."""
        arrs = [None if a is None else _f64(a) for a in (x, y, vx, vy)]
        n = next(len(a) for a in arrs if a is not None)
        idp = None
        if ids is not None:
            ids = _u64(ids)
            idp = _p(ids, N.c_u64p)
        N.check(self._h, self._lib.rcs_set_state(self._h, n, idp, *[_p(a, N.c_f64p) for a in arrs]))

    def route_set_target(self, ids) -> None:
        """HighLevelPlanner::set_target for agents of a RouteFollowPlan: enter the cache at route point 0."""
        ids = _u64(ids)
        N.check(self._h, self._lib.rcs_hl_route_set_target(self._h, len(ids), _p(ids, N.c_u64p)))

    def route_table_set_target(self, planner: RouteTablePlan, ids, targets) -> None:
        """HighLevelPlanner::set_target(agent, targets[i], ..) of a RouteTablePlan for the agents ids[i], which it must
        drive: each enters the cache at the head of the leg its target selects.  An unknown id, an agent of another
        planner or a target without a leg raises CrowdsimError and changes nothing."""
        ids = _u64(ids)
        xy = _f64(targets).reshape(-1)
        if len(xy) != 2 * len(ids):
            raise CrowdsimError(N.RCS_ERR_ARG, "route_table_set_target: one target point per id")
        N.check(self._h, self._lib.rcs_hl_route_table_set_target(self._h, self._hl(planner), len(ids),
                                                                 _p(ids, N.c_u64p), _p(xy, N.c_f64p)))

    def set_preferred_velocity(self, ids, vxy) -> None:
        vxy = _f64(vxy).reshape(-1)
        idp = None
        if ids is not None:
            ids = _u64(ids)
            idp = _p(ids, N.c_u64p)
        N.check(self._h, self._lib.rcs_set_preferred_velocity(self._h, len(vxy) // 2, idp, _p(vxy, N.c_f64p)))

    # -- parity / measurement helpers ------------------------------------------------------------
    def set_trace(self, on: bool) -> None:
        N.check(self._h, self._lib.rcs_set_trace(self._h, 1 if on else 0))

    def read_trace(self, neighbours: bool = True) -> Dict[str, np.ndarray]:
        """Trace of the last step in ascending-id order.  neighbours=False skips the neighbour id lists (their
        lengths are still in nb_offsets): the lists of a 2^24-agent crowd are 1.4 GB."""
        na, nn = C.c_uint64(), C.c_uint64()
        N.check(self._h, self._lib.rcs_trace_sizes(self._h, C.byref(na), C.byref(nn)))
        ids = np.zeros(na.value, dtype=np.uint64)
        ti, fx, fy = (np.zeros(na.value, dtype=np.float64) for _ in range(3))
        off = np.zeros(na.value + 1, dtype=np.uint64)
        nb = np.zeros(max(nn.value, 1) if neighbours else 0, dtype=np.uint64)
        N.check(self._h, self._lib.rcs_read_trace(self._h, _p(ids, N.c_u64p), _p(ti, N.c_f64p), _p(fx, N.c_f64p),
                                                  _p(fy, N.c_f64p), _p(off, N.c_u64p),
                                                  _p(nb, N.c_u64p) if neighbours else None))
        return {"id": ids, "t_i": ti, "fx": fx, "fy": fy, "nb_offsets": off,
                "nb_ids": nb[: nn.value] if neighbours else None}

    def set_option(self, option: int, value: int) -> None:
        N.check(self._h, self._lib.rcs_set_option(self._h, int(option), int(value)))

    def stats(self) -> N.Stats:
        st = N.Stats()
        N.check(self._h, self._lib.rcs_step_stats(self._h, C.byref(st)))
        return st

    def event_record(self, slot: int) -> None:
        N.check(self._h, self._lib.rcs_event_record(self._h, slot))

    def event_elapsed_ms(self, a: int, b: int) -> float:
        out = C.c_float()
        N.check(self._h, self._lib.rcs_event_elapsed_ms(self._h, a, b, C.byref(out)))
        return out.value

    def flush_l2(self, nbytes: int = 256 << 20) -> None:
        N.check(self._h, self._lib.rcs_flush_l2(self._h, nbytes))

    def graph_stats(self) -> Tuple[int, int]:
        """(steps that ran as one CUDA graph launch, graphs captured) -- RCS_OPT_GRAPHS."""
        a, b = C.c_uint64(), C.c_uint64()
        N.check(self._h, self._lib.rcs_graph_stats(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def launch_count(self) -> int:
        out = C.c_uint64()
        N.check(self._h, self._lib.rcs_launch_count(self._h, C.byref(out)))
        return out.value
