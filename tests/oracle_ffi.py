"""ctypes wrapper of the CPU oracle (oracle/oracle_capi.cpp).  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB = os.path.join(ORACLE_DIR, "_build", "liboracle.so")
SELFTEST = os.path.join(ORACLE_DIR, "_build", "selftest")

u64p = C.POINTER(C.c_uint64)
i64p = C.POINTER(C.c_int64)
f64p = C.POINTER(C.c_double)

_lib = None


def build() -> None:
    srcs = [os.path.join(ORACLE_DIR, f) for f in ("oracle_capi.cpp", "flat_parallel.cpp", "crowdsim_oracle.hpp", "selftest.cpp")]
    stale = (not os.path.exists(LIB)) or (not os.path.exists(SELFTEST)) or any(
        os.path.getmtime(s) > min(os.path.getmtime(LIB), os.path.getmtime(SELFTEST)) for s in srcs)
    if stale:
        subprocess.run(["make", "-C", ORACLE_DIR, "-s"], check=True)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB)
        L.orc_sim_create.restype = C.c_void_p
        L.orc_sim_create.argtypes = [C.c_double] * 5 + [C.c_int] * 3
        L.orc_sim_destroy.argtypes = [C.c_void_p]
        L.orc_last_error.restype = C.c_char_p
        L.orc_last_error.argtypes = [C.c_void_p]
        L.orc_lp_none.argtypes = [C.c_void_p]
        L.orc_lp_zanlungo.argtypes = [C.c_void_p] + [C.c_double] * 6
        for f in (L.orc_hl_constant, L.orc_hl_parity):
            f.argtypes = [C.c_void_p, C.c_double, C.c_double]
        L.orc_hl_host.argtypes = [C.c_void_p]
        L.orc_hl_route.argtypes = [C.c_void_p, C.c_uint64, f64p]
        L.orc_hl_set_target.argtypes = [C.c_void_p, C.c_int, C.c_uint64, u64p]
        L.orc_add_agents.argtypes = [C.c_void_p, C.c_uint64, f64p, C.c_int, C.c_int, C.c_double, u64p]
        L.orc_remove_agent.argtypes = [C.c_void_p, C.c_uint64]
        L.orc_set_state.argtypes = [C.c_void_p, C.c_uint64, u64p, f64p, f64p, f64p, f64p]
        L.orc_set_preferred_velocity.argtypes = [C.c_void_p, C.c_int, C.c_uint64, u64p, f64p]
        L.orc_add_source_sink.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int,
                                          C.c_int, C.c_uint64, f64p, C.c_int, C.c_double, u64p]
        L.orc_enable_trace.argtypes = [C.c_void_p, C.c_int]
        L.orc_set_custom_order.argtypes = [C.c_void_p, C.c_uint64, u64p]
        L.orc_step.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32]
        L.orc_agent_count.restype = C.c_uint64
        L.orc_agent_count.argtypes = [C.c_void_p]
        L.orc_read_agents.argtypes = [C.c_void_p, u64p, f64p, f64p, f64p, f64p, u64p]
        L.orc_trace_agent_count.restype = C.c_uint64
        L.orc_trace_agent_count.argtypes = [C.c_void_p]
        L.orc_trace_neighbour_total.restype = C.c_uint64
        L.orc_trace_neighbour_total.argtypes = [C.c_void_p]
        L.orc_read_trace.argtypes = [C.c_void_p, u64p, f64p, f64p, f64p, u64p, u64p]
        L.orc_poll_events.argtypes = [C.c_void_p, u64p, f64p, C.c_uint64, u64p, u64p, C.c_uint64, u64p]
        L.orc_index_add_or_update.argtypes = [C.c_void_p, C.c_uint64, C.c_double, C.c_double]
        L.orc_index_remove.argtypes = [C.c_void_p, C.c_uint64]
        L.orc_cell_of.restype = C.c_int64
        L.orc_cell_of.argtypes = [C.c_void_p, C.c_double, C.c_double]
        L.orc_query_radius.restype = C.c_uint64
        L.orc_query_radius.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, u64p, C.c_uint64]
        L.orc_query_knn.restype = C.c_uint64
        L.orc_query_knn.argtypes = [C.c_void_p, C.c_uint64, C.c_double, C.c_double, u64p, C.c_uint64]
        L.orc_query_bounds.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, i64p]
        L.orc_ttc.restype = C.c_double
        L.orc_ttc.argtypes = [C.c_double] * 5
        L.orc_agent_force.argtypes = [f64p, C.c_uint64, f64p, C.c_uint64, f64p, C.c_double, f64p]
        L.orc_flat_step.restype = C.c_int
        L.orc_flat_step.argtypes = [C.c_uint64, f64p, f64p, f64p, f64p, C.c_double, C.c_double, C.c_double, C.c_double,
                                    C.c_double, f64p, C.c_double, C.c_double, C.c_double, C.c_uint64, C.c_uint32,
                                    C.c_int, f64p]
        L.orc_flat_step_trace.restype = C.c_int
        L.orc_flat_step_trace.argtypes = L.orc_flat_step.argtypes + [C.POINTER(C.c_uint32), f64p, f64p, u64p]
        L.orc_duration_as_secs_f64.restype = C.c_double
        L.orc_duration_as_secs_f64.argtypes = [C.c_uint64, C.c_uint32]
        _lib = L
    return _lib


def _p(a, ty):
    return a.ctypes.data_as(ty) if a is not None else None


class OracleError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(msg)
        self.code = code


DEFERRED, IN_LOOP = 0, 1
ASCENDING_ID, MAP_ORDER, CUSTOM = 0, 1, 2


class OracleSim:
    """Drives the C++ restatement with the same call shapes as rmf_crowdsim_b200.Simulation."""

    def __init__(self, width, height, cell, offset, index_mode=DEFERRED, iter_order=ASCENDING_ID, canonical=True):
        self.L = lib()
        self.h = C.c_void_p(self.L.orc_sim_create(width, height, cell, offset[0], offset[1], index_mode, iter_order,
                                                  1 if canonical else 0))

    def __del__(self):
        try:
            self.L.orc_sim_destroy(self.h)
        except Exception:
            pass

    def _check(self, rc):
        if rc:
            raise OracleError(rc, self.L.orc_last_error(self.h).decode())

    def lp_none(self):
        return self.L.orc_lp_none(self.h)

    def lp_zanlungo(self, *p):
        return self.L.orc_lp_zanlungo(self.h, *[float(v) for v in p])

    def hl_constant(self, v):
        return self.L.orc_hl_constant(self.h, float(v[0]), float(v[1]))

    def hl_parity(self, v):
        return self.L.orc_hl_parity(self.h, float(v[0]), float(v[1]))

    def hl_host(self):
        return self.L.orc_hl_host(self.h)

    def hl_route(self, route):
        r = np.ascontiguousarray(route, dtype=np.float64).reshape(-1, 2)
        return self.L.orc_hl_route(self.h, r.shape[0], _p(r, f64p))

    def hl_set_target(self, hl, ids):
        """set_target on planner `hl` for the given agents (Simulation.route_set_target)."""
        ids = np.ascontiguousarray(ids, dtype=np.uint64)
        if self.L.orc_hl_set_target(self.h, hl, len(ids), _p(ids, u64p)):
            raise OracleError(1, "unknown agent id")

    def add_agents(self, xy, hl, lp, eyesight):
        xy = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
        ids = np.zeros(xy.shape[0], dtype=np.uint64)
        self._check(self.L.orc_add_agents(self.h, xy.shape[0], _p(xy, f64p), hl, lp, float(eyesight), _p(ids, u64p)))
        return ids

    def remove_agent(self, i):
        self._check(self.L.orc_remove_agent(self.h, int(i)))

    def set_state(self, ids, x, y, vx, vy):
        ids = np.ascontiguousarray(ids, dtype=np.uint64)
        a = [np.ascontiguousarray(v, dtype=np.float64) for v in (x, y, vx, vy)]
        self._check(self.L.orc_set_state(self.h, len(ids), _p(ids, u64p), *[_p(v, f64p) for v in a]))

    def set_preferred_velocity(self, hl, ids, vxy):
        ids = np.ascontiguousarray(ids, dtype=np.uint64)
        vxy = np.ascontiguousarray(vxy, dtype=np.float64).reshape(-1)
        self._check(self.L.orc_set_preferred_velocity(self.h, hl, len(ids), _p(ids, u64p), _p(vxy, f64p)))

    def add_source_sink(self, source, radius_sink, rate, hl, lp, waypoints, loop_forever, eyesight):
        wp = np.ascontiguousarray(waypoints, dtype=np.float64).reshape(-1, 2)
        out = C.c_uint64()
        self._check(self.L.orc_add_source_sink(self.h, source[0], source[1], radius_sink, rate, hl, lp, wp.shape[0],
                                               _p(wp, f64p), 1 if loop_forever else 0, eyesight, C.byref(out)))
        return out.value

    def enable_trace(self, on=True):
        self.L.orc_enable_trace(self.h, 1 if on else 0)

    def set_custom_order(self, ids):
        ids = np.ascontiguousarray(ids, dtype=np.uint64)
        self.L.orc_set_custom_order(self.h, len(ids), _p(ids, u64p))

    def step(self, secs, nanos):
        self._check(self.L.orc_step(self.h, int(secs), int(nanos)))

    def agent_count(self):
        return int(self.L.orc_agent_count(self.h))

    def read_state(self):
        n = self.agent_count()
        ids = np.zeros(n, dtype=np.uint64)
        x, y, vx, vy = (np.zeros(n, dtype=np.float64) for _ in range(4))
        wp = np.zeros(n, dtype=np.uint64)
        self.L.orc_read_agents(self.h, _p(ids, u64p), _p(x, f64p), _p(y, f64p), _p(vx, f64p), _p(vy, f64p),
                               _p(wp, u64p))
        return {"id": ids, "x": x, "y": y, "vx": vx, "vy": vy, "next_waypoint": wp}

    def read_trace(self):
        """Ascending id (the oracle's canonical iteration order)."""
        n = int(self.L.orc_trace_agent_count(self.h))
        t = int(self.L.orc_trace_neighbour_total(self.h))
        ids = np.zeros(n, dtype=np.uint64)
        ti, fx, fy = (np.zeros(n, dtype=np.float64) for _ in range(3))
        off = np.zeros(n + 1, dtype=np.uint64)
        nb = np.zeros(max(t, 1), dtype=np.uint64)
        self.L.orc_read_trace(self.h, _p(ids, u64p), _p(ti, f64p), _p(fx, f64p), _p(fy, f64p), _p(off, u64p),
                              _p(nb, u64p))
        order = np.argsort(ids, kind="stable")
        if not np.array_equal(order, np.arange(n)):
            # re-pack CSR in ascending id
            new_off = np.zeros(n + 1, dtype=np.uint64)
            chunks = []
            for r, k in enumerate(order):
                seg = nb[int(off[k]):int(off[k + 1])]
                chunks.append(seg)
                new_off[r + 1] = new_off[r] + len(seg)
            nb = np.concatenate(chunks) if chunks else nb[:0]
            ids, ti, fx, fy, off = ids[order], ti[order], fx[order], fy[order], new_off
        return {"id": ids, "t_i": ti, "fx": fx, "fy": fy, "nb_offsets": off, "nb_ids": nb[:t]}

    def poll_events(self):
        cap = 1 << 16
        sid = np.zeros(cap, dtype=np.uint64)
        sxy = np.zeros(2 * cap, dtype=np.float64)
        did = np.zeros(cap, dtype=np.uint64)
        ns, nd = C.c_uint64(), C.c_uint64()
        self.L.orc_poll_events(self.h, _p(sid, u64p), _p(sxy, f64p), cap, C.byref(ns), _p(did, u64p), cap,
                               C.byref(nd))
        return sid[: ns.value].copy(), sxy[: 2 * ns.value].reshape(-1, 2).copy(), did[: nd.value].copy()

    # SpatialIndex surface
    def index_add_or_update(self, i, p):
        if self.L.orc_index_add_or_update(self.h, int(i), float(p[0]), float(p[1])):
            raise OracleError(1, "Index out of bounds")

    def index_remove(self, i):
        self.L.orc_index_remove(self.h, int(i))

    def cell_of(self, xy):
        xy = np.asarray(xy, dtype=np.float64).reshape(-1, 2)
        return np.array([self.L.orc_cell_of(self.h, float(p[0]), float(p[1])) for p in xy], dtype=np.int64)

    def query_radius(self, radius, p, cap=1 << 16):
        out = np.zeros(cap, dtype=np.uint64)
        n = self.L.orc_query_radius(self.h, float(radius), float(p[0]), float(p[1]), _p(out, u64p), cap)
        return out[: int(n)].copy()

    def query_knn(self, n, p, cap=1 << 16):
        out = np.zeros(cap, dtype=np.uint64)
        m = self.L.orc_query_knn(self.h, int(n), float(p[0]), float(p[1]), _p(out, u64p), cap)
        if m == 2**64 - 1:
            raise OracleError(1, self.L.orc_last_error(self.h).decode())
        return out[: int(m)].copy()


def flat_step(scene, x, y, vx, vy, dt, threads, want_t_i=False):
    """oracle/flat_parallel.cpp: one deferred step of a single-group parity / Zanlungo crowd on flat arrays with
    `threads` threads (NOT the reference: a strong CPU implementation for comparison).  Arrays are updated in place."""
    assert scene.hl[0] == "parity" and scene.lp[0] == "zanlungo"
    zan = np.ascontiguousarray(scene.lp[1:], dtype=np.float64)
    t_i = np.zeros(len(x), dtype=np.float64) if want_t_i else None
    rc = lib().orc_flat_step(len(x), _p(x, f64p), _p(y, f64p), _p(vx, f64p), _p(vy, f64p), scene.width, scene.height,
                             scene.cell, scene.offset[0], scene.offset[1], _p(zan, f64p), scene.eyesight,
                             scene.hl[1][0], scene.hl[1][1], int(dt[0]), int(dt[1]), int(threads), _p(t_i, f64p))
    if rc:
        raise OracleError(rc, "Index out of bounds")
    return t_i


def flat_step_trace(scene, x, y, vx, vy, dt, threads, ids=None):
    """flat_step plus the per-agent trace (t_i, neighbour-list length, summed force) in array = id order; the
    benchmark-size parity tests compare the CUDA path against it (bit-identical to the oracle's deferred mode,
    tests/test_oracle_reference.py).  ids: the agents' ids (strictly ascending) when the arrays are a window cut out of
    a larger crowd; None = array index."""
    assert scene.hl[0] == "parity" and scene.lp[0] == "zanlungo"
    zan = np.ascontiguousarray(scene.lp[1:], dtype=np.float64)
    n = len(x)
    t_i, fx, fy = (np.zeros(n, dtype=np.float64) for _ in range(3))
    nbc = np.zeros(n, dtype=np.uint32)
    rc = lib().orc_flat_step_trace(n, _p(x, f64p), _p(y, f64p), _p(vx, f64p), _p(vy, f64p), scene.width, scene.height,
                                   scene.cell, scene.offset[0], scene.offset[1], _p(zan, f64p), scene.eyesight,
                                   scene.hl[1][0], scene.hl[1][1], int(dt[0]), int(dt[1]), int(threads), _p(t_i, f64p),
                                   nbc.ctypes.data_as(C.POINTER(C.c_uint32)), _p(fx, f64p), _p(fy, f64p),
                                   _p(None if ids is None else np.ascontiguousarray(ids, dtype=np.uint64), u64p))
    if rc:
        raise OracleError(rc, "Index out of bounds" if rc == 1 else "ids must be strictly ascending")
    return {"t_i": t_i, "nbc": nbc, "fx": fx, "fy": fy}


def ttc(agent_radius, rel_vel, rel_pos) -> float:
    return lib().orc_ttc(float(agent_radius), float(rel_vel[0]), float(rel_vel[1]), float(rel_pos[0]),
                         float(rel_pos[1]))
