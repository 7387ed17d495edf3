"""The CPU oracle with RouteTablePlan (tests/oracle_route_table.cpp on top of oracle/).  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import oracle_ffi as O

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_route_table.cpp")
LIB = os.path.join(O.ORACLE_DIR, "_build", "liboracle_route_table.so")
DEPS = [SRC] + [os.path.join(O.ORACLE_DIR, f) for f in ("oracle_capi.cpp", "flat_parallel.cpp", "crowdsim_oracle.hpp")]

_lib = None


def lib() -> C.CDLL:
    """liboracle.so's whole orc_* surface (same signatures) plus orc_hl_route_table / orc_hl_route_table_set_target."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in DEPS):
            os.makedirs(os.path.dirname(LIB), exist_ok=True)
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall",
                            "-pthread", "-shared", "-o", LIB, SRC, os.path.join(O.ORACLE_DIR, "flat_parallel.cpp")],
                           check=True)
        L = C.CDLL(LIB)
        base = O.lib()
        for name, fn in vars(base).items():  # the signatures oracle_ffi declared
            if name.startswith("orc_"):
                f = getattr(L, name)
                f.restype, f.argtypes = fn.restype, fn.argtypes
        L.orc_hl_route_table.argtypes = [C.c_void_p, C.c_uint64, O.f64p, O.u64p, O.f64p]
        L.orc_hl_route_table_set_target.argtypes = [C.c_void_p, C.c_int, C.c_uint64, O.u64p, O.f64p]
        _lib = L
    return _lib


class RouteTableOracle(O.OracleSim):
    """OracleSim with hl_route_table / hl_route_table_set_target."""

    def __init__(self, width, height, cell, offset, index_mode=O.DEFERRED, iter_order=O.ASCENDING_ID, canonical=True):
        self.L = lib()
        self.h = C.c_void_p(self.L.orc_sim_create(width, height, cell, offset[0], offset[1], index_mode, iter_order,
                                                  1 if canonical else 0))

    def hl_route_table(self, routes):
        """routes: {target: polyline}, in insertion order (RouteTablePlan's argument)."""
        legs = list(routes.items())
        t = np.ascontiguousarray([tp for tp, _ in legs], dtype=np.float64).reshape(-1)
        n = np.ascontiguousarray([len(r) for _, r in legs], dtype=np.uint64)
        xy = np.ascontiguousarray([p for _, r in legs for p in r], dtype=np.float64).reshape(-1)
        return self.L.orc_hl_route_table(self.h, len(legs), O._p(t, O.f64p), O._p(n, O.u64p), O._p(xy, O.f64p))

    def hl_route_table_set_target(self, hl, ids, targets):
        ids = np.ascontiguousarray(ids, dtype=np.uint64)
        t = np.ascontiguousarray(targets, dtype=np.float64).reshape(-1)
        rc = self.L.orc_hl_route_table_set_target(self.h, hl, len(ids), O._p(ids, O.u64p), O._p(t, O.f64p))
        if rc:
            raise O.OracleError(rc, "unknown agent id" if rc == 1 else self.L.orc_last_error(self.h).decode())
