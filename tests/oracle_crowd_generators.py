"""The CPU oracle with keyed PoissonCrowd and host-count generators (tests/oracle_crowd_generators.cpp on top of
oracle/), plus a numpy restatement of the keyed draw.  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import math
import os
import subprocess

import numpy as np

import oracle_ffi as O

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_crowd_generators.cpp")
LIB = os.path.join(O.ORACLE_DIR, "_build", "liboracle_crowd_generators.so")
DEPS = [SRC] + [os.path.join(O.ORACLE_DIR, f) for f in ("oracle_capi.cpp", "flat_parallel.cpp", "crowdsim_oracle.hpp")]

MONOTONIC, POISSON, HOST = 0, 1, 2
M64 = (1 << 64) - 1

_lib = None


def lib() -> C.CDLL:
    """liboracle.so's whole orc_* surface (same signatures) plus the generator calls of oracle_crowd_generators.cpp."""
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
        L.orc_add_source_sink_gen.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_int, C.c_double,
                                              C.c_uint64, C.c_int, C.c_int, C.c_uint64, O.f64p, C.c_int, C.c_double,
                                              O.u64p]
        L.orc_remove_source_sink_gen.argtypes = [C.c_void_p, C.c_uint64]
        L.orc_set_spawn_counts.argtypes = [C.c_void_p, C.c_uint64, O.u64p, O.u64p]
        L.orc_step_gen.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32]
        L.orc_gen_steps.restype = C.c_uint64
        L.orc_gen_steps.argtypes = [C.c_void_p]
        L.orc_gen_release.argtypes = [C.c_void_p]
        L.orc_poisson_wants.argtypes = [C.c_double, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint64, C.c_uint64]
        L.orc_philox4x64_10_w0.restype = C.c_uint64
        L.orc_philox4x64_10_w0.argtypes = [C.c_uint64] * 3
        _lib = L
    return _lib


class GenOracle(O.OracleSim):
    """OracleSim whose source sinks take a generator kind, and whose step is orc_step_gen."""

    def __init__(self, width, height, cell, offset, index_mode=O.DEFERRED, iter_order=O.ASCENDING_ID, canonical=True):
        self.L = lib()
        self.h = C.c_void_p(self.L.orc_sim_create(width, height, cell, offset[0], offset[1], index_mode, iter_order,
                                                  1 if canonical else 0))

    def __del__(self):
        try:
            self.L.orc_gen_release(self.h)
        except Exception:
            pass
        super().__del__()

    def add_source_sink_gen(self, source, radius_sink, kind, rate, seed, hl, lp, waypoints, loop_forever, eyesight):
        wp = np.ascontiguousarray(waypoints, dtype=np.float64).reshape(-1, 2)
        out = C.c_uint64()
        self._check(self.L.orc_add_source_sink_gen(self.h, source[0], source[1], radius_sink, kind, rate, seed, hl, lp,
                                                   wp.shape[0], O._p(wp, O.f64p), 1 if loop_forever else 0, eyesight,
                                                   C.byref(out)))
        return out.value

    def remove_source_sink(self, sid):
        self.L.orc_remove_source_sink_gen(self.h, int(sid))

    def set_spawn_counts(self, ids, counts):
        ids = np.ascontiguousarray(ids, dtype=np.uint64)
        counts = np.ascontiguousarray(counts, dtype=np.uint64)
        if self.L.orc_set_spawn_counts(self.h, len(ids), O._p(ids, O.u64p), O._p(counts, O.u64p)):
            raise O.OracleError(1, "not a host-count source sink")

    def step(self, secs, nanos):
        self._check(self.L.orc_step_gen(self.h, int(secs), int(nanos)))

    def steps(self):
        return int(self.L.orc_gen_steps(self.h))


# ---- the keyed draw, restated with numpy's Philox (which increments its counter before the first block) ----------
def numpy_word0(seed: int, k: int, sid: int) -> int:
    """Word 0 of Philox4x64-10 with counter (k + 1, sid, 0, 0) and key (seed, 0), through numpy.random.Philox."""
    bg = np.random.Philox(key=np.array([seed, 0], dtype=np.uint64), counter=np.array([k, sid, 0, 0], dtype=np.uint64))
    return int(bg.random_raw())


def python_word0(seed: int, k: int, sid: int) -> int:
    """The same word, restated in plain Python (Salmon et al., SC'11)."""
    c = [(k + 1) & M64, sid, 0, 0]
    key = [seed, 0]
    for _ in range(10):
        p0 = 0xD2E7470EE14C6C93 * c[0]
        p1 = 0xCA5A826395121157 * c[2]
        c = [(p1 >> 64) ^ c[1] ^ key[0], p1 & M64, (p0 >> 64) ^ c[3] ^ key[1], p0 & M64]
        key = [(key[0] + 0x9E3779B97F4A7C15) & M64, (key[1] + 0xBB67AE8584CAA73B) & M64]
    return c[0]


def threshold(lam: float) -> int:
    """ceil(exp(-lambda) * 2^53) (Python's math.exp is the C library's exp)."""
    return math.ceil(math.ldexp(math.exp(-lam), 53))


def poisson_wants(rate: float, seed: int, dt: float, k: int, sid: int) -> bool:
    return (numpy_word0(seed, k, sid) >> 11) >= threshold(dt * rate)
