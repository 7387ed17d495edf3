"""ctypes binding of the C ABI in include/rcs.h.

This is the only way Python reaches the compute path.  There is no CPU fallback: if the CUDA
library is missing or no device is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

from . import _build

c_u8p = C.POINTER(C.c_uint8)
c_u32p = C.POINTER(C.c_uint32)
c_u64p = C.POINTER(C.c_uint64)
c_i64p = C.POINTER(C.c_int64)
c_f64p = C.POINTER(C.c_double)
c_f32p = C.POINTER(C.c_float)

RCS_OK = 0
RCS_ERR_OUT_OF_BOUNDS = 1
RCS_ERR_SPAWN = 2
RCS_ERR_CUDA = 3
RCS_ERR_NCCL = 4
RCS_ERR_CAPACITY = 5
RCS_ERR_ARG = 6
RCS_ERR_NO_DEVICE = 7
RCS_ERR_HALO = 8

RCS_ORDER_STORAGE = 0
RCS_ORDER_ID = 1
RCS_STEP_DEFAULT = 0
RCS_STEP_NO_COMMIT = 1
RCS_NUM_EVENTS = 64
RCS_OPT_STEP_KERNEL = 1
RCS_OPT_BIN_AHEAD = 2
RCS_OPT_GRAPHS = 3
RCS_OPT_PDL = 4


class SimDesc(C.Structure):
    _fields_ = [
        ("width", C.c_double),
        ("height", C.c_double),
        ("cell_size", C.c_double),
        ("offset_x", C.c_double),
        ("offset_y", C.c_double),
        ("capacity", C.c_uint64),
        ("device", C.c_int32),
        ("flags", C.c_uint32),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("n_agents", C.c_uint64),
        ("oob_count", C.c_uint64),
        ("first_oob_id", C.c_uint64),
        ("nonfinite_count", C.c_uint64),
        ("finite_tti_count", C.c_uint64),
        ("neighbour_total", C.c_uint64),
        ("candidate_total", C.c_uint64),
        ("spawned", C.c_uint64),
        ("destroyed", C.c_uint64),
        ("steps", C.c_uint64),
    ]


class SourceSinkDesc(C.Structure):
    _fields_ = [
        ("source_x", C.c_double),
        ("source_y", C.c_double),
        ("radius_sink", C.c_double),
        ("monotonic_rate", C.c_double),
        ("hl", C.c_uint32),
        ("lp", C.c_uint32),
        ("n_waypoints", C.c_uint64),
        ("waypoints_xy", c_f64p),
        ("loop_forever", C.c_int32),
        ("agent_eyesight_range", C.c_double),
    ]


# name -> (restype, argtypes); every symbol include/rcs.h declares
SIGNATURES = {
    "rcs_abi_version": (C.c_uint32, []),
    "rcs_sim_create": (C.c_int, [C.POINTER(SimDesc), C.POINTER(C.c_void_p)]),
    "rcs_sim_destroy": (None, [C.c_void_p]),
    "rcs_last_error": (C.c_char_p, [C.c_void_p]),
    "rcs_lp_none": (C.c_int, [C.c_void_p, c_u32p]),
    "rcs_lp_zanlungo": (C.c_int, [C.c_void_p] + [C.c_double] * 6 + [c_u32p]),
    "rcs_hl_constant": (C.c_int, [C.c_void_p, C.c_double, C.c_double, c_u32p]),
    "rcs_hl_parity": (C.c_int, [C.c_void_p, C.c_double, C.c_double, c_u32p]),
    "rcs_hl_host": (C.c_int, [C.c_void_p, c_u32p]),
    "rcs_hl_route": (C.c_int, [C.c_void_p, C.c_uint64, c_f64p, c_u32p]),
    "rcs_hl_route_set_target": (C.c_int, [C.c_void_p, C.c_uint64, c_u64p]),
    "rcs_hl_none": (C.c_int, [C.c_void_p, c_u32p]),
    "rcs_add_agents": (C.c_int, [C.c_void_p, C.c_uint64, c_f64p, C.c_uint32, C.c_uint32, C.c_double, c_u64p]),
    "rcs_remove_agents": (C.c_int, [C.c_void_p, C.c_uint64, c_u64p]),
    "rcs_set_state": (C.c_int, [C.c_void_p, C.c_uint64, c_u64p, c_f64p, c_f64p, c_f64p, c_f64p]),
    "rcs_set_preferred_velocity": (C.c_int, [C.c_void_p, C.c_uint64, c_u64p, c_f64p]),
    "rcs_read_agents": (
        C.c_int,
        [C.c_void_p, C.c_uint32, C.c_uint64, c_u64p, c_f64p, c_f64p, c_f64p, c_f64p, c_u32p, c_u64p],
    ),
    "rcs_agent_count": (C.c_int, [C.c_void_p, c_u64p]),
    "rcs_read_agents_async": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64, c_u64p, c_f64p, c_f64p, c_f64p, c_f64p, c_u64p]),
    "rcs_read_wait": (C.c_int, [C.c_void_p]),
    "rcs_step": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32]),
    "rcs_step_async": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32]),
    "rcs_sync": (C.c_int, [C.c_void_p]),
    "rcs_step_stats": (C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    "rcs_step_in_loop": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, c_u64p, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint32)]),
    "rcs_poll_events": (
        C.c_int,
        [C.c_void_p, C.c_uint64, c_u64p, c_f64p, c_u64p, C.c_uint64, c_u64p, c_u64p],
    ),
    "rcs_add_source_sink": (C.c_int, [C.c_void_p, C.POINTER(SourceSinkDesc), c_u64p]),
    "rcs_remove_source_sink": (C.c_int, [C.c_void_p, C.c_uint64]),
    "rcs_cell_of": (C.c_int, [C.c_void_p, C.c_uint64, c_f64p, c_i64p]),
    "rcs_index_add_or_update": (C.c_int, [C.c_void_p, C.c_uint64, c_u64p, c_f64p]),
    "rcs_index_remove": (C.c_int, [C.c_void_p, C.c_uint64, c_u64p]),
    "rcs_query_radius": (C.c_int, [C.c_void_p, C.c_uint64, c_f64p, c_f64p, c_u64p, c_u64p, C.c_uint64]),
    "rcs_query_knn": (C.c_int, [C.c_void_p, C.c_uint64, c_f64p, C.c_uint64, c_u64p, c_u64p]),
    "rcs_set_trace": (C.c_int, [C.c_void_p, C.c_int32]),
    "rcs_trace_sizes": (C.c_int, [C.c_void_p, c_u64p, c_u64p]),
    "rcs_read_trace": (C.c_int, [C.c_void_p, c_u64p, c_f64p, c_f64p, c_f64p, c_u64p, c_u64p]),
    "rcs_set_option": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64]),
    "rcs_event_record": (C.c_int, [C.c_void_p, C.c_uint32]),
    "rcs_event_elapsed_ms": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, c_f32p]),
    "rcs_host_alloc": (C.c_int, [C.c_uint64, C.POINTER(C.c_void_p)]),
    "rcs_host_free": (C.c_int, [C.c_void_p]),
    "rcs_flush_l2": (C.c_int, [C.c_void_p, C.c_uint64]),
    "rcs_kernel_timing": (C.c_int, [C.c_void_p, C.c_int32]),
    "rcs_kernel_time_ms": (C.c_int, [C.c_void_p, c_f64p, c_u64p]),
    "rcs_launch_count": (C.c_int, [C.c_void_p, c_u64p]),
    "rcs_graph_stats": (C.c_int, [C.c_void_p, c_u64p, c_u64p]),
    "rcs_fp64_peak": (C.c_int, [C.c_int32, c_f64p, c_f64p]),
    "rcs_nccl_unique_id": (C.c_int, [c_u8p]),
    "rcs_dist_init": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, c_u8p, C.c_uint64]),
    "rcs_dist_init_local": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_uint64]),
    "rcs_dist_step_local": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_uint64, C.c_uint32, C.c_uint32]),
    "rcs_dist_strip": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, c_u64p, c_u64p]),
    "rcs_dist_set_boundaries": (C.c_int, [C.c_void_p, C.c_int32, c_u64p]),
    "rcs_dist_reserve_ids": (C.c_int, [C.c_void_p, C.c_uint64]),
    "rcs_dist_peer_export": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint8)]),
    "rcs_dist_peer_connect": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_uint8)]),
    "rcs_dist_peer_disable": (C.c_int, [C.c_void_p]),
    "rcs_dist_add_agents": (
        C.c_int,
        [C.c_void_p, C.c_uint64, c_u64p, c_f64p, c_f64p, C.c_uint32, C.c_uint32, C.c_double],
    ),
}

_lib = None


def library_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load librcs.so (building it in-tree first if it is absent or stale and nvcc is available)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if build_if_missing and _build.needs_build():
        try:
            _build.build()
        except Exception as exc:  # stale-but-present library is still usable
            if not os.path.exists(path):
                raise RuntimeError(
                    "rmf_crowdsim_b200: the CUDA extension librcs.so is missing and could not be built "
                    f"({exc}).  There is no CPU fallback."
                ) from exc
    if not os.path.exists(path):
        raise RuntimeError(
            "rmf_crowdsim_b200: the CUDA extension librcs.so is missing "
            "(run `python -c 'import __graft_entry__ as g; g.build()'`).  There is no CPU fallback."
        )
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class RcsError(RuntimeError):
    """A non-zero status from the C ABI; .code is the RCS_ERR_* value, str() the library's message
    (the reference's literal strings where it has one, e.g. "Index out of bounds")."""

    def __init__(self, code: int, message: str):
        super().__init__(message)
        self.code = code
        self.message = message


def check(handle, rc: int) -> None:
    if rc != RCS_OK:
        msg = load().rcs_last_error(handle)
        raise RcsError(rc, (msg or b"").decode() or f"rcs error {rc}")
