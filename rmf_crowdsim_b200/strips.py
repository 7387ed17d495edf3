"""Spatial strips over several GPUs (SURVEY.md section 8e): host-side plumbing over the C ABI.

Strips are whole cell columns in x (the LocationHash2D cell index is x-major, location_hash_2d.rs:59).
`StripSimulation` is one rank of a `torch.distributed` job (one process per GPU, NCCL halo exchange inside
librcs.so); `LocalStripGroup` drives all ranks from one process with peer copies, which is how the strip
kernels are tested on a single GPU.  Both give results that are bit-identical to a single handle.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional, Tuple

import numpy as np

from . import _native as N
from . import sim as S


def strip_columns(sim: S.Simulation, rank: int, world: int) -> Tuple[int, int]:
    """Cell columns [c0, c1) owned by `rank` (rcs_dist_strip)."""
    c0, c1 = C.c_uint64(), C.c_uint64()
    N.check(sim._h, sim._lib.rcs_dist_strip(sim._h, rank, world, C.byref(c0), C.byref(c1)))
    return c0.value, c1.value


def column_of(x: np.ndarray, offset_x: float, cell: float) -> np.ndarray:
    """x_idx of LocationHash2D::location_to_index (location_hash_2d.rs:56): IEEE sub, IEEE div, then the
    saturating `as usize` (truncation; negatives and NaN -> 0)."""
    q = (np.asarray(x, dtype=np.float64) - offset_x) / cell
    q = np.where(q > 0, q, 0.0)
    return np.minimum(q, 1.8e19).astype(np.uint64)


def owned_mask(x: np.ndarray, offset_x: float, cell: float, c0: int, c1: int) -> np.ndarray:
    cx = column_of(x, offset_x, cell)
    return (cx >= np.uint64(c0)) & (cx < np.uint64(c1))


def add_agents_with_ids(sim: S.Simulation, ids: np.ndarray, xy: np.ndarray, vxy: Optional[np.ndarray], hl, lp,
                        eyesight: float) -> None:
    """rcs_dist_add_agents: add_agents with caller-supplied global ids and initial velocities."""
    ids = np.ascontiguousarray(ids, dtype=np.uint64)
    xy = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
    vp = None
    if vxy is not None:
        vxy = np.ascontiguousarray(vxy, dtype=np.float64).reshape(-1, 2)
        vp = vxy.ctypes.data_as(N.c_f64p)
    N.check(sim._h, sim._lib.rcs_dist_add_agents(sim._h, len(ids), ids.ctypes.data_as(N.c_u64p),
                                                 xy.ctypes.data_as(N.c_f64p), vp, sim._hl(hl), sim._lp(lp),
                                                 float(eyesight)))


class HostPlan(S.HighLevelPlanner):
    """A HighLevelPlanner evaluated by the caller: its results are uploaded with set_preferred_velocity."""


def _planners(scene):
    kind, v = scene.hl
    hl = HostPlan() if kind == "host" else {"parity": S.ParityVelocityPlan,
                                            "constant": S.ConstantVelocityPlan}[kind](v)
    lp = S.NoLocalPlan() if scene.lp[0] == "none" else S.Zanlungo(*scene.lp[1:])
    return hl, lp


def torch_peer_gather(dist, torch):
    """`peer_gather` for StripSimulation over a torch.distributed process group: every rank's 64-byte CUDA IPC handle
    to every rank (only the two neighbours' are used)."""
    def gather(handle: bytes):
        dev = "cuda" if dist.get_backend() == "nccl" else "cpu"
        mine = torch.tensor(list(handle), dtype=torch.uint8, device=dev)
        parts = [torch.zeros_like(mine) for _ in range(dist.get_world_size())]
        dist.all_gather(parts, mine)
        return [bytes(p.cpu().tolist()) for p in parts]
    return gather


def neighbour_handles(handles, rank: int, world: int):
    """(left, right) of `rank` out of the all-gathered handles; None where the strip has no neighbour."""
    assert len(handles) == world and all(len(hd) == 64 for hd in handles)
    return tuple(handles[r] if 0 <= r < world else None for r in (rank - 1, rank + 1))


class StripSimulation(S.Simulation):
    """One rank of a strip-partitioned simulation (one process per GPU).  `nccl_id` is the 128-byte id made by
    `nccl_unique_id()` on rank 0 and distributed by the caller (e.g. torch.distributed.broadcast).
    `peer_gather` (e.g. `torch_peer_gather(dist, torch)`) switches the halo exchange from ncclSend / ncclRecv to the
    peer-store transport (rcs_dist_peer_export / rcs_dist_peer_connect): every rank must pass it, and every rank must
    have its own GPU."""

    def __init__(self, spatial_index: S.LocationHash2D, rank: int, world: int, nccl_id: Optional[bytes],
                 halo_capacity: int = 0, boundaries=None, peer_gather=None):
        super().__init__(spatial_index)
        self.rank, self.world = rank, world
        if boundaries is not None:  # world + 1 cell-column boundaries instead of the equal split (every rank alike)
            b = np.ascontiguousarray(boundaries, dtype=np.uint64)
            assert len(b) == world + 1
            N.check(self._h, self._lib.rcs_dist_set_boundaries(self._h, world, b.ctypes.data_as(N.c_u64p)))
        buf = None
        if world > 1:
            assert nccl_id is not None and len(nccl_id) == 128
            buf = (C.c_uint8 * 128).from_buffer_copy(nccl_id)
        N.check(self._h, self._lib.rcs_dist_init(self._h, rank, world, buf, int(halo_capacity)))
        self.c0, self.c1 = strip_columns(self, rank, world)
        self.transport = "nccl"
        if world > 1 and peer_gather is not None:
            # every rank tries; the transport is used only if every rank could map both neighbours (the verdicts travel
            # through the same gather), otherwise every rank goes back to ncclSend / ncclRecv
            mine = (C.c_uint8 * 64)()
            ok = self._lib.rcs_dist_peer_export(self._h, mine) == N.RCS_OK
            handles = peer_gather(bytes(mine) if ok else bytes(64))
            if ok and all(any(hd) for hd in handles):
                nb = [None if hd is None else (C.c_uint8 * 64).from_buffer_copy(hd)
                      for hd in neighbour_handles(handles, rank, world)]
                ok = self._lib.rcs_dist_peer_connect(self._h, nb[0], nb[1]) == N.RCS_OK
            else:
                ok = False
            if os.environ.get("RCS_PEER_FAIL_RANK") == str(rank):  # test hook: this rank reports a failed mapping
                ok = False
            self.peer_error = "" if ok else (self._lib.rcs_last_error(self._h) or b"").decode()
            verdicts = peer_gather(bytes([1 if ok else 0] * 64))
            if all(v[0] == 1 for v in verdicts):
                self.transport = "peer stores"
            else:
                N.check(self._h, self._lib.rcs_dist_peer_disable(self._h))

    def add_scene_agents(self, scene, ids: Optional[np.ndarray] = None, xy=None, vxy=None) -> int:
        """Adds the agents of `scene` (or of the given id / xy / vxy arrays) that fall into this strip."""
        hl, lp = _planners(scene)
        self._scene_planners = (hl, lp)
        if xy is None:
            xy, vxy, ids = scene.xy, scene.vxy, np.arange(scene.n, dtype=np.uint64)
        m = owned_mask(xy[:, 0], scene.offset[0], scene.cell, self.c0, self.c1)
        add_agents_with_ids(self, ids[m], xy[m], None if vxy is None else vxy[m], hl, lp, scene.eyesight)
        if len(ids):  # source sinks number their spawns after every rank's agents
            N.check(self._h, self._lib.rcs_dist_reserve_ids(self._h, int(np.max(ids)) + 1))
        return int(m.sum())


def nccl_unique_id() -> bytes:
    buf = (C.c_uint8 * 128)()
    lib = N.load()
    rc = lib.rcs_nccl_unique_id(buf)
    if rc != N.RCS_OK:
        raise N.RcsError(rc, (lib.rcs_last_error(None) or b"").decode())
    return bytes(buf)


class LocalStripGroup:
    """All ranks of a strip-partitioned simulation inside one process (single-process transport)."""

    def __init__(self, scene, world: int, devices: Optional[List[int]] = None, capacity: Optional[int] = None,
                 halo_capacity: int = 0, boundaries=None):
        self.scene, self.world = scene, world
        devices = devices or [0] * world
        cap = capacity or max(scene.n, 64)
        self.sims: List[S.Simulation] = []
        for r in range(world):
            idx = S.LocationHash2D(scene.width, scene.height, scene.cell, scene.offset, capacity=cap,
                                   device=devices[r])
            self.sims.append(S.Simulation(idx))
            if boundaries is not None:
                b = np.ascontiguousarray(boundaries, dtype=np.uint64)
                N.check(self.sims[-1]._h, self.sims[-1]._lib.rcs_dist_set_boundaries(self.sims[-1]._h, world,
                                                                                     b.ctypes.data_as(N.c_u64p)))
        self._lib = self.sims[0]._lib
        self._handles = (C.c_void_p * world)(*[s._h for s in self.sims])
        rc = self._lib.rcs_dist_init_local(self._handles, world, int(halo_capacity))
        if rc != N.RCS_OK:
            self._raise(rc)
        ids = np.arange(scene.n, dtype=np.uint64)
        self.counts = []
        for r, sm in enumerate(self.sims):
            c0, c1 = strip_columns(sm, r, world)
            m = owned_mask(scene.xy[:, 0], scene.offset[0], scene.cell, c0, c1)
            hl, lp = _planners(scene)
            sm._scene_planners = (hl, lp)
            add_agents_with_ids(sm, ids[m], scene.xy[m], scene.vxy[m], hl, lp, scene.eyesight)
            N.check(sm._h, self._lib.rcs_dist_reserve_ids(sm._h, scene.n))  # spawned ids follow the scene's agents
            self.counts.append(int(m.sum()))
        assert sum(self.counts) == scene.n

    def _raise(self, rc: int):
        for sm in self.sims:
            msg = (self._lib.rcs_last_error(sm._h) or b"").decode()
            if msg:
                raise N.RcsError(rc, msg)
        raise N.RcsError(rc, f"rcs error {rc}")

    def step(self, dur: S.Duration, no_commit: bool = False, sync: bool = True) -> None:
        flags = N.RCS_STEP_NO_COMMIT if no_commit else N.RCS_STEP_DEFAULT
        for sm in self.sims:  # every rank's host generators are called; the rank that owns a source decides
            sm._run_host_generators(dur)
        rc = self._lib.rcs_dist_step_local(self._handles, self.world, int(dur.secs), int(dur.nanos), flags)
        if rc != N.RCS_OK:
            self._raise(rc)
        if sync:
            for sm in self.sims:
                sm.sync()

    def read_state(self) -> Dict[str, np.ndarray]:
        """All ranks' agents merged in ascending id."""
        parts = [sm.read_state() for sm in self.sims]
        out = {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
        order = np.argsort(out["id"], kind="stable")
        return {k: v[order] for k, v in out.items()}

    def read_trace(self) -> Dict[str, np.ndarray]:
        """All ranks' traces (owned agents only) merged in ascending id."""
        parts = [sm.read_trace() for sm in self.sims]
        ids = np.concatenate([p["id"] for p in parts])
        order = np.argsort(ids, kind="stable")
        rank_of = np.concatenate([np.full(len(p["id"]), r) for r, p in enumerate(parts)])
        local = np.concatenate([np.arange(len(p["id"])) for p in parts])
        chunks, off = [], np.zeros(len(ids) + 1, dtype=np.uint64)
        for k, g in enumerate(order):
            p = parts[rank_of[g]]
            a, b = int(p["nb_offsets"][local[g]]), int(p["nb_offsets"][local[g] + 1])
            chunks.append(p["nb_ids"][a:b])
            off[k + 1] = off[k] + np.uint64(b - a)
        cat = lambda key: np.concatenate([p[key] for p in parts])[order]  # noqa: E731
        return {"id": ids[order], "t_i": cat("t_i"), "fx": cat("fx"), "fy": cat("fy"), "nb_offsets": off,
                "nb_ids": np.concatenate(chunks) if chunks else np.zeros(0, dtype=np.uint64)}

    def set_trace(self, on: bool) -> None:
        for sm in self.sims:
            sm.set_trace(on)

    def agent_counts(self) -> List[int]:
        return [sm.agent_count() for sm in self.sims]

    def add_source_sink(self, make_source_sink) -> int:
        """Every rank holds every source sink (same calls in the same order); the rank that owns the source's cell
        column spawns for it.  `make_source_sink()` returns a fresh SourceSink (planner objects are per handle)."""
        ids = [sm.add_source_sink(make_source_sink()) for sm in self.sims]
        assert len(set(ids)) == 1
        return ids[0]

    def add_event_listener(self, listener) -> None:
        for sm in self.sims:
            sm.add_event_listener(listener)

    def dispatch_events(self) -> None:
        for sm in self.sims:
            sm._dispatch_events()
