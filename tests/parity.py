"""Shared helpers of the parity tests: build oracle and CUDA simulations from one Scene and
compare them step by step.  Tolerances are the ones BASELINE.json's north_star states:
cell assignments and neighbour sets bit-exact, t_i bit-exact (only IEEE +,-,*,/,sqrt feed it),
forces / velocities <= 1e-9 relative (CUDA's exp/asin/sin differ from glibc's by <= 2 ulp)."""
from __future__ import annotations

import math

import numpy as np

import oracle_ffi as O
from rmf_crowdsim_b200 import scenes as SC

REL_TOL = 1e-9
INF, NAN = float("inf"), float("nan")


def _nx(x, k):
    """k steps of nextafter from x (toward +inf for k > 0)."""
    for _ in range(abs(k)):
        x = math.nextafter(x, INF if k > 0 else -INF)
    return x


def radius_threshold(r):
    """Smallest double T with sqrt(T) >= r (r > 0 finite): sqrt(d2) < r <=> d2 < T."""
    t = r * r
    while math.sqrt(t) >= r:
        t = math.nextafter(t, 0.0)
    while math.sqrt(t) < r:
        t = math.nextafter(t, INF)
    return t


def threshold_points(r, x, diagonal, m_max=400):
    """A probe at (x, -dy/2) and neighbours near (x + dx, +dy/2) -- along the x axis (dy ~ 0.05 r) or the diagonal --
    at which the computed fl(dx*dx + dy*dy) (dx = fl(qx - px), dy = fl(qy - py)) is T(r) - 1 ulp, T(r) and T(r) + 1 ulp;
    found by stepping qy (and, where that skips a target, qx) with nextafter.  y stays near 0, where the steps are
    finer than one unit of T."""
    t = radius_threshold(r)
    ang = math.pi / 4 if diagonal else 0.05
    p = np.array([x, -0.5 * r * math.sin(ang)])
    targets = (math.nextafter(t, 0.0), t, math.nextafter(t, INF))
    for k in range(64):
        qx = _nx(x + r * math.cos(ang), (k + 1) // 2 * (-1) ** k)
        y0 = np.float64(p[1] + math.sqrt(t - (qx - p[0]) ** 2))  # aim at T with the dx the rounding of qx left
        ys = (y0.view(np.int64) + np.arange(-m_max, m_max + 1)).view(np.float64)  # consecutive doubles (y0 > 0)
        dx, dy = qx - p[0], ys - p[1]
        d2 = dx * dx + dy * dy
        hits = [np.nonzero(d2 == tg)[0] for tg in targets]
        if all(len(h) for h in hits):
            return p, [np.array([qx, ys[h[len(h) // 2]]]) for h in hits]
    raise AssertionError((r, x, diagonal))


PROBE_RADIUS = 0.4  # the spawn probe's hard-coded radius (lib.rs:214)
CELLS = [(0.3, (0.0, 0.0)), (0.7, (-7.7, 13.1)), (1.1, (0.0, 0.0)), (2.6, (-7.7, 13.1))]
SINK_RADII = [0.3, 0.6, 1.1, 0.5, 2.0]  # r*r inexact, then exact


def probe_threshold_configs(x0=5.0, spacing=11.0):
    """(source, agent, blocked): an agent at T(0.4) - 1 ulp, T and T + 1 ulp from a source (the computed fl(dx*dx +
    dy*dy)), along an axis and a diagonal; only T - 1 ulp blocks.  Sources `spacing` apart along y ~ 0."""
    out, x = [], x0
    for diagonal in (False, True):
        for which in range(3):
            p, qs = threshold_points(PROBE_RADIUS, x, diagonal)
            out.append((p, qs[which], which == 0))
            x += spacing
    return out


PROBE_EDGE_ULPS = [(0, 0), (1, 0), (-1, 0), (0, 1), (0, -1), (1, 1), (-1, -1), (2, -2), (-2, 2), (4, -1), (-4, 1),
                   (8, 8), (-8, -8), (3, -5), (-3, 5), (6, 0)]


def probe_edge_configs(cell, off, k0=3, stride=6, row=5):
    """(source, agent) pairs at the spawn probe's stencil edges: source +- 0.4 within a few ulps of the cell edge
    e = k*cell + off (so that the stencil's last column ends there) and the agent within a few ulps of e on the same
    row (column) -- inside or just outside the 0.4 m, in the stencil's edge column or the next.  Right and left edge,
    along x and along y; pairs `stride` cells apart, isolated from each other."""
    out, k = [], k0
    for axis in (0, 1):
        other = (row + 0.5) * cell + off[1 - axis]
        for side in (1, -1):  # source + 0.4 (right / top edge) or source - 0.4 (left / bottom edge)
            for us, ua in PROBE_EDGE_ULPS:
                e = k * cell + off[axis]
                s = _nx(e - side * PROBE_RADIUS, us)
                a = _nx(e, ua)
                src, ag = [0.0, 0.0], [0.0, 0.0]
                src[axis], ag[axis] = s, a
                src[1 - axis] = ag[1 - axis] = other
                out.append((np.array(src), np.array(ag)))
                k += stride
    return out


def sink_threshold_configs(x0=5.0, spacing=11.0):
    """(r, waypoint, agent, inside): agents at T(r) - 1 ulp, T and T + 1 ulp from a waypoint, along an axis and a
    diagonal, for every radius of SINK_RADII; only T - 1 ulp is `norm < r`."""
    out, x = [], x0
    for r in SINK_RADII:
        for diagonal in (False, True):
            for which in range(3):
                p, qs = threshold_points(r, x, diagonal)
                out.append((r, p, qs[which], which == 0))
                x += spacing
    return out


def _bits(a):
    """Bit patterns, every NaN as the one quiet NaN: the sign of a NaN that an arithmetic operation produces is not
    specified by IEEE 754 (nor used by the reference), and the forms reach the same NaN through different operations."""
    if a.dtype != np.float64:
        return a
    return np.where(np.isnan(a), np.float64(NAN), a).view(np.uint64)


def _same(ta, tb, keys):
    for k in keys:
        a, b = _bits(ta[k]), _bits(tb[k])
        bad = np.nonzero(a != b)[0] if a.shape == b.shape else []
        assert a.shape == b.shape and len(bad) == 0, (k, [(int(i), hex(int(a[i])), hex(int(b[i]))) for i in bad[:8]])


def build_oracle(scene: SC.Scene, index_mode=O.DEFERRED, inject_velocity=True, order=None) -> O.OracleSim:
    """order: the iteration order as agent ids (the oracle's Custom order); None = ascending id."""
    o = O.OracleSim(scene.width, scene.height, scene.cell, scene.offset, index_mode=index_mode,
                    iter_order=O.ASCENDING_ID if order is None else O.CUSTOM)
    if order is not None:
        o.set_custom_order(order)
    kind, v = scene.hl
    hl = o.hl_parity(v) if kind == "parity" else o.hl_constant(v)
    lp = o.lp_none() if scene.lp[0] == "none" else o.lp_zanlungo(*scene.lp[1:])
    ids = o.add_agents(scene.xy, hl, lp, scene.eyesight)
    assert np.array_equal(ids, np.arange(scene.n, dtype=np.uint64))
    if inject_velocity and np.any(scene.vxy):
        o.set_state(ids, scene.xy[:, 0], scene.xy[:, 1], scene.vxy[:, 0], scene.vxy[:, 1])
    return o


def rel_err(a: np.ndarray, b: np.ndarray, scale=None) -> float:
    """max |a-b| / max(|a|,|b|,scale) with identical non-finite patterns required."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert np.array_equal(np.isnan(a), np.isnan(b)), "NaN pattern differs"
    assert np.array_equal(np.isinf(a), np.isinf(b)), "inf pattern differs"
    fin = np.isfinite(a) & np.isfinite(b)
    assert np.array_equal(a[~fin & ~np.isnan(a)], b[~fin & ~np.isnan(b)]), "inf signs differ"
    if not fin.any():
        return 0.0
    den = np.maximum(np.abs(a[fin]), np.abs(b[fin]))
    if scale is not None:
        den = np.maximum(den, np.broadcast_to(scale, a.shape)[fin] if np.ndim(scale) else scale)
    den = np.maximum(den, 1e-300)
    return float(np.max(np.abs(a[fin] - b[fin]) / den))


def compare_traces(tg: dict, to: dict) -> dict:
    """GPU trace vs oracle trace (both ascending id).  Returns summary numbers."""
    assert np.array_equal(tg["id"], to["id"])
    assert np.array_equal(tg["nb_offsets"], to["nb_offsets"]), "neighbour counts differ"
    assert np.array_equal(tg["nb_ids"], to["nb_ids"]), "neighbour lists differ (bit-exact, canonical order)"
    # t_i: bit-exact (compare the bit patterns so that inf == inf and -0 != +0 are both caught)
    assert np.array_equal(tg["t_i"].view(np.uint64), to["t_i"].view(np.uint64)), "t_i not bit-exact"
    fmag = np.sqrt(to["fx"] ** 2 + to["fy"] ** 2)
    fmag = np.where(np.isfinite(fmag), fmag, 0.0)
    ex = rel_err(tg["fx"], to["fx"], scale=fmag)
    ey = rel_err(tg["fy"], to["fy"], scale=fmag)
    return {"force_rel_err": max(ex, ey), "finite_tti": int(np.isfinite(to["t_i"]).sum()),
            "neighbours": int(to["nb_offsets"][-1])}


def csr_subset(t: dict, keep: np.ndarray) -> dict:
    """Restrict a trace (ascending id) to the agents selected by the boolean mask `keep`."""
    off = t["nb_offsets"].astype(np.int64)
    chunks = [t["nb_ids"][off[k]:off[k + 1]] for k in np.nonzero(keep)[0]]
    new_off = np.zeros(int(keep.sum()) + 1, dtype=np.uint64)
    if chunks:
        new_off[1:] = np.cumsum([len(c) for c in chunks])
    nb = np.concatenate(chunks) if chunks else t["nb_ids"][:0]
    return {"id": t["id"][keep], "t_i": t["t_i"][keep], "fx": t["fx"][keep], "fy": t["fy"][keep],
            "nb_offsets": new_off, "nb_ids": nb}


def compare_states(sg: dict, so: dict) -> dict:
    assert np.array_equal(sg["id"], so["id"])
    vmag = np.sqrt(so["vx"] ** 2 + so["vy"] ** 2)
    vmag = np.where(np.isfinite(vmag), vmag, 0.0)
    ev = max(rel_err(sg["vx"], so["vx"], scale=vmag), rel_err(sg["vy"], so["vy"], scale=vmag))
    ep = max(rel_err(sg["x"], so["x"]), rel_err(sg["y"], so["y"]))
    assert np.array_equal(sg["next_waypoint"].astype(np.uint64), so["next_waypoint"].astype(np.uint64))
    return {"vel_rel_err": ev, "pos_rel_err": ep}


def step_both(g, o, scene: SC.Scene):
    from rmf_crowdsim_b200 import Duration

    g.step(Duration(*scene.dt))
    o.step(*scene.dt)


def resync(g, o) -> None:
    """Make the CUDA simulation's state bit-identical to the oracle's (ascending-id arrays)."""
    so = o.read_state()
    if len(so["id"]):
        g.set_state(None, so["x"], so["y"], so["vx"], so["vy"])


def _cell_centres(cells, nx, cell=1.0):
    """Insertable points at the centre of data cells (x = idx // nx, y = idx % nx: the index formula's own inverse)."""
    return np.array([[(c // nx + 0.5) * cell, (c % nx + 0.5) * cell] for c in cells], dtype=np.float64)


def saturated_knn_cases():
    """(name, (width, height, cell, offset), agents, query, k) for the kNN ring walk at a saturated query cell.
    x = +inf floors to x_idx = i64::MAX; with an even nx, MAX * nx wraps to -nx, so a row y_idx in [nx, nx + len)
    lands inside the grid and the walk goes on; from ring 1 the sides whose upper bound wraps are empty.  With an odd
    nx the same query is outside at ring 0.  x = (2^63 - 1024) cells on a row 1024 * nx up hits the data through the
    wrapped index in every ring until its bounds wrap at ring 1024, which is then all outside."""
    even = (8.0, 8.0, 1.0, (0.0, 0.0))
    odd = (9.0, 9.0, 1.0, (0.0, 0.0))
    wide = (64.0, 4.0, 1.0, (0.0, 0.0))  # nx = 64, ny = 4: rows >= 4 alias into the next columns
    a_even = _cell_centres([12, 3, 4, 45, 63], 8)
    a_odd = _cell_centres([12, 3, 4, 45, 80], 9)
    a_wide = _cell_centres([100, 37, 200, 5, 255], 64)
    far = 2.0 ** 63 - 1024.0
    return [
        ("inf_even", even, a_even, (INF, 20.5), 10),     # ring 0: data cell 20 - 8 = 12; ring 1: cells 3, 4
        ("inf_even_k1", even, a_even, (INF, 20.5), 1),
        ("inf_even_row", even, a_even, (INF, 71.5), 10),  # the last aliased row: data cell 63
        ("inf_odd", odd, a_odd, (INF, 20.5), 10),
        ("inf_inf", even, a_even, (INF, INF), 10),
        ("minus_inf", even, a_even, (-INF, 3.5), 10),
        ("y_inf", even, a_even, (3.5, INF), 10),
        ("far_x", wide, a_wide, (far, 1024.0 * 64 + 100.5), 4000),
        ("far_x_k3", wide, a_wide, (far, 1024.0 * 64 + 100.5), 3),
    ]


# kNN around NaN distances on an 8 x 8 grid of 1 m cells at the origin: (agents with id = row, query, k, error?).
# The reference's sort panics on a NaN distance once two candidates are compared; a single candidate is returned.
NAN_KNN_CASES = [
    ([(NAN, NAN), (0.5, 0.5), (3.5, 3.5)], (0.2, 0.3), 1, True),    # cell 0 holds two, one NaN: k = 1 is enough
    ([(NAN, NAN), (0.5, 0.5), (3.5, 3.5)], (3.5, 3.6), 1, False),   # the walk stops before cell 0
    ([(NAN, NAN), (0.5, 0.5), (3.5, 3.5)], (3.5, 3.6), 3, True),
    ([(NAN, 2.0), (0.5, 0.5)], (6.5, 6.5), 9, True),                  # NaN x only
    ([(NAN, NAN)], (0.5, 0.5), 5, False),                             # one candidate: no comparison
    ([(NAN, NAN)], (1.5, 1.5), 5, True),                              # cell 0 is ring 1's doubled corner
    ([(0.5, 0.5), (3.5, 3.5)], (NAN, NAN), 1, False),                 # NaN query, one candidate in cell 0
    ([(0.5, 0.5), (3.5, 3.5)], (NAN, NAN), 2, True),
    ([(0.5, 0.5), (3.5, 3.5)], (NAN, 3.5), 1, True),                  # column 0, row 3: ring 3 brings both
    ([(0.5, 0.5), (3.5, 3.5)], (NAN, NAN), 0, False),
]
