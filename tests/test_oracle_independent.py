"""A second, independently written restatement of local_planners/zanlungo.rs -- plain Python floats (IEEE double,
the platform libm), transcribed line by line from the Rust source -- checked against the C++ oracle's golden
vectors.  `compute_agent_force`, `right_of_way_vel`, `slerp` and `compute_tti` have no test in the reference; two
restatements written separately and agreeing to the last bits is the strongest pin available without a Rust
toolchain (DESIGN.md section 6)."""
import math
import os

import numpy as np

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
INF = float("inf")
NAN = float("nan")


def _div(x, y):
    """IEEE-754 x / y, as Rust divides; Python raises on a zero divisor: x / +-0 is +-inf by the signs, 0 / 0 NaN."""
    if y != 0.0:
        return x / y
    if x != x or x == 0.0:
        return NAN
    return math.copysign(INF, x) * math.copysign(1.0, y)


def _exp(x):
    """f64::exp: overflows to inf where Python raises."""
    try:
        return math.exp(x)
    except OverflowError:
        return INF


def _norm(v):
    return math.sqrt(v[0] * v[0] + v[1] * v[1])


def _dot(a, b):
    return a[0] * b[0] + a[1] * b[1]


def slerp(t, p0, p1, sin_theta):  # zanlungo.rs:23-28
    theta = math.asin(sin_theta)
    t0 = math.sin((1.0 - t) * theta) / sin_theta if sin_theta != 0.0 else float("nan")
    t1 = math.sin(t * theta) / sin_theta if sin_theta != 0.0 else float("nan")
    return (p0[0] * t0 + p1[0] * t1, p0[1] * t0 + p1[1] * t1)


class Zanlungo:
    def __init__(self, agent_scale, obstacle_scale, reaction_time, force_distance, agent_mass, agent_radius):
        self.agent_scale, self.force_distance = agent_scale, force_distance
        self.agent_mass, self.agent_radius = agent_mass, agent_radius

    def time_to_collision(self, rel_vel, rel_pos):  # zanlungo.rs:49-74
        a = _dot(rel_vel, rel_vel)
        b = 2.0 * _dot(rel_vel, rel_pos)
        c = _dot(rel_pos, rel_pos) - self.agent_radius * self.agent_radius
        discriminant = b * b - 4.0 * a * c
        if discriminant < 0.0:
            return INF
        sq = math.sqrt(discriminant)
        t0 = _div(-b - sq, 2.0 * a)  # a == 0 divides by +0: +-inf, or NaN for a zero numerator
        t1 = _div(-b + sq, 2.0 * a)
        if (t0 < 0.0 and t1 > 0.0) or (t1 < 0.0 and t0 > 0.0):
            return 0.0
        if t0 < t1 and t0 > 0.0:
            return t0
        if t1 > 0.0:
            return t1
        return INF

    def right_of_way_vel(self, agent_id, agent_vel, self_pref, other_vel, other_pref, other_priority):  # :173-198
        row = min(max(float(agent_id) - other_priority, -1.0), 1.0)
        if row < 0.0:
            r_2 = math.sqrt(-row)
            adj = (other_vel[0] + r_2 * (other_pref[0] - other_vel[0]), other_vel[1] + r_2 * (other_pref[1] - other_vel[1]))
            return -r_2, agent_vel, adj
        if row > 0.0:
            r_2 = math.sqrt(row)
            vel = (agent_vel[0] + r_2 * (self_pref[0] - agent_vel[0]), agent_vel[1] + r_2 * (self_pref[1] - agent_vel[1]))
            return r_2, vel, other_vel
        return 0.0, agent_vel, other_vel

    def compute_agent_force(self, agent, other, t_i):  # :93-170; agent = (id, pos, vel, pref)
        aid, apos, avel, apref = agent
        oid, opos, ovel, opref = other
        weight, my_vel, other_vel = self.right_of_way_vel(aid, avel, apref, ovel, opref, float(oid))
        weight = 1.0 - weight
        fut = (apos[0] + my_vel[0] * t_i, apos[1] + my_vel[1] * t_i)
        ofut = (opos[0] + other_vel[0] * t_i, opos[1] + other_vel[1] * t_i)
        d_ij = (fut[0] - ofut[0], fut[1] - ofut[1])
        dist = _norm(d_ij)
        if weight > 1.0:
            interpolate = True
            perp = (0.0, 0.0)
            if _norm(opref) < 0.0001:
                crp = (apos[0] - opos[0], apos[1] - opos[1])
                perp = (-crp[1], crp[0])
                if _dot(perp, avel) < 0.0:
                    perp = (-perp[0], -perp[1])
            else:
                if _dot(opref, d_ij) > 0.0:
                    perp = (-opref[1], opref[0])
                    if _dot(perp, d_ij) < 0.0:
                        perp = (-perp[0], -perp[1])
                else:
                    interpolate = False
            if interpolate:
                sin_theta = perp[0] * d_ij[1] - perp[1] * d_ij[0]
                if sin_theta < 0.0:
                    sin_theta = -sin_theta
                if sin_theta > 1.0:
                    sin_theta = 1.0
                d_ij = slerp(weight - 1.0, d_ij, perp, sin_theta)
        if dist > _norm((fut[0] - ofut[0], fut[1] - ofut[1])):
            return (0.0, 0.0)
        n = _norm(d_ij)
        dn = (d_ij[0] / n, d_ij[1] / n) if n != 0.0 else (float("nan"), float("nan"))
        surface_dist = dist - self.agent_radius * 2.0
        rv = (my_vel[0] - other_vel[0], my_vel[1] - other_vel[1])
        magnitude = _div(weight * self.agent_scale * _norm(rv), t_i)
        if magnitude >= 1e15:
            magnitude = 1e15
        s = magnitude * _exp(_div(-surface_dist, self.force_distance))
        return (dn[0] * s, dn[1] * s)


def _rel(a, b, scale=0.0):
    return abs(a - b) / max(abs(a), abs(b), scale, 1e-300)


def test_pair_table_agrees_with_the_independent_restatement():
    g = np.load(os.path.join(G, "pair_table.npz"))
    z = Zanlungo(*g["params"])
    worst = 0.0
    for k in range(len(g["t_i"])):
        a, o = g["agent"][k], g["other"][k]
        f = z.compute_agent_force((int(g["aid"][k]), (a[0], a[1]), (a[2], a[3]), (a[4], a[5])),
                                  (int(g["oid"][k]), (o[0], o[1]), (o[2], o[3]), (o[4], o[5])), float(g["t_i"][k]))
        mag = math.hypot(*g["force"][k])
        worst = max(worst, _rel(f[0], g["force"][k][0], mag), _rel(f[1], g["force"][k][1], mag))
    assert worst <= 1e-14
    z = Zanlungo(1, 1, 0, 1, 1, float(g["ttc_radius"][0]))
    for k in range(len(g["ttc"])):
        t = z.time_to_collision(tuple(g["rel_vel"][k]), tuple(g["rel_pos"][k]))
        assert np.float64(t).view(np.uint64) == g["ttc"][k].view(np.uint64), k  # bit-exact


def test_crowd_step_agrees_with_the_independent_restatement():
    """t_i (compute_tti, :76-91) and the force sum (get_desired_velocity, :201-218) of all 576 agents, recomputed
    from the golden neighbour lists in list order; neighbours' preferred_vel is (0,0) (lib.rs:57,285)."""
    g = np.load(os.path.join(G, "crowd_576.npz"))
    z = Zanlungo(0.05, 1.0, 0.0, 0.5, 1.0, 0.2)
    xy, v = g["in_xy"], g["in_vxy"]
    off, nb = g["nb_offsets"].astype(np.int64), g["nb_ids"].astype(np.int64)
    worst, finite = 0.0, 0
    for i in range(len(xy)):
        pref = (-1.3, 0.0) if i % 2 == 0 else (1.3, 0.0)  # parity planner (main.rs:26-29) with v = (1.3, 0)
        me = (i, (xy[i, 0], xy[i, 1]), (v[i, 0], v[i, 1]), pref)
        t_i = INF
        for j in nb[off[i]:off[i + 1]]:
            ct = z.time_to_collision((v[j, 0] - v[i, 0], v[j, 1] - v[i, 1]), (xy[j, 0] - xy[i, 0], xy[j, 1] - xy[i, 1]))
            if ct < t_i:
                t_i = ct
        assert np.float64(t_i).view(np.uint64) == g["t_i"][i].view(np.uint64), i
        fx = fy = 0.0
        if t_i != INF:
            finite += 1
            for j in nb[off[i]:off[i + 1]]:
                f = z.compute_agent_force(me, (int(j), (xy[j, 0], xy[j, 1]), (v[j, 0], v[j, 1]), (0.0, 0.0)), t_i)
                fx += f[0]
                fy += f[1]
        mag = math.hypot(g["fx"][i], g["fy"][i])
        worst = max(worst, _rel(fx, g["fx"][i], mag), _rel(fy, g["fy"][i], mag))
        vx, vy = pref[0] + fx * (1.0 / 1.0), pref[1] + fy * (1.0 / 1.0)
        assert _rel(vx, g["vx"][i], 1.0) <= 1e-14 and _rel(vy, g["vy"][i], 1.0) <= 1e-14
    assert finite > 100 and worst <= 1e-13


def _nx(x, k):
    """k steps of nextafter from x (toward +inf for k > 0)."""
    for _ in range(abs(k)):
        x = math.nextafter(x, INF if k > 0 else -INF)
    return x


# (agent_radius, rel_vel, rel_pos, what) at the edges of time_to_collision (zanlungo.rs:49-74): where a and b*b
# underflow, where the discriminant is 0 or one unit from it, where the pair touches or overlaps, where b*b
# overflows, and non-finite components.
TTC_EDGES = [
    (0.2, (1.4e-162, 0.0), (1.0, 0.0), "a underflows to 0, b*b subnormal, b > 0: t0 = -inf, t1 = +inf -> 0"),
    (0.2, (-1.4e-162, 0.0), (1.0, 0.0), "a underflows to 0, b*b subnormal, b < 0 -> 0"),
    (0.2, (7e-163, 7e-163), (0.8, 0.9), "a == 0, sqrt(fl(b*b)) < b, b > 0: numerator < 0 -> inf"),
    (0.2, (-7e-163, -7e-163), (0.8, 0.9), "a == 0, sqrt(fl(b*b)) < |b|, b < 0: both roots +inf -> inf"),
    (0.2, (1e-163, 0.0), (-1.0, 0.0), "a == 0, b*b == 0, b != 0"),
    (0.2, (0.0, 0.0), (1.0, 0.0), "a == 0, b == 0"),
    (0.2, (0.0, -0.0), (0.1, 0.0), "a == 0, b == 0, overlapping"),
    (0.2, (1e-160, 0.0), (-1.0, 0.0), "a subnormal > 0, approaching"),
    (0.2, (1e-160, 0.0), (1.0, 0.0), "a subnormal > 0, receding"),
    (0.2, (3e-155, 0.0), (-1.0, 0.0), "a and b*b tiny but normal"),
    (0.5, (-1.0, 0.0), (3.0, 0.5), "grazing: disc == 0 exactly, t = 3"),
    (0.5, (-1.0, 0.0), (3.0, _nx(0.5, -17)), "disc one unit of b*b = 36 above 0"),
    (0.5, (-1.0, 0.0), (3.0, _nx(0.5, 9)), "disc one unit of b*b = 36 below 0"),
    (0.5, (-1.0, 0.0), (0.5, 0.0), "touching: c == 0"),
    (0.5, (1.0, 0.0), (0.5, 0.0), "touching, receding"),
    (0.5, (-1.0, 0.0), (0.3, 0.0), "overlap: c < 0 -> 0"),
    (0.5, (0.0, 1e-150), (0.3, 0.0), "overlap, tiny perpendicular speed -> 0"),
    (1e100, (1e60, 0.0), (-1e100, 0.0), "b*b overflows to inf, c == 0: disc = inf"),
    (0.2, (1e150, 0.0), (-1e10, 0.0), "b*b and 4ac overflow: disc NaN"),
    (0.2, (1e200, 0.0), (-1.0, 0.0), "a overflows to inf"),
    (0.2, (INF, 0.0), (-1.0, 0.0), "relative velocity inf"),
    (0.2, (NAN, 0.0), (-1.0, 0.0), "relative velocity NaN"),
    (0.2, (-1.0, 0.0), (INF, 0.0), "relative position inf"),
    (0.2, (-1.0, 0.0), (NAN, 1.0), "relative position NaN"),
    (0.0, (-1.0, 0.0), (1.0, 0.0), "radius 0"),
]


def _bits(x):
    return int(np.float64(x).view(np.uint64))


def _same_force(f, g):
    """Components: identical NaN / inf patterns and signs, finite values within the pair-table tolerance."""
    mag = math.hypot(g[0], g[1]) if all(math.isfinite(v) for v in g) else 0.0
    for a, b in zip(f, g):
        if math.isnan(a) or math.isnan(b) or math.isinf(a) or math.isinf(b):
            if not ((math.isnan(a) and math.isnan(b)) or a == b):
                return False
        elif _rel(a, b, mag) > 1e-14:
            return False
    return True


def test_time_to_collision_edges_agree_with_the_independent_restatement():
    """Every edge class of time_to_collision bit for bit, and the force of each such pair (both id orders: the yield
    and the weight-0 branch of right_of_way_vel) at the existing tolerance, NaN and inf patterns included."""
    import oracle_ffi as O

    L = O.lib()
    results = set()
    for r, rv, rp, what in TTC_EDGES:
        want = O.ttc(r, rv, rp)
        got = Zanlungo(1, 1, 0, 1, 1, r).time_to_collision(rv, rp)
        assert _bits(got) == _bits(want), (what, got, want)
        results.add(want if want == want else "nan")
        params = np.array([0.05, 1.0, 0.0, 0.5, 1.0, r])
        z = Zanlungo(*params.tolist())
        me = (0.25, -0.5, 0.3, 0.1, 1.3, 0.0)  # x, y, vx, vy, preferred vx, vy
        other = (me[0] + rp[0], me[1] + rp[1], me[2] + rv[0], me[3] + rv[1], 0.0, 0.0)
        for aid, oid in ((3, 7), (7, 3)):
            out = np.zeros(2)
            a, o = np.array(me), np.array(other)
            L.orc_agent_force(params.ctypes.data_as(O.f64p), aid, a.ctypes.data_as(O.f64p), oid,
                              o.ctypes.data_as(O.f64p), want, out.ctypes.data_as(O.f64p))
            f = z.compute_agent_force((aid, me[:2], me[2:4], me[4:]), (oid, other[:2], other[2:4], other[4:]), want)
            assert _same_force(f, tuple(out)), (what, aid, f, tuple(out))
    # the table reaches every kind of result: 0, finite > 0, inf
    assert 0.0 in results and INF in results and any(isinstance(t, float) and 0.0 < t < INF for t in results)
    # the classes are what their names say
    assert O.ttc(0.2, (1.4e-162, 0.0), (1.0, 0.0)) == 0.0 and O.ttc(0.5, (-1.0, 0.0), (3.0, 0.5)) == 3.0
    unit = math.ulp(36.0)
    for y, disc in ((0.5, 0.0), (_nx(0.5, -17), unit), (_nx(0.5, 9), -unit)):
        assert 36.0 - 4.0 * ((9.0 + y * y) - 0.25) == disc, y


def test_underflowing_relative_speed_gives_t_i_zero_and_a_nan_force():
    """Two agents 1 m apart whose parity velocities (+-7e-163 m/s) make |v_rel|^2 underflow to 0 while (2 v.p)^2 is a
    non-zero subnormal: the reference divides by 2a = +0 and returns t_i = 0 (zanlungo.rs:60-70), and the force
    (2 scale |v|) / 0 is NaN.  Positions go NaN in the second step and stay NaN."""
    import oracle_ffi as O

    za = (0.05, 1.0, 0.0, 0.5, 1.0, 0.2)
    o = O.OracleSim(16.0, 16.0, 2.0, (0.0, 0.0))
    o.add_agents(np.array([[5.0, 5.0], [6.0, 5.0]]), o.hl_parity((7e-163, 0.0)), o.lp_zanlungo(*za), 2.0)
    o.enable_trace(True)
    z = Zanlungo(*za)
    want_t = [[INF, INF], [0.0, 0.0], None]
    for step in range(3):
        s = o.read_state()
        o.step(0, 16_666_667)
        t = o.read_trace()
        xy, v = np.stack([s["x"], s["y"]], axis=1), np.stack([s["vx"], s["vy"]], axis=1)
        for i, j in ((0, 1), (1, 0)):
            ti = z.time_to_collision((v[j, 0] - v[i, 0], v[j, 1] - v[i, 1]), (xy[j, 0] - xy[i, 0], xy[j, 1] - xy[i, 1]))
            if math.isnan(xy[i, 0]):
                continue  # the NaN agents sit in cell 0 and no longer see each other
            assert _bits(ti) == _bits(t["t_i"][i]), (step, i)
            if ti != INF:
                pref = (-7e-163, 0.0) if i % 2 == 0 else (7e-163, 0.0)
                f = z.compute_agent_force((i, tuple(xy[i]), tuple(v[i]), pref), (j, tuple(xy[j]), tuple(v[j]), (0, 0)),
                                          ti)
                assert math.isnan(f[0]) and math.isnan(t["fx"][i]), (step, i)
        if want_t[step] is not None:
            assert [_bits(x) for x in t["t_i"]] == [_bits(x) for x in want_t[step]], step
    s = o.read_state()
    assert np.isnan(s["x"]).all() and np.isnan(s["y"]).all()


class _Hash2D:
    """location_hash_2d.rs, second restatement: per-cell id sets (visited in ascending id: the canonical stand-in for
    the reference's HashSet order), insert cell by truncation (:54-66), query cells by floor (:68-72, :103-122), the
    width cell count as stride for both coordinates (:59, :74-85)."""

    def __init__(self, width, height, cell, off):
        self.res, self.off = cell, off
        self.nx = int(width / cell)
        self.len = self.nx * int(height / cell)
        self.cells = {}
        self.where = {}
        self.loc = {}

    @staticmethod
    def _as_usize(v):
        if v != v or v <= 0.0:
            return 0
        return int(v)  # trunc toward zero (values here are far below 2^64)

    def index(self, p):
        idx = self._as_usize((p[0] - self.off[0]) / self.res) * self.nx + self._as_usize((p[1] - self.off[1]) / self.res)
        return idx if idx < self.len else None

    def add_or_update(self, i, p):
        idx = self.index(p)
        if idx is None:
            raise ValueError("Index out of bounds")
        old = self.where.get(i)
        if old != idx:
            if old is not None:
                self.cells[old].discard(i)
            self.cells.setdefault(idx, set()).add(i)
            self.where[i] = idx
        self.loc[i] = p

    def neighbours_in_radius(self, radius, p):
        fl = lambda v: math.floor(v)  # noqa: E731
        right = fl(((p[0] + radius) - self.off[0]) / self.res)
        left = fl(((p[0] - radius) - self.off[0]) / self.res)
        top = fl(((p[1] + radius) - self.off[1]) / self.res)
        bottom = fl(((p[1] - radius) - self.off[1]) / self.res)
        out = []
        for x in range(left, right + 1):
            for y in range(bottom, top + 1):
                if x < 0 or y < 0:
                    continue
                idx = x * self.nx + y
                if idx >= self.len:
                    continue
                for j in sorted(self.cells.get(idx, ())):
                    q = self.loc[j]
                    if _norm((q[0] - p[0], q[1] - p[1])) < radius:
                        out.append(j)
        return out


def test_in_loop_step_agrees_with_the_independent_restatement():
    """lib.rs:259-359 with the index updated INSIDE the loop (:299), written a second time in plain Python: the
    neighbour set of an agent is decided by the new positions of the agents before it in the iteration order, the
    planner gets their old states (:281-286).  Against the golden vector the C++ oracle generated in that mode: same
    neighbour lists, t_i to the bit, forces and new state to the last bits."""
    g = np.load(os.path.join(G, "in_loop_400.npz"))
    xy, v, order = g["in_xy"], g["in_vxy"], [int(i) for i in g["order"]]
    dt = float(int(g["dt"][0])) + float(int(g["dt"][1])) / 1e9
    z = Zanlungo(0.05, 1.0, 0.0, 0.5, 200.0, 0.1)
    n = len(xy)
    side = 20
    dom = math.ceil((side * 1.0 + 2 * 8.0) / 2.0) * 2.0  # scenes.uniform_crowd(20, margin=8, cell=2)
    h = _Hash2D(dom, dom, 2.0, (-8.0, -8.0))
    for i in range(n):
        h.add_or_update(i, (xy[i, 0], xy[i, 1]))
    off, nb = g["nb_offsets"].astype(np.int64), g["nb_ids"].astype(np.int64)
    new_state = {}
    worst, finite = 0.0, 0
    for i in order:
        pref = (-1.3, 0.0) if i % 2 == 0 else (1.3, 0.0)
        pos_i, vel_i = (xy[i, 0], xy[i, 1]), (v[i, 0], v[i, 1])
        me = (i, pos_i, vel_i, pref)
        lst = [j for j in h.neighbours_in_radius(2.0, pos_i) if j != i]
        assert lst == [int(j) for j in nb[off[i]:off[i + 1]]], i
        t_i = INF
        for j in lst:  # OLD states of the neighbours
            ct = z.time_to_collision((v[j, 0] - vel_i[0], v[j, 1] - vel_i[1]), (xy[j, 0] - pos_i[0], xy[j, 1] - pos_i[1]))
            if ct < t_i:
                t_i = ct
        assert np.float64(t_i).view(np.uint64) == g["t_i"][i].view(np.uint64), i
        fx = fy = 0.0
        if t_i != INF:
            finite += 1
            for j in lst:
                f = z.compute_agent_force(me, (j, (xy[j, 0], xy[j, 1]), (v[j, 0], v[j, 1]), (0.0, 0.0)), t_i)
                fx += f[0]
                fy += f[1]
        mag = math.hypot(g["fx"][i], g["fy"][i])
        worst = max(worst, _rel(fx, g["fx"][i], mag), _rel(fy, g["fy"][i], mag))
        vel = (pref[0] + fx * (1.0 / 200.0), pref[1] + fy * (1.0 / 200.0))
        new_pos = (pos_i[0] + vel[0] * dt, pos_i[1] + vel[1] * dt)
        h.add_or_update(i, new_pos)  # lib.rs:299: the agents after this one see it here
        new_state[i] = (new_pos, vel)
    for i in range(n):
        (px, py), (vx, vy) = new_state[i]
        assert _rel(px, g["x"][i], 1.0) <= 1e-14 and _rel(py, g["y"][i], 1.0) <= 1e-14
        assert _rel(vx, g["vx"][i], 1.0) <= 1e-14 and _rel(vy, g["vy"][i], 1.0) <= 1e-14
    assert finite > 50 and worst <= 1e-13


def test_radius_query_agrees_with_the_independent_hash_grid():
    """get_neighbours_in_radius (location_hash_2d.rs:240-258) of all 576 agents of the golden crowd step through the
    second hash-grid restatement: the same lists in the same order (cells x-major then y, ascending id in a cell)."""
    g = np.load(os.path.join(G, "crowd_576.npz"))
    xy = g["in_xy"]
    dom = math.ceil((24 * 1.0 + 2 * 8.0) / 2.0) * 2.0  # scenes.uniform_crowd(24, margin=8, cell=2)
    h = _Hash2D(dom, dom, 2.0, (-8.0, -8.0))
    for i in range(len(xy)):
        h.add_or_update(i, (xy[i, 0], xy[i, 1]))
        assert h.where[i] == int(g["cells"][i])
    off, nb = g["nb_offsets"].astype(np.int64), g["nb_ids"].astype(np.int64)
    for i in range(len(xy)):
        lst = [j for j in h.neighbours_in_radius(2.0, (xy[i, 0], xy[i, 1])) if j != i]
        assert lst == [int(j) for j in nb[off[i]:off[i + 1]]], i


def _nearest(h, n, p):
    """get_nearest_neighbours (location_hash_2d.rs:151-238), second restatement: rings of cells around the query cell
    with HALF-OPEN sides (the (x-s, y-s) corner is visited twice, the (x+s, y+s) corner never), stop at the first ring
    that brings the candidate count to n or when a whole ring is outside the grid, then a stable sort by distance."""
    x_idx = math.floor((p[0] - h.off[0]) / h.res)
    y_idx = math.floor((p[1] - h.off[1]) / h.res)
    ring = []

    def visit(cx, cy, stat):
        stat[1] += 1
        if cx < 0 or cy < 0 or cx * h.nx + cy >= h.len:
            stat[0] += 1
            return
        for j in sorted(h.cells.get(cx * h.nx + cy, ())):
            ring.append((h.loc[j], j))

    step, all_out = 0, False
    while len(ring) < n and not all_out:
        stat = [0, 0]
        if step == 0:
            visit(x_idx, y_idx, stat)
        else:
            for i in range(x_idx - step, x_idx + step):
                visit(i, y_idx + step, stat)
            for i in range(x_idx - step, x_idx + step):
                visit(i, y_idx - step, stat)
            for i in range(y_idx - step, y_idx + step):
                visit(x_idx - step, i, stat)
            for i in range(y_idx - step, y_idx + step):
                visit(x_idx + step, i, stat)
        all_out = stat[0] == stat[1]
        step += 1
    ring.sort(key=lambda e: _norm((e[0][0] - p[0], e[0][1] - p[1])))  # list.sort is stable, like the reference's
    return [j for _, j in ring[:n]]


def test_nearest_neighbours_agree_with_the_independent_hash_grid():
    """The 10 x 10 point grid of the reference's own test (location_hash_2d.rs:310-339) and 61 random queries of the
    golden vector: the second restatement returns the oracle's lists, duplicates and misses of the ring walk included."""
    g = np.load(os.path.join(G, "knn_radius_100.npz"))
    h = _Hash2D(10.0, 10.0, 0.5, (0.0, 0.0))
    for x in range(10):
        for y in range(10):
            h.add_or_update(10 * x + y, (x + 0.5, y + 0.5))
    assert _nearest(h, 1, (0.6, 0.6)) == [0]                     # the reference's assertions
    assert _nearest(h, 4, (1.7, 1.6)) == [11, 21, 12, 10]
    for k, q in enumerate(g["q"]):
        want = [int(v) for v in g["knn4"][k, : int(g["knn4_count"][k])]]
        assert _nearest(h, 4, (q[0], q[1])) == want, (k, q)
        lo, hi = int(g["rad_offsets"][k]), int(g["rad_offsets"][k + 1])
        assert h.neighbours_in_radius(float(g["radius"][0]), (q[0], q[1])) == [int(v) for v in g["rad_ids"][lo:hi]]


def test_source_sink_stream_agrees_with_the_independent_restatement():
    """lib.rs:195-383 around one SourceSink, written a second time: MonotonicCrowd (source_sink.rs:96-100,
    round(dt * rate)), the 0.4 m emptiness probe on the start-of-step index (lib.rs:208-217), sequential ids
    (:128-129), the waypoint test on the OLD position (:305-336) and removal after the commit (:378-380).  Scenario of
    tests/event_listeners_test.rs; per-step agent count, spawns and despawns and the final state of the golden vector."""
    g = np.load(os.path.join(G, "source_sink.npz"))
    h = _Hash2D(1000.0, 1000.0, 20.0, (-500.0, -500.0))
    source, waypoints, radius_sink, rate, dt = (0.0, 0.0), [(20.0, 0.0)], 1.0, 1.0, 1.0
    agents, next_id = {}, 0  # id -> [pos, next_waypoint]
    for step in range(40):
        spawned = destroyed = 0
        number = int(math.floor(dt * rate + 0.5))  # f64::round of a positive value
        if number > 0 and not h.neighbours_in_radius(0.4, source):
            agents[next_id] = [source, 0]
            h.add_or_update(next_id, source)
            next_id += 1
            spawned = 1
        updates, leaving = {}, []
        for i in sorted(agents):
            pos, wp = agents[i]
            vel = (1.0, 0.0)  # the stub high-level planner of the test, NoLocalPlan keeps it
            new_pos = (pos[0] + vel[0] * dt, pos[1] + vel[1] * dt)
            if _norm((pos[0] - waypoints[wp][0], pos[1] - waypoints[wp][1])) < radius_sink:
                if wp == len(waypoints) - 1:
                    leaving.append(i)
                else:
                    wp += 1
            updates[i] = [new_pos, wp]
        for i, st in updates.items():
            agents[i] = st
            h.add_or_update(i, st[0])
        for i in leaving:
            del agents[i]
            h.cells[h.where.pop(i)].discard(i)
            del h.loc[i]
            destroyed += 1
        assert (len(agents), spawned, destroyed) == (int(g["count"][step]), int(g["spawned"][step]),
                                                      int(g["destroyed"][step])), step
    ids = sorted(agents)
    assert ids == [int(v) for v in g["final_id"]]
    assert [agents[i][0][0] for i in ids] == [float(v) for v in g["final_x"]]
