"""GPU: rcs_step_in_loop (the reference's in-loop index semantic, lib.rs:299, as a fixed-point iteration of sweeps) at
its edges, against the oracle's IN_LOOP mode running the literal sequential loop: partial, noisy and repeated
iteration orders, max_sweeps at its limit, a dependency chain that needs one sweep per agent, non-finite values in
the per-sweep index, crowded cells of that index, and mixed planner groups.  Neighbour lists and t_i bit-exact,
forces and state within 1e-9 with identical NaN/inf patterns.  Each family asserts that its edge class is hit."""
import numpy as np
import pytest

import oracle_ffi as O
import parity as P
import rmf_crowdsim_b200 as R
from rmf_crowdsim_b200 import scenes as SC

pytestmark = pytest.mark.gpu

DT = (0, 250_000_000)
ZAN = ("zanlungo", 0.05, 1.0, 0.0, 0.5, 200.0, 0.1)
NO_FIXED_POINT = "no fixed point within max_sweeps"


def _crowd(side=10, seed=13, cell=1.0, eyesight=2.5):
    rng = np.random.default_rng(seed)
    scene = SC.uniform_crowd(side, "shuffled", cell=cell, eyesight=eyesight, margin=8.0, seed=seed, lp=ZAN)
    scene.vxy = scene.vxy + rng.uniform(-0.3, 0.3, size=scene.vxy.shape)
    return scene


def _pair(scene, order=None):
    g = SC.build_simulation(scene)
    g.set_trace(True)
    o = P.build_oracle(scene, index_mode=O.IN_LOOP, order=order)
    o.enable_trace(True)
    return g, o


def _compare(g, o, zan=None):
    """zan: per id, True for the Zanlungo agents (the device lists no neighbours for NoLocalPlan agents)."""
    tg, to = g.read_trace(), o.read_trace()
    if zan is not None:
        tg, to = P.csr_subset(tg, zan[tg["id"].astype(np.int64)]), P.csr_subset(to, zan[to["id"].astype(np.int64)])
    r = P.compare_traces(tg, to)
    assert r["force_rel_err"] <= P.REL_TOL
    s = P.compare_states(g.read_state(), o.read_state())
    assert s["vel_rel_err"] <= P.REL_TOL and s["pos_rel_err"] <= P.REL_TOL
    return r


def _step(g, o, order=None, max_sweeps=0, dt=DT, zan=None):
    sweeps = g.step_in_loop(R.Duration(*dt), order=order, max_sweeps=max_sweeps)
    o.step(*dt)
    return sweeps, _compare(g, o, zan)


def _same_state(a, b):
    P._same(a, b, ("id", "x", "y", "vx", "vy"))


@pytest.mark.parametrize("kind", ["ascending", "descending", "random", "partial", "noisy"])
def test_in_loop_orders(kind):
    """Permutations, a partial order (the live ids it leaves out are visited after it, in ascending id) and an order
    with ids that were never allocated or were removed (ignored)."""
    scene = _crowd()
    n = scene.n
    rng = np.random.default_rng(3)
    perm = rng.permutation(n).astype(np.uint64)
    gone = int(perm[-1])
    order = {"ascending": np.arange(n, dtype=np.uint64), "descending": np.arange(n, dtype=np.uint64)[::-1].copy(),
             "random": perm, "partial": perm[: n // 2].copy(),
             "noisy": np.concatenate([[n + 5, gone], perm[:40], [2 ** 40], perm[40:-1]]).astype(np.uint64)}[kind]
    g, o = _pair(scene, order)
    if kind == "noisy":
        g.remove_agents(gone)
        o.remove_agent(gone)
    for _ in range(2):
        P.resync(g, o)
        sweeps, r = _step(g, o, order)
        assert sweeps >= 2 and r["finite_tti"] > 0
    assert len(g.read_trace()["id"]) == n - (kind == "noisy")  # every live agent was stepped


def test_in_loop_repeated_id_is_refused_and_nothing_changes():
    scene = _crowd(side=8)
    order = np.random.default_rng(4).permutation(scene.n).astype(np.uint64)
    g, o = _pair(scene, order)
    _step(g, o, order)
    before, tr, steps = g.read_state(), g.read_trace(), g.stats().steps
    bad = np.concatenate([order[:10], order[5:6], order[10:]])
    with pytest.raises(R.CrowdsimError, match="an id occurs twice in the order"):
        g.step_in_loop(R.Duration(*DT), order=bad)
    _same_state(g.read_state(), before)
    P._same(g.read_trace(), tr, ("id", "t_i", "fx", "fy", "nb_offsets", "nb_ids"))
    assert g.stats().steps == steps
    o2 = P.build_oracle(scene, index_mode=O.IN_LOOP, order=bad)
    with pytest.raises(O.OracleError, match="an id occurs twice in the order"):
        o2.step(*DT)
    _step(g, o, order)


def test_in_loop_max_sweeps_at_its_edge():
    """S sweeps (learned with max_sweeps = 0): S - 1 fails and commits nothing, S succeeds and matches the oracle.
    max_sweeps = 1 always fails: sweep 0 has no previous sweep to agree with."""
    scene = _crowd(side=12, seed=21)
    g, o = _pair(scene)
    s = SC.build_simulation(scene).step_in_loop(R.Duration(*DT))
    assert s >= 3
    before, steps = g.read_state(), g.stats().steps
    for m in (1, s - 1):
        with pytest.raises(R.CrowdsimError, match=NO_FIXED_POINT):
            g.step_in_loop(R.Duration(*DT), max_sweeps=m)
        _same_state(g.read_state(), before)
        assert g.stats().steps == steps
    sweeps, _ = _step(g, o, max_sweeps=s)
    assert sweeps == s and g.stats().steps == steps + 1


def _chain(n_links):
    """Agents on a line, each D = 2.5 m ahead of the previous one in the iteration order (eyesight 2 m), all heading +x
    at 2.004 m/s: a predecessor that keeps its line lands 1.999 m behind, inside the eyesight, one that a force pushed
    sideways lands outside.  An agent is pushed exactly when it sees its predecessor (t_i is finite: the old velocities
    close in along the line), so every link's neighbour set flips on the link before it; a pusher behind the first link
    starts the chain.  Ids descend along the line: the right-of-way weight is 2 only against a higher id."""
    D, c = 2.5, 0.3
    xy = np.array([[D * (n_links - 1 - i), 0.0] for i in range(n_links)] + [[-1.5, 0.0]])
    vxy = np.zeros_like(xy)
    vxy[:n_links, 0] = [-c * (n_links - i) for i in range(n_links)]
    vxy[n_links, 0] = 0.5
    scene = SC.Scene("chain", 80.0, 80.0, 2.0, (-10.0, -10.0), xy, vxy, 2.0, hl=("constant", (2.004, 0.0)),
                     lp=("zanlungo", 1.0, 1.0, 0.0, 30.0, 1.0, 0.2))
    return scene, np.arange(n_links + 1, dtype=np.uint64)[::-1].copy()


def test_in_loop_long_dependency_chain():
    scene, order = _chain(24)
    g, o = _pair(scene, order)
    sweeps, r = _step(g, o, order)
    assert sweeps >= 16, sweeps
    t = o.read_trace()
    seen = np.isfinite(t["t_i"][:24])
    assert 6 <= seen.sum() <= 20  # the links alternate: seen, pushed out of sight, not seen, ...


def test_in_loop_non_finite_values():
    """NaN start positions piling up in cell 0; a -inf velocity, which turns its neighbours' forces and new positions
    non-finite (cell 0 of the per-sweep index); and a pair with t_i = 0 and a NaN force whose positions go NaN."""
    scene = _crowd(side=8, seed=9)
    xy = scene.xy.copy()
    xy[[3, 17, 29]] = np.nan
    scene.xy = xy
    g, o = _pair(scene)
    v = o.read_state()
    vx = v["vx"].copy()
    vx[40] = -np.inf
    g.set_state(None, v["x"], v["y"], vx, v["vy"])
    o.set_state(v["id"], v["x"], v["y"], vx, v["vy"])
    _step(g, o)
    bad = ~np.isfinite(o.read_state()["x"])
    assert bad[[3, 17, 29]].all() and bad.sum() > 3
    za = (0.05, 1.0, 0.0, 0.5, 1.0, 0.2)
    pair = SC.Scene("nan_pair", 16.0, 16.0, 2.0, (0.0, 0.0), np.array([[5.0, 5.0], [6.0, 5.0], [9.0, 9.0]]),
                    np.zeros((3, 2)), 2.0, hl=("parity", (7e-163, 0.0)), lp=("zanlungo",) + za)
    g, o = _pair(pair)
    ti = []
    for _ in range(3):
        _step(g, o, dt=(0, 16_666_667))
        ti.append(o.read_trace()["t_i"][:2].tolist())
    # agent 0 goes first: t_i = 0, a NaN force, a NaN new position in cell 0, where agent 1 no longer finds it
    x = o.read_state()["x"]
    assert ti[1] == [0.0, float("inf")] and np.isnan(x[0]) and np.isfinite(x[1])


def _two_groups(w, cell, off, xs, groups):
    """A Simulation and an IN_LOOP oracle with the agents of `groups` [(rows, lp params or None, eyesight)] added in
    turn, all with the constant planner (4, 0); returns (g, o, per id: Zanlungo?)."""
    idx = R.LocationHash2D(w, w, cell, off, capacity=len(xs) + 16)
    g = R.Simulation(idx)
    g.set_trace(True)
    o = O.OracleSim(w, w, cell, off, index_mode=O.IN_LOOP)
    o.enable_trace(True)
    hl, ohl = R.ConstantVelocityPlan((4.0, 0.0)), o.hl_constant((4.0, 0.0))
    g._keep = [hl]
    zmask = []
    for rows, zan, eye in groups:
        lp = R.NoLocalPlan() if zan is None else R.Zanlungo(*zan)
        g._keep.append(lp)
        olp = o.lp_none() if zan is None else o.lp_zanlungo(*zan)
        ids = g.add_agents(xs[rows], hl, lp, eye)
        assert list(o.add_agents(xs[rows], ohl, olp, eye)) == ids
        zmask += [zan is not None] * len(ids)
    return g, o, np.array(zmask)


@pytest.mark.parametrize("members", [40, 5000])
def test_in_loop_crowded_cells_of_the_per_sweep_index(members):
    """The new positions of a sweep gather in one cell with > 32 members (the block sorter) or > 4096 (rank_huge_cell):
    a dense blob of NoLocalPlan agents moving as one into the next cell, whose Zanlungo neighbours list the blob's
    members from that cell in ascending id."""
    rng = np.random.default_rng(members)
    blob = rng.uniform([2.05, 2.05], [2.95, 2.95], size=(members, 2))
    ring = rng.uniform([1.0, 1.0], [5.0, 5.0], size=(60, 2))
    xs = np.concatenate([blob, ring])
    perm = rng.permutation(len(xs))
    xs = xs[perm]
    is_blob = perm < members  # the blob goes in first: its ids precede the ring's, so the ring sees its new positions
    g, o, zan = _two_groups(12.0, 1.0, (-3.0, -3.0), xs, [(np.nonzero(is_blob)[0], None, 0.01),
                                                           (np.nonzero(~is_blob)[0], ZAN[1:], 1.5)])
    _, r = _step(g, o, zan=zan)
    s = o.read_state()
    cells = np.floor(s["x"] + 3.0).astype(int) * 12 + np.floor(s["y"] + 3.0).astype(int)
    assert np.bincount(cells).max() >= members
    assert r["neighbours"] > members


def test_in_loop_more_oversized_cells_than_the_big_list_holds():
    """4225 cells of the per-sweep index with 33 members each: more oversized cells (> 32) than big_list's 4096
    entries, so the sorter's overflow branch ranks every cell.  Zanlungo agents among them list the members in
    ascending id."""
    rng = np.random.default_rng(17)
    side, per = 65, 33
    cx, cy = np.meshgrid(np.arange(side), np.arange(side), indexing="ij")
    base = np.repeat(np.stack([cx.ravel(), cy.ravel()], axis=1).astype(np.float64), per, axis=0)
    dense = base + rng.uniform(0.05, 0.95, size=base.shape)
    sparse = rng.uniform(0.0, side, size=(100, 2))
    xs = np.concatenate([dense, sparse])
    n_dense = len(dense)
    g, o, zan = _two_groups(80.0, 1.0, (-3.0, -3.0), xs, [(np.arange(n_dense), None, 0.01),
                                                           (np.arange(n_dense, len(xs)), ZAN[1:], 1.5)])
    _, r = _step(g, o, zan=zan)
    s = o.read_state()
    cells = np.floor(s["x"] + 3.0).astype(int) * 80 + np.floor(s["y"] + 3.0).astype(int)
    assert int((np.bincount(cells) > 32).sum()) > 4096
    assert r["neighbours"] > 100 * per


def test_in_loop_mixed_groups():
    """NoLocalPlan agents interleaved (by id) with Zanlungo ones, a host-evaluated planner group, and an eyesight wider
    than a cell, against the oracle's IN_LOOP mode."""
    rng = np.random.default_rng(8)
    w, cell, off = 24.0, 1.0, (-4.0, -4.0)
    gx, gy = np.meshgrid(np.arange(15), np.arange(12), indexing="ij")  # a jittered lattice: no overlapping pairs
    pts = np.stack([gx.ravel(), gy.ravel()], axis=1)[:180] + rng.uniform(0.3, 0.7, size=(180, 2))
    pts = pts[rng.permutation(180)]
    vel = rng.uniform(-0.5, 0.5, size=(180, 2))
    idx = R.LocationHash2D(w, w, cell, off, capacity=256)
    g = R.Simulation(idx)
    g.set_trace(True)
    o = O.OracleSim(w, w, cell, off, index_mode=O.IN_LOOP)
    o.enable_trace(True)
    zan = (0.05, 1.0, 0.0, 0.5, 20.0, 0.1)

    class Host(R.HighLevelPlanner):
        def get_desired_velocity(self, agent, time):
            return (0.3 * ((agent.agent_id % 3) - 1), 0.7)

    host = Host()
    hl_c, hl_p = R.ConstantVelocityPlan((1.1, -0.4)), R.ParityVelocityPlan((0.9, 0.2))
    lp_z, lp_n = R.Zanlungo(*zan), R.NoLocalPlan()
    o_hc, o_hp, o_hh = o.hl_constant((1.1, -0.4)), o.hl_parity((0.9, 0.2)), o.hl_host()
    o_z, o_n = o.lp_zanlungo(*zan), o.lp_none()
    plan = [(hl_c, o_hc, lp_z, o_z, 2.5), (hl_c, o_hc, lp_n, o_n, 2.5), (hl_p, o_hp, lp_z, o_z, 0.6),
            (host, o_hh, lp_z, o_z, 3.2)]
    host_ids, zan_ids = [], []
    for k in range(0, 180, 10):  # groups of 10 in turn: ids interleave between groups
        hl, ohl, lp, olp, eye = plan[(k // 10) % 4]
        ids = g.add_agents(pts[k:k + 10], hl, lp, eye)
        assert list(o.add_agents(pts[k:k + 10], ohl, olp, eye)) == ids
        if hl is host:
            host_ids += ids
        if lp is lp_z:
            zan_ids += ids
    zan = np.isin(np.arange(180), zan_ids)
    g.set_state(None, vx=vel[:, 0].copy(), vy=vel[:, 1].copy())
    o.set_state(np.arange(180, dtype=np.uint64), pts[:, 0], pts[:, 1], vel[:, 0], vel[:, 1])
    o.set_preferred_velocity(o_hh, host_ids, [(0.3 * ((i % 3) - 1), 0.7) for i in host_ids])
    for _ in range(2):
        P.resync(g, o)
        sweeps = g.step_in_loop(R.Duration(0, 200_000_000))
        o.step(0, 200_000_000)
        r = _compare(g, o, zan)
        assert sweeps >= 2 and r["finite_tti"] > 0


def test_in_loop_refusals():
    """Study mode runs one handle without source sinks or route followers: both are refused before anything runs."""
    idx = R.LocationHash2D(20.0, 20.0, 1.0, (0.0, 0.0), capacity=64)
    g = R.Simulation(idx)
    g.add_agents([(3.0, 3.0)], R.ConstantVelocityPlan((1.0, 0.0)), R.NoLocalPlan(), 1.0)
    g.add_source_sink(R.SourceSink((5.0, 5.0), 0.5, R.MonotonicCrowd(1.0), R.ConstantVelocityPlan((1.0, 0.0)),
                                   R.NoLocalPlan(), [(9.0, 5.0)], False, 1.0))
    before = g.read_state()
    with pytest.raises(R.CrowdsimError, match="without strips, source sinks or route followers"):
        g.step_in_loop(R.Duration(0, 100_000_000))
    _same_state(g.read_state(), before)
    idx = R.LocationHash2D(20.0, 20.0, 1.0, (0.0, 0.0), capacity=64)
    g = R.Simulation(idx)
    g.add_agents([(3.0, 3.0)], R.RouteFollowPlan([(4.0, 4.0), (8.0, 4.0)]), R.NoLocalPlan(), 1.0)
    with pytest.raises(R.CrowdsimError, match="without strips, source sinks or route followers"):
        g.step_in_loop(R.Duration(0, 100_000_000))
