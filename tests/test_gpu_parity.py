"""GPU: parity of the CUDA path against the CPU oracle on identical seeded inputs, through the C ABI.
Bar (BASELINE.json north_star): cell assignments and neighbour sets bit-exact, t_i bit-exact,
forces and velocities within 1e-9 relative."""
import numpy as np
import pytest

import oracle_ffi as O
import parity as P
import rmf_crowdsim_b200 as R
from rmf_crowdsim_b200 import scenes as SC

pytestmark = pytest.mark.gpu


def _run(scene, steps, trace=True, resync=True):
    """Per-step parity on IDENTICAL inputs: before every step the oracle's state is injected into the
    CUDA simulation (CUDA's exp/asin/sin differ from glibc's in the last ulp, so free-running
    trajectories separate at the 1e-16 level after the first interaction; that drift is reported by
    test_gpu_drift.py, not asserted bit-exact here)."""
    g = SC.build_simulation(scene)
    o = P.build_oracle(scene)
    g.set_trace(trace)
    o.enable_trace(trace)
    worst = {"force_rel_err": 0.0, "vel_rel_err": 0.0, "pos_rel_err": 0.0, "finite_tti": 0}
    for _ in range(steps):
        if resync:
            P.resync(g, o)
        P.step_both(g, o, scene)
        if trace:
            r = P.compare_traces(g.read_trace(), o.read_trace())
            worst["force_rel_err"] = max(worst["force_rel_err"], r["force_rel_err"])
            worst["finite_tti"] += r["finite_tti"]
        r = P.compare_states(g.read_state(), o.read_state())
        worst["vel_rel_err"] = max(worst["vel_rel_err"], r["vel_rel_err"])
        worst["pos_rel_err"] = max(worst["pos_rel_err"], r["pos_rel_err"])
    return worst, g, o


def test_cell_assignment_bit_exact():
    rng = np.random.default_rng(7)
    for (w, h, c, off) in [(164.0, 164.0, 2.0, (-32.0, -32.0)), (10.0, 10.0, 0.5, (0.0, 0.0)),
                           (4.0, 8.0, 1.0, (0.0, 0.0)), (8.0, 4.0, 1.0, (0.0, 0.0)),
                           (100.0, 100.0, 0.3, (-7.7, 13.1))]:
        xy = np.concatenate([
            rng.uniform(off[0] - 5, off[0] + w + 5, size=(4000, 1)),
            rng.uniform(off[1] - 5, off[1] + h + 5, size=(4000, 1))], axis=1)
        # exact cell boundaries and specials
        edge = np.array([[off[0], off[1]], [off[0] + w, off[1] + h], [off[0] + c, off[1] + 3 * c],
                         [np.nan, 1.0], [1.0, np.inf], [-np.inf, 1.0], [off[0] - 1e-300, off[1]],
                         [off[0] + w - 1e-12, off[1] + h - 1e-12]])
        xy = np.concatenate([xy, edge])
        g = R.LocationHash2D(w, h, c, off, capacity=16)
        o = O.OracleSim(w, h, c, off)
        assert np.array_equal(g.cell_of(xy), o.cell_of(xy))


def test_c1_viz_scene_matches_oracle_every_step():
    scene = SC.config_c1()
    worst, g, o = _run(scene, 400)
    assert worst["finite_tti"] > 0  # the interaction at step 301.. is exercised
    assert worst["force_rel_err"] <= P.REL_TOL
    assert worst["vel_rel_err"] <= P.REL_TOL and worst["pos_rel_err"] <= P.REL_TOL


@pytest.mark.parametrize("variant", ["shuffled", "lane"])
def test_small_uniform_crowd(variant):
    scene = SC.uniform_crowd(32, variant, margin=16.0, seed=3)
    worst, g, o = _run(scene, 3)
    if variant == "shuffled":
        assert worst["finite_tti"] > 0
    assert worst["force_rel_err"] <= P.REL_TOL
    assert worst["vel_rel_err"] <= P.REL_TOL and worst["pos_rel_err"] <= P.REL_TOL


def test_c2_10k_one_step_and_stats():
    scene = SC.config_c2("shuffled")
    worst, g, o = _run(scene, 2)
    assert worst["force_rel_err"] <= P.REL_TOL
    assert worst["vel_rel_err"] <= P.REL_TOL and worst["pos_rel_err"] <= P.REL_TOL
    st = g.stats()
    tr = o.read_trace()
    assert st.neighbour_total == int(tr["nb_offsets"][-1])
    assert st.finite_tti_count == int(np.isfinite(tr["t_i"]).sum())
    assert st.oob_count == 0


def test_wide_stencil_and_mixed_groups():
    """cell < R (11 x 11 stencil as in the viz scene), two groups with different eyesight and planners,
    positions left of / below the grid origin (insert cell saturates to 0, query floors)."""
    rng = np.random.default_rng(11)
    w = h = 40.0
    off = (-5.0, -5.0)
    o = O.OracleSim(w, h, 1.0, off)
    g = R.Simulation(R.LocationHash2D(w, h, 1.0, off, capacity=4096))
    # jittered lattices (no pair inside agent_radius: the model turns overlaps into 1e15 forces)
    lat = SC.jittered_lattice(30, 30, 1.2, 21) - 7.0          # spans [-7, 29]: some agents left of / below the origin
    sel = rng.permutation(900)
    xy_a = lat[sel[:600]]
    xy_b = lat[sel[600:]] + 0.37
    za = (0.3, 1.0, 0.0, 0.7, 1.5, 0.25)
    oa = o.add_agents(xy_a, o.hl_parity((0.8, 0.3)), o.lp_zanlungo(*za), 4.5)
    ob = o.add_agents(xy_b, o.hl_constant((0.1, -0.4)), o.lp_none(), 2.0)
    ga = g.add_agents(xy_a, R.ParityVelocityPlan((0.8, 0.3)), R.Zanlungo(*za), 4.5)
    gb = g.add_agents(xy_b, R.ConstantVelocityPlan((0.1, -0.4)), R.NoLocalPlan(), 2.0)
    assert list(oa) == ga and list(ob) == gb
    v = rng.uniform(-0.5, 0.5, size=(900, 2))
    ids = np.arange(900, dtype=np.uint64)
    allxy = np.concatenate([xy_a, xy_b])
    o.set_state(ids, allxy[:, 0], allxy[:, 1], v[:, 0], v[:, 1])
    g.set_state(ids, allxy[:, 0], allxy[:, 1], v[:, 0], v[:, 1])
    g.set_trace(True)
    o.enable_trace(True)
    for _ in range(2):
        P.resync(g, o)
        g.step(R.Duration(0, 10_000_000))
        o.step(0, 10_000_000)
        tg, to = g.read_trace(), o.read_trace()
        # the oracle also runs (and traces) the radius query of NoLocalPlan agents, whose result cannot
        # influence anything (no_local_plan.rs:10-17); the CUDA path skips it: compare the Zanlungo group
        keep = tg["id"] < 600
        r = P.compare_traces(P.csr_subset(tg, keep), P.csr_subset(to, keep))
        assert r["force_rel_err"] <= P.REL_TOL and r["neighbours"] > 0
        s = P.compare_states(g.read_state(), o.read_state())
        assert s["vel_rel_err"] <= P.REL_TOL and s["pos_rel_err"] <= P.REL_TOL


def test_crowded_cells_use_the_block_sorter():
    """> 32 agents in one cell exercises sort_big_cells_kernel; order must still be canonical.
    15 x 15 agents at 0.25 m spacing in 2 x 2 cells of 2 m; agent_radius 0.05 so nobody overlaps."""
    rng = np.random.default_rng(5)
    scene = SC.uniform_crowd(15, "shuffled", s=0.25, margin=8.0, seed=2,
                             lp=("zanlungo", 0.01, 1.0, 0.0, 0.5, 1.0, 0.05))
    scene.vxy = rng.uniform(-0.2, 0.2, size=(225, 2))
    worst, g, o = _run(scene, 2)
    assert worst["finite_tti"] > 0
    assert worst["force_rel_err"] <= P.REL_TOL and worst["vel_rel_err"] <= P.REL_TOL


@pytest.mark.parametrize("lower_id_on_the_right", [True, False])
def test_overlapping_agents_behave_identically(lower_id_on_the_right):
    """Two agents inside each other's agent_radius: t_i = 0 => 1e15-magnitude tangential force for the
    lower id (zanlungo.rs:64-66,165-167).  Pushed towards +y the new position fails location_to_index
    => Err("Index out of bounds") from both implementations and the CUDA state stays the pre-step
    snapshot; pushed towards -y the saturating cast (location_hash_2d.rs:57) files the agent in row 0
    and NO error is raised -- by either implementation."""
    z = (0.05, 1.0, 0.0, 0.5, 1.0, 0.2)
    xy = np.array([[5.1, 5.0], [5.0, 5.0], [8.0, 8.0]]) if lower_id_on_the_right else \
        np.array([[5.0, 5.0], [5.1, 5.0], [8.0, 8.0]])
    g = R.Simulation(R.LocationHash2D(16, 16, 2.0, (0.0, 0.0), capacity=8))
    g.add_agents(xy, R.ParityVelocityPlan((1.0, 0.0)), R.Zanlungo(*z), 2.0)
    o = O.OracleSim(16, 16, 2.0, (0.0, 0.0))
    o.add_agents(xy, o.hl_parity((1.0, 0.0)), o.lp_zanlungo(*z), 2.0)
    # first step: velocities are 0 => a = 0 => t_i = inf (SURVEY.md section 9); the second step interacts
    g.step(R.Duration(0, 1_000_000))
    o.step(0, 1_000_000)
    P.resync(g, o)
    before = g.read_state()
    err_o = err_g = None
    try:
        o.step(0, 16_666_667)
    except O.OracleError as e:
        err_o = str(e)
    try:
        g.step(R.Duration(0, 16_666_667))
    except R.CrowdsimError as e:
        err_g = str(e)
    assert err_o == err_g
    after = g.read_state()
    if err_o is not None:
        assert err_o == "Index out of bounds"
        for k in ("x", "y", "vx", "vy"):
            assert np.array_equal(before[k].view(np.uint64), after[k].view(np.uint64))
        assert g.stats().first_oob_id == 0
    else:
        so = o.read_state()
        assert abs(so["vy"][0]) > 1e14  # the 1e15 cap was hit
        s = P.compare_states(after, so)
        assert s["vel_rel_err"] <= P.REL_TOL and s["pos_rel_err"] <= P.REL_TOL
        assert g.spatial_index.cell_of(np.stack([after["x"], after["y"]], axis=1))[0] >= 0


def test_host_planner_slow_path_matches_oracle_table_planner():
    class Swirl(R.HighLevelPlanner):
        def get_desired_velocity(self, agent, time):
            if agent.agent_id % 5 == 0:
                return None
            x, y = agent.position
            return (-0.1 * y, 0.1 * x)

    rng = np.random.default_rng(3)
    xy = SC.jittered_lattice(18, 18, 0.9, 8)[rng.permutation(324)[:300]] + 2.0
    z = (0.05, 1.0, 0.0, 0.5, 1.0, 0.2)
    g = R.Simulation(R.LocationHash2D(24, 24, 2.0, (-2.0, -2.0), capacity=512))
    g.add_agents(xy, Swirl(), R.Zanlungo(*z), 2.0)
    o = O.OracleSim(24, 24, 2.0, (-2.0, -2.0))
    hl = o.hl_host()
    o.add_agents(xy, hl, o.lp_zanlungo(*z), 2.0)
    for _ in range(3):
        P.resync(g, o)
        so = o.read_state()
        sel = so["id"] % 5 != 0
        vxy = np.stack([-0.1 * so["y"][sel], 0.1 * so["x"][sel]], axis=1)
        o.set_preferred_velocity(hl, so["id"][sel], vxy)
        o.step(0, 50_000_000)
        g.step(R.Duration(0, 50_000_000))
        s = P.compare_states(g.read_state(), o.read_state())
        assert s["vel_rel_err"] <= P.REL_TOL and s["pos_rel_err"] <= P.REL_TOL


def test_remove_agents_then_step():
    scene = SC.uniform_crowd(16, "shuffled", margin=8.0, seed=9)
    g = SC.build_simulation(scene)
    o = P.build_oracle(scene)
    for i in (3, 77, 200, 255, 0):
        g.remove_agents(i)
        o.remove_agent(i)
    assert g.agent_count() == o.agent_count() == 251
    for _ in range(2):
        P.resync(g, o)
        P.step_both(g, o, scene)
        s = P.compare_states(g.read_state(), o.read_state())
        assert s["vel_rel_err"] <= P.REL_TOL and s["pos_rel_err"] <= P.REL_TOL


def test_empty_simulation_steps():
    g = R.Simulation(R.LocationHash2D(10, 10, 1, (0, 0), capacity=4))
    g.step(R.Duration(1, 0))
    assert g.agent_count() == 0 and g.agents == {}


def test_results_do_not_depend_on_insertion_order():
    """Canonical (cell, id) summation order: the same crowd inserted in two different storage orders
    gives bit-identical per-id results."""
    scene = SC.uniform_crowd(24, "shuffled", margin=8.0, seed=4)
    a = SC.build_simulation(scene)
    # second handle: same ids, storage order reversed, through the explicit-id entry point
    from rmf_crowdsim_b200 import _native as N

    b = R.Simulation(R.LocationHash2D(scene.width, scene.height, scene.cell, scene.offset, capacity=scene.n))
    hl = R.ParityVelocityPlan(scene.hl[1])
    lp = R.Zanlungo(*scene.lp[1:])
    ids = np.arange(scene.n, dtype=np.uint64)[::-1].copy()
    xy = scene.xy[::-1].copy()
    vxy = scene.vxy[::-1].copy()
    N.check(b._h, b._lib.rcs_dist_add_agents(b._h, scene.n, ids.ctypes.data_as(N.c_u64p),
                                             xy.ctypes.data_as(N.c_f64p), vxy.ctypes.data_as(N.c_f64p),
                                             b._hl(hl), b._lp(lp), scene.eyesight))
    for _ in range(3):
        a.step(R.Duration(*scene.dt))
        b.step(R.Duration(*scene.dt))
    sa, sb = a.read_state(), b.read_state()
    for k in ("id", "x", "y", "vx", "vy"):
        assert np.array_equal(sa[k].view(np.uint64), sb[k].view(np.uint64)), k


@pytest.mark.parametrize("variant", ["shuffled", "lane"])
def test_warp_cooperative_kernel_is_bit_identical_to_thread_per_agent(variant):
    """The three forms of the hot kernel (rcs_kernels.cuh step_kernel, rcs_step_warp.cuh step_warp_kernel through
    L1, rcs_step_tile.cuh step_tile_kernel with the stencil staged in shared memory) evaluate the same operations
    in the same canonical order: every output bit must agree."""
    from rmf_crowdsim_b200 import _native as N

    scene = SC.uniform_crowd(96, variant, margin=16.0, seed=6)
    sims = []
    for kern in (1, 2, 3):
        g = SC.build_simulation(scene)
        g.set_option(N.RCS_OPT_STEP_KERNEL, kern)
        g.set_trace(True)
        sims.append(g)
    for _ in range(3):
        for g in sims:
            g.step(R.Duration(*scene.dt))
        ta, sa = sims[0].read_trace(), sims[0].read_state()
        for other in sims[1:]:
            tb, sb = other.read_trace(), other.read_state()
            for k in ("id", "nb_offsets", "nb_ids"):
                assert np.array_equal(ta[k], tb[k]), k
            for k in ("t_i", "fx", "fy"):
                assert np.array_equal(ta[k].view(np.uint64), tb[k].view(np.uint64)), k
            for k in ("x", "y", "vx", "vy"):
                assert np.array_equal(sa[k].view(np.uint64), sb[k].view(np.uint64)), k
    for other in sims[1:]:
        assert sims[0].stats().neighbour_total == other.stats().neighbour_total
        assert sims[0].stats().candidate_total == other.stats().candidate_total


@pytest.mark.parametrize("cell,eyesight,s", [
    (1.0, 2.0, 1.0),    # 5 stencil columns: two rounds of chunks
    (0.5, 2.2, 1.0),    # 9-10 columns, mostly empty cells
    (4.0, 2.0, 0.5),    # 64 agents per cell: up to 4 chunks per column, 3 columns
    (8.0, 3.0, 1.0),    # coarse cells, 64-128 candidates per column
    (3.0, 2.0, 1.0),    # mixed: some agents fit the three-slice path, some do not
])
def test_wide_and_crowded_stencils_are_bit_identical_to_thread_per_agent(cell, eyesight, s):
    """step_aside_kernel (chunked stencil columns, two passes) against the sequential routine of step_kernel: same
    neighbour lists, t_i, forces, state, statistics -- every bit."""
    from rmf_crowdsim_b200 import _native as N

    rng = np.random.default_rng(17)
    scene = SC.uniform_crowd(72, "shuffled", s=s, cell=cell, eyesight=eyesight, margin=16.0, seed=9,
                             lp=("zanlungo", 0.05, 1.0, 0.0, 0.5, 50.0, 0.05))  # heavy agents: the crowd stays sane
    scene.vxy = scene.vxy + rng.uniform(-0.3, 0.3, size=scene.vxy.shape)
    scene.dt = (0, 10_000_000)
    sims = []
    for kern in (1, 0):
        g = SC.build_simulation(scene)
        g.set_option(N.RCS_OPT_STEP_KERNEL, kern)
        g.set_trace(True)
        sims.append(g)
    finite = 0
    for _ in range(2):
        for g in sims:
            g.step(R.Duration(*scene.dt))
        ta, tb = sims[0].read_trace(), sims[1].read_trace()
        for k in ("id", "nb_offsets", "nb_ids"):
            assert np.array_equal(ta[k], tb[k]), k
        for k in ("t_i", "fx", "fy"):
            assert np.array_equal(ta[k].view(np.uint64), tb[k].view(np.uint64)), k
        finite += int(np.isfinite(ta["t_i"]).sum())
        sa, sb = sims[0].read_state(), sims[1].read_state()
        for k in ("x", "y", "vx", "vy"):
            assert np.array_equal(sa[k].view(np.uint64), sb[k].view(np.uint64)), k
    assert finite > 100
    sta, stb = sims[0].stats(), sims[1].stats()
    assert sta.neighbour_total == stb.neighbour_total and sta.candidate_total == stb.candidate_total
    assert sta.finite_tti_count == stb.finite_tti_count


def test_more_oversized_cells_than_the_big_cell_list_holds():
    """4900 cells with 40 agents each (> 32 per cell, > 4096 such cells): the block sorter sweeps all cells and
    storage order is still canonical (cell, then ascending id)."""
    rng = np.random.default_rng(3)
    side, per = 70, 40
    cell = 4.0
    cx, cy = np.meshgrid(np.arange(side), np.arange(side), indexing="ij")
    base = np.stack([cx.reshape(-1), cy.reshape(-1)], axis=1).astype(np.float64) * cell
    xy = (base[:, None, :] + rng.uniform(0.05, cell - 0.05, size=(side * side, per, 2))).reshape(-1, 2)
    xy = xy[rng.permutation(len(xy))]
    idx = R.LocationHash2D(side * cell, side * cell, cell, (0.0, 0.0), capacity=len(xy))
    sim = R.Simulation(idx)
    sim.add_agents(xy, R.ConstantVelocityPlan((0.0, 0.0)), R.Zanlungo(0.05, 1.0, 0.0, 0.5, 1.0, 0.01), 0.05)
    sim.step(R.Duration(0, 1_000_000))
    st = sim.read_state(order=R._native.RCS_ORDER_STORAGE)
    cells = idx.cell_of(np.stack([st["x"], st["y"]], axis=1))
    key = cells.astype(np.uint64) * np.uint64(1 << 32) + st["id"]
    assert np.all(key[1:] > key[:-1])
    assert len(st["id"]) == len(xy) and sim.stats().oob_count == 0


def test_one_cell_larger_than_the_sorters_shared_memory_tile():
    """9500 agents in one cell (> BIG_SMEM_KEYS = 4096: ranks accumulate over three key tiles) next to ordinary
    cells -- the shape of cell 0 once a crowd has gone non-finite.  Storage order is still (cell, ascending id)."""
    rng = np.random.default_rng(4)
    cell = 50.0
    big = rng.uniform(0.5, cell - 0.5, size=(9500, 2))
    rest = rng.uniform(cell + 1.0, 4 * cell - 1.0, size=(3000, 2))
    xy = np.concatenate([big, rest])
    xy = xy[rng.permutation(len(xy))]
    idx = R.LocationHash2D(4 * cell, 4 * cell, cell, (0.0, 0.0), capacity=len(xy))
    sim = R.Simulation(idx)
    sim.add_agents(xy, R.ConstantVelocityPlan((0.0, 0.0)), R.Zanlungo(0.05, 1.0, 0.0, 0.5, 1.0, 0.01), 0.05)
    for _ in range(2):
        sim.step(R.Duration(0, 1_000_000))
    st = sim.read_state(order=R._native.RCS_ORDER_STORAGE)
    cells = idx.cell_of(np.stack([st["x"], st["y"]], axis=1))
    key = cells.astype(np.uint64) * np.uint64(1 << 32) + st["id"]
    assert np.all(key[1:] > key[:-1])
    assert np.array_equal(np.sort(st["id"]), np.arange(len(xy), dtype=np.uint64))


def test_agents_with_non_finite_positions_pile_up_in_cell_0_and_see_nobody():
    """NaN / inf positions are filed in cell 0 by the reference (`NaN as usize` = 0) and can have no neighbour (no d2
    passes the strict `<`); the cooperative kernels skip their query.  Same state, neighbour lists and statistics
    as the thread-per-agent kernel, and the finite part of the crowd is unaffected."""
    from rmf_crowdsim_b200 import _native as N

    scene = SC.uniform_crowd(64, "shuffled", margin=16.0, seed=12)
    rng = np.random.default_rng(8)
    bad = rng.choice(scene.n, size=400, replace=False).astype(np.uint64)
    sims = []
    for kern in (1, 0):
        g = SC.build_simulation(scene)
        g.set_option(N.RCS_OPT_STEP_KERNEL, kern)
        g.set_trace(True)
        x = scene.xy[bad.astype(np.int64), 0].copy()
        y = scene.xy[bad.astype(np.int64), 1].copy()
        x[:200] = np.nan
        y[100:300] = -np.inf   # (+inf would saturate the insert cell and fail the step: "Index out of bounds")
        x[300:] = -np.inf
        g.set_state(bad, x=x, y=y)
        sims.append(g)
    for _ in range(2):
        for g in sims:
            g.step(R.Duration(*scene.dt))
        ta, tb = sims[0].read_trace(), sims[1].read_trace()
        for k in ("id", "nb_offsets", "nb_ids"):
            assert np.array_equal(ta[k], tb[k]), k
        for k in ("t_i", "fx", "fy"):
            assert np.array_equal(ta[k].view(np.uint64), tb[k].view(np.uint64)), k
        sa, sb = sims[0].read_state(), sims[1].read_state()
        for k in ("x", "y", "vx", "vy"):
            assert np.array_equal(np.isnan(sa[k]), np.isnan(sb[k])), k
            ok = ~np.isnan(sa[k])
            assert np.array_equal(sa[k][ok].view(np.uint64), sb[k][ok].view(np.uint64)), k
    sta, stb = sims[0].stats(), sims[1].stats()
    assert sta.neighbour_total == stb.neighbour_total and sta.candidate_total == stb.candidate_total
    assert sta.nonfinite_count == stb.nonfinite_count == 400


@pytest.mark.parametrize("n_side", [31, 64])
def test_streaming_kernel_of_no_local_plan_crowds_matches_the_generic_kernel_and_the_oracle(n_side):
    """NoLocalPlan-only crowds take step_stream_kernel (two agents per thread, no index): same bits as the
    thread-per-agent kernel and as the oracle (only IEEE mul/add are involved); odd agent counts hit the tail."""
    scene = SC.uniform_crowd(n_side, "shuffled", margin=8.0, seed=6, lp=("none",))
    a = SC.build_simulation(scene)
    b = SC.build_simulation(scene)
    b.set_option(R._native.RCS_OPT_STEP_KERNEL, 1)
    o = P.build_oracle(scene)
    # a host-evaluated planner for half of the agents (None for a few of them)
    for _ in range(5):
        P.step_both(a, o, scene)
        b.step(R.Duration(*scene.dt))
    sa, sb, so = a.read_state(), b.read_state(), o.read_state()
    for k in ("x", "y", "vx", "vy"):
        assert np.array_equal(sa[k].view(np.uint64), sb[k].view(np.uint64)), k
        assert np.array_equal(sa[k].view(np.uint64), so[k].view(np.uint64)), k
    assert a.launch_count() < b.launch_count() + 100  # both ran; no index was built on either path

