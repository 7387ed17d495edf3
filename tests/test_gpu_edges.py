"""GPU: edge cases of the C ABI -- capacities, unknown ids, empty and ragged inputs, degenerate grids (the
reference's width-stride aliasing), non-finite state, zero time steps -- each against the oracle where the
reference defines a behaviour."""
import ctypes as C

import numpy as np
import pytest

import oracle_ffi as O
import parity as P
import rmf_crowdsim_b200 as R
from rmf_crowdsim_b200 import _native as N

pytestmark = pytest.mark.gpu


def test_capacity_is_enforced_on_add_and_on_spawn():
    sim = R.Simulation(R.LocationHash2D(100.0, 100.0, 2.0, (0.0, 0.0), capacity=4))
    hl, lp = R.ConstantVelocityPlan((1.0, 0.0)), R.NoLocalPlan()
    sim.add_agents([(1.0, 1.0), (2.0, 2.0), (3.0, 3.0)], hl, lp, 1.0)
    with pytest.raises(R.CrowdsimError) as e:
        sim.add_agents([(4.0, 4.0), (5.0, 5.0)], hl, lp, 1.0)
    assert e.value.code == N.RCS_ERR_CAPACITY and sim.agent_count() == 3
    # a source that keeps spawning into a full handle: the failing step is reported and not committed
    sim.add_source_sink(R.SourceSink((50.0, 50.0), 1.0, R.MonotonicCrowd(1.0), hl, lp, [(90.0, 50.0)], False, 1.0))
    sim.step(R.Duration(1, 0))  # 4th agent fits
    assert sim.agent_count() == 4
    before = sim.read_state()
    with pytest.raises(R.CrowdsimError) as e:
        sim.step(R.Duration(1, 0))
    assert e.value.code == N.RCS_ERR_CAPACITY
    after = sim.read_state()
    assert np.array_equal(np.sort(before["x"]), np.sort(after["x"]))


def test_unknown_ids_are_errors_and_leave_the_state_alone():
    sim = R.Simulation(R.LocationHash2D(10.0, 10.0, 1.0, (0.0, 0.0), capacity=8))
    ids = sim.add_agents([(1.0, 1.0), (2.0, 2.0)], R.ConstantVelocityPlan((0.0, 0.0)), R.NoLocalPlan(), 1.0)
    with pytest.raises(R.CrowdsimError):
        sim.remove_agents(77)
    with pytest.raises(R.CrowdsimError):
        sim.set_state([5], x=[1.0], y=[1.0])
    with pytest.raises(R.CrowdsimError) as e:
        sim.set_state([ids[0]], x=[50.0], y=[1.0])  # add_or_update would reject it (location_hash_2d.rs:126-130)
    assert str(e.value) == "Index out of bounds"
    assert sim.agent_count() == 2
    sim.spatial_index.remove_agent(12345)  # SpatialIndex::remove_agent of an unknown id is a no-op (:260-267)
    assert sim.agent_count() == 2
    for option in (2, 4):  # retired option numbers are unknown options, whatever the value
        for value in (0, 1):
            with pytest.raises(R.CrowdsimError) as e:
                sim.set_option(option, value)
            assert e.value.code == N.RCS_ERR_ARG and str(e.value) == "unknown option or value"
    steps = sim.stats().steps
    sim.step(R.Duration(1, 0))
    assert sim.stats().steps == steps + 1 and sim.agent_count() == 2


def test_empty_and_ragged_batches():
    idx = R.LocationHash2D(10.0, 10.0, 1.0, (0.0, 0.0), capacity=8)
    off, ids = idx.query_radius(np.zeros((0, 2)), np.zeros(0))
    assert len(off) == 1 and len(ids) == 0
    got, cnt = idx.query_knn(np.zeros((0, 2)), 3)
    assert got.shape[0] == 0
    assert len(idx.cell_of(np.zeros((0, 2)))) == 0
    idx.add_or_update_many(np.array([3, 1, 2], dtype=np.uint64), np.array([[0.5, 0.5], [0.6, 0.5], [5.5, 5.5]]))
    # ragged CSR: queries with 2, 0 and 1 hits; ids inside a cell come back in ascending order
    off, ids = idx.query_radius(np.array([[0.5, 0.5], [8.5, 1.5], [5.4, 5.4]]), np.array([0.3, 0.3, 0.3]))
    assert list(off) == [0, 2, 2, 3] and list(ids) == [1, 3, 2]
    sim = R.Simulation(idx)
    sim.step(R.Duration(0, 0))  # index-only handle: agents without planners do not move (lib.rs:263-292)


@pytest.mark.parametrize("w,h", [(12.0, 6.0), (6.0, 12.0)])
def test_non_square_grids_keep_the_reference_aliasing(w, h):
    """idx = x_idx * n_x + y_idx with the WIDTH cell count as stride (location_hash_2d.rs:59): with n_x > n_y large x
    is out of bounds although it lies inside the rectangle, with n_y > n_x rows alias into the next column."""
    rng = np.random.default_rng(int(w))
    o = O.OracleSim(w, h, 1.0, (0.0, 0.0))
    g = R.LocationHash2D(w, h, 1.0, (0.0, 0.0), capacity=512)
    pts = rng.uniform([0.0, 0.0], [w, h], size=(400, 2))
    cells = o.cell_of(pts)
    assert np.array_equal(g.cell_of(pts), cells)
    ok = cells >= 0
    assert (~ok).any() or w < h  # the wide grid rejects points inside its own rectangle
    pts, ids = pts[ok], np.arange(int(ok.sum()), dtype=np.uint64)
    g.add_or_update_many(ids, pts)
    for i, p in zip(ids, pts):
        o.index_add_or_update(int(i), p)
    q = rng.uniform([-1.0, -1.0], [w + 1, h + 1], size=(60, 2))
    off, got = g.query_radius(q, np.full(len(q), 1.7))
    for k in range(len(q)):
        # the canonical order sorts every data cell by id; an aliased cell is visited where the reference visits it
        assert list(got[int(off[k]):int(off[k + 1])]) == list(o.query_radius(1.7, q[k])), k


def test_zero_dt_and_nan_state_behave_like_the_reference():
    scene_xy = np.array([[10.0, 10.0], [10.5, 10.0], [30.0, 30.0]])
    o = O.OracleSim(64.0, 64.0, 2.0, (0.0, 0.0))
    g = R.Simulation(R.LocationHash2D(64.0, 64.0, 2.0, (0.0, 0.0), capacity=8))
    za = (0.05, 1.0, 0.0, 0.5, 1.0, 0.2)
    o.add_agents(scene_xy, o.hl_parity((1.3, 0.0)), o.lp_zanlungo(*za), 2.0)
    g.add_agents(scene_xy, R.ParityVelocityPlan((1.3, 0.0)), R.Zanlungo(*za), 2.0)
    v = np.array([[-1.3, 0.0], [1.3, 0.0], [0.0, 0.0]])
    ids = np.arange(3, dtype=np.uint64)
    o.set_state(ids, scene_xy[:, 0], scene_xy[:, 1], v[:, 0], v[:, 1])
    g.set_state(ids, scene_xy[:, 0], scene_xy[:, 1], v[:, 0], v[:, 1])
    g.step(R.Duration(0, 0))  # dt = 0: velocities are planned, positions stay
    o.step(0, 0)
    r = P.compare_states(g.read_state(), o.read_state())
    assert r["pos_rel_err"] == 0.0 and r["vel_rel_err"] <= P.REL_TOL
    # a NaN position is filed under cell 0 by the index (saturating cast of NaN, location_hash_2d.rs:56-57) and
    # stays NaN; that is not an error in the reference, only counted here
    so = o.read_state()
    x = so["x"].copy()
    x[2] = np.nan
    o.set_state(ids, x, so["y"], so["vx"], so["vy"])
    g.set_state(None, x, so["y"], so["vx"], so["vy"])
    for _ in range(2):
        g.step(R.Duration(0, 100_000_000))
        o.step(0, 100_000_000)
    a, b = g.read_state(), o.read_state()
    assert np.isnan(a["x"][2]) and np.isnan(b["x"][2])
    assert np.allclose(a["x"][:2], b["x"][:2], rtol=1e-9) and np.allclose(a["y"], b["y"], rtol=1e-9)
    assert g.stats().nonfinite_count == 1 and g.stats().oob_count == 0


def test_async_read_back_returns_the_same_bits_as_the_blocking_read():
    from rmf_crowdsim_b200 import scenes as SC

    scene = SC.uniform_crowd(40, "lane", margin=8.0, seed=2)
    sim = SC.build_simulation(scene)
    lib, h, n = sim._lib, sim._h, scene.n
    bufs = [np.zeros(n) for _ in range(4)]
    ids = np.zeros(n, dtype=np.uint64)
    out_n = C.c_uint64()
    for step in range(3):
        sim.step_async(R.Duration(*scene.dt))
        N.check(h, lib.rcs_read_agents_async(h, N.RCS_ORDER_ID, n, ids.ctypes.data_as(N.c_u64p),
                                             *[b.ctypes.data_as(N.c_f64p) for b in bufs], C.byref(out_n)))
        sim.step_async(R.Duration(*scene.dt))  # enqueued while the copies of the previous step may still run
        N.check(h, lib.rcs_read_wait(h))
        snap = [b.copy() for b in bufs]
        # the blocking read now sees the state one step later; rewind by comparing with a second simulation
        ref = SC.build_simulation(scene)
        for _ in range(2 * step + 1):
            ref.step(R.Duration(*scene.dt))
        st = ref.read_state()
        assert out_n.value == n and np.array_equal(ids, st["id"])
        for b, k in zip(snap, ("x", "y", "vx", "vy")):
            assert np.array_equal(b.view(np.uint64), st[k].view(np.uint64)), (step, k)
