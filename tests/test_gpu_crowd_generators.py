"""GPU: PoissonCrowd (keyed draw, include/rcs.h) and user-implemented CrowdGenerators in source sinks -- decisions
against the numpy pin, parity with the oracle, reproducibility, CUDA graphs, strips, refusals and the host-count
contract."""

import numpy as np
import pytest

import oracle_crowd_generators as G
import parity as P
import rmf_crowdsim_b200 as R
from rmf_crowdsim_b200 import _native as N
from rmf_crowdsim_b200 import scenes as SC
from rmf_crowdsim_b200.strips import LocalStripGroup

pytestmark = pytest.mark.gpu

DT = R.Duration(0, 100_000_000)


class Rec(R.EventListener):
    def __init__(self):
        self.added, self.removed = [], []

    def agent_spawned(self, position, agent):
        self.added.append((agent, position))

    def agent_destroyed(self, agent):
        self.removed.append(agent)


class PatternCrowd(R.CrowdGenerator):
    """A stateful user generator: the k-th call returns pattern[k % len(pattern)]; every call is logged."""

    def __init__(self, pattern, log=None, tag=None):
        self.pattern, self.calls, self.log, self.tag = list(pattern), 0, log, tag

    def get_number_to_spawn(self, time_elapsed):
        c = self.pattern[self.calls % len(self.pattern)]
        self.calls += 1
        if self.log is not None:
            self.log.append((self.tag, time_elapsed))
        return c


def _decisions(specs, n_steps, dt):
    """[step, source] -> the numpy-pinned PoissonCrowd decision (counters (k + 1, sid) for k = 0 .. n_steps - 1)."""
    out = np.zeros((n_steps, len(specs)), dtype=bool)
    for sid, (rate, seed) in enumerate(specs):
        bg = np.random.Philox(key=np.array([seed, 0], dtype=np.uint64), counter=np.array([0, sid, 0, 0], dtype=np.uint64))
        w0 = bg.random_raw(4 * n_steps)[::4]
        out[:, sid] = (w0 >> np.uint64(11)) >= np.uint64(G.threshold(dt * rate))
    return out


def _fast_stream(specs, capacity=1 << 15, graphs=1):
    """One source per row at x = 5, agents at 10 m/s (1 m per 0.1 s step: out of the 0.4 m probe within one step), sinks
    at x = 250: the probe never blocks, so the spawns are exactly the generators' decisions.  specs: (rate, seed) of
    PoissonCrowd, or a CrowdGenerator."""
    g = R.Simulation(R.LocationHash2D(256.0, 256.0, 2.0, (0.0, 0.0), capacity=capacity))
    g.set_option(N.RCS_OPT_GRAPHS, graphs)
    g._keep = []
    for k, sp in enumerate(specs):
        gen = R.PoissonCrowd(*sp) if isinstance(sp, tuple) else sp
        hl, lp = R.ConstantVelocityPlan((10.0, 0.0)), R.NoLocalPlan()
        g._keep.append((hl, lp))
        g.add_source_sink(R.SourceSink((5.0, 2.0 + 3.0 * k), 2.0, gen, hl, lp, [(250.0, 2.0 + 3.0 * k)], False, 1.0))
    return g


def _row(p):
    return int(round((p[1] - 2.0) / 3.0))


def _mixed_specs(n=64, seed=1):
    rng = np.random.default_rng(seed)
    rates = [0.5, 2.0, 5.0, 10.0, 30.0]
    return [(rates[k % len(rates)], int(rng.integers(0, 1 << 63)) * 2 + (k & 1)) for k in range(n)]


def test_spawns_are_the_numpy_pinned_decisions():
    specs = _mixed_specs(64)
    n_steps = 220
    want = _decisions(specs, n_steps, DT.as_secs_f64())
    g = _fast_stream(specs)
    rec = Rec()
    g.add_event_listener(rec)
    for k in range(n_steps):
        assert g.stats().steps == k
        rec.added.clear()
        g.step(DT)
        got = sorted(_row(p) for _, p in rec.added)
        assert got == list(np.nonzero(want[k])[0]), k
    assert want.sum() > 3000 and (~want).sum() > 3000


def _ring_specs(n_sources, seed):
    rng = np.random.default_rng(seed)
    specs = []
    for k in range(n_sources):
        ang = 2 * np.pi * k / n_sources
        src = (20.0 * np.cos(ang), 20.0 * np.sin(ang))
        mid = (float(rng.uniform(-1.5, 1.5)), float(rng.uniform(-1.5, 1.5)))
        dst = (-src[0], -src[1])
        specs.append((src, [mid, dst], ((dst[0] - src[0]) / 40.0 * 1.5, (dst[1] - src[1]) / 40.0 * 1.5), False,
                      k % 3))
    return specs


def _lane_specs():
    """The overtaking lanes of test_gpu_source_sink._pair (Monotonic: an irregular spawn order breaks the overtaking
    pair's id order, and the reference model drives it non-finite within a few steps), a Poisson and a host lane."""
    return [((-20.0, 0.0), [(0.0, 0.0), (20.0, 0.0)], (1.5, 0.0), True, 0),
            ((-20.0, 0.15), [(0.0, 0.15), (20.0, 0.15)], (1.0, 0.0), True, 0),
            ((-20.0, 12.0), [(0.0, 12.0), (20.0, 12.0)], (1.0, 0.0), True, 1),
            ((-20.0, -12.0), [(0.0, -12.0), (20.0, -12.0)], (1.0, 0.0), True, 2)]


PATTERN = [1, 0, 0, 2, 1, 0, 1]


def _mixed_pair(specs, graphs=1, seed0=11):
    """The same source sinks in the oracle and on the device; kind 0: MonotonicCrowd, 1: PoissonCrowd, 2: a host
    generator."""
    w = h = 64.0
    off = (-32.0, -32.0)
    o = G.GenOracle(w, h, 2.0, off)
    g = R.Simulation(R.LocationHash2D(w, h, 2.0, off, capacity=4096))
    g.set_option(N.RCS_OPT_GRAPHS, graphs)
    za = (0.05, 1.0, 0.0, 0.5, 1.0, 0.2)
    keep, host = [], []
    for k, (src, wps, vel, zan, kind) in enumerate(specs):
        rate = 2.0
        seed = seed0 + 1000 * k
        ohl, olp = o.hl_constant(vel), (o.lp_zanlungo(*za) if zan else o.lp_none())
        sid = o.add_source_sink_gen(src, 3.0, kind, rate, seed, ohl, olp, wps, False, 2.0)
        gen = [R.MonotonicCrowd(rate), R.PoissonCrowd(rate, seed), PatternCrowd(PATTERN)][kind]
        ghl, glp = R.ConstantVelocityPlan(vel), (R.Zanlungo(*za) if zan else R.NoLocalPlan())
        keep.append((ghl, glp))
        assert g.add_source_sink(R.SourceSink(src, 3.0, gen, ghl, glp, wps, False, 2.0)) == sid
        if kind == 2:
            host.append(sid)
    g._keep = keep
    return g, o, host


def _oracle_step(o, host, step, dt):
    if host:
        o.set_spawn_counts(host, [PATTERN[step % len(PATTERN)]] * len(host))
    o.step(dt.secs, dt.nanos)


def _assert_same_state(g, o, exact):
    sg, so = g.read_state(), o.read_state()
    assert np.array_equal(sg["id"], so["id"])
    assert np.array_equal(sg["next_waypoint"].astype(np.uint64), so["next_waypoint"])
    if exact:
        for k in ("x", "y", "vx", "vy"):
            assert np.array_equal(sg[k].view(np.uint64), so[k].view(np.uint64)), k
    else:
        r = P.compare_states(sg, so)
        assert r["vel_rel_err"] <= P.REL_TOL and r["pos_rel_err"] <= P.REL_TOL


@pytest.mark.parametrize("zan", [False, True])
def test_mixed_generators_match_the_oracle(zan):
    specs = _lane_specs() if zan else _ring_specs(12, 3)
    g, o, host = _mixed_pair(specs)
    rec = Rec()
    g.add_event_listener(rec)
    dt = R.Duration(0, 500_000_000)
    despawned = 0
    for step in range(90):
        if zan and o.agent_count():
            P.resync(g, o)  # the Zanlungo force uses exp: the device's may differ from glibc's in the last bits
        rec.added.clear()
        rec.removed.clear()
        g.step(dt)
        _oracle_step(o, host, step, dt)
        s, sxy, d = o.poll_events()
        assert [a for a, _ in rec.added] == [int(v) for v in s], step
        assert [p for _, p in rec.added] == [tuple(v) for v in sxy.tolist()], step
        assert sorted(rec.removed) == sorted(int(v) for v in d), step
        despawned += len(d)
        assert g.stats().steps == o.steps() == step + 1
        _assert_same_state(g, o, exact=not zan)
    assert despawned > 0


def test_same_seed_same_run_other_seed_other_spawns_and_removal_keeps_the_other_draws():
    specs = _mixed_specs(16, seed=4)
    a, b = _fast_stream(specs), _fast_stream(specs)
    c = _fast_stream([(r, s ^ 0x5DEECE66D) for r, s in specs])
    d = _fast_stream(specs)
    recs = [Rec() for _ in range(4)]
    for sim, rec in zip((a, b, c, d), recs):
        sim.add_event_listener(rec)
    per_step = {id(r): [] for r in recs}
    for k in range(80):
        if k == 30:
            d.remove_source_sink(5)
        for sim, rec in zip((a, b, c, d), recs):
            rec.added.clear()
            sim.step(DT)
            per_step[id(rec)].append(sorted(_row(p) for _, p in rec.added))
    sa, sb = a.read_state(), b.read_state()
    for key in sa:
        assert np.array_equal(sa[key], sb[key]), key
    assert per_step[id(recs[0])] == per_step[id(recs[1])]
    assert per_step[id(recs[0])] != per_step[id(recs[2])]
    for k in range(80):
        full = per_step[id(recs[0])][k]
        assert per_step[id(recs[3])][k] == (full if k < 30 else [s for s in full if s != 5]), k


def _run_async(g, o, host, dts, oracle=True):
    for step, dt in enumerate(dts):
        g.step_async(dt)
        if oracle:
            _oracle_step(o, host, step, dt)
    g.sync()


def test_graphs_on_and_off_give_the_same_bits_and_replay_at_constant_dt():
    specs = _ring_specs(12, 5)
    (a, oa, ha), (b, _, _) = _mixed_pair(specs, graphs=1), _mixed_pair(specs, graphs=0)
    dts = [R.Duration(0, 500_000_000)] * 60
    _run_async(a, oa, ha, dts)
    _run_async(b, None, [], dts, oracle=False)
    sa, sb = a.read_state(), b.read_state()
    for key in sa:
        assert np.array_equal(sa[key].view(np.uint64) if sa[key].dtype == np.float64 else sa[key],
                              sb[key].view(np.uint64) if sb[key].dtype == np.float64 else sb[key]), key
    assert a.graph_stats()[0] > 0 and b.graph_stats() == (0, 0)
    _assert_same_state(a, oa, exact=True)


def test_dt_alternating_every_step_matches_the_oracle():
    g, o, host = _mixed_pair(_ring_specs(12, 6))
    rec = Rec()
    g.add_event_listener(rec)
    dts = [R.Duration(0, 500_000_000) if k % 2 == 0 else R.Duration(0, 300_000_000) for k in range(60)]
    _run_async(g, o, host, dts)
    g._dispatch_events()
    s, _, d = o.poll_events()
    assert [a for a, _ in rec.added] == [int(v) for v in s]
    assert sorted(rec.removed) == sorted(int(v) for v in d)
    assert g.stats().steps == o.steps() == 60
    _assert_same_state(g, o, exact=True)


def _stream_scene():
    return SC.Scene(name="stream", width=96.0, height=96.0, cell=2.0, offset=(0.0, 0.0), xy=np.zeros((0, 2)),
                    vxy=np.zeros((0, 2)), eyesight=2.0, hl=("constant", (0.0, 0.0)), lp=("none",), seed=0)


def _stream_makers():
    """Source sinks whose agents walk across the strip boundaries to sinks in other strips; Poisson and host
    generators alternate.  Every call of a maker returns fresh objects (one set per handle)."""
    makers = []
    for k, (x0, x1, y) in enumerate([(5.0, 85.0, 10.0), (85.0, 9.0, 20.0), (41.0, 90.0, 30.0), (53.0, 7.0, 40.0),
                                     (11.0, 70.0, 50.0), (75.0, 40.0, 60.0), (21.0, 50.0, 70.0), (89.0, 3.0, 80.0)]):
        v = (1.0 if x1 > x0 else -1.0, 0.0)

        def make(x0=x0, x1=x1, y=y, v=v, k=k):
            gen = R.PoissonCrowd(1.5, 77 + k) if k % 2 == 0 else PatternCrowd([1, 0, 1, 1, 0, 0, 2][k % 3:] + [1])
            return R.SourceSink((x0, y), 0.6, gen, R.ConstantVelocityPlan(v), R.NoLocalPlan(),
                                [((x0 + x1) / 2, y), (x1, y)], False, 2.0)
        makers.append(make)
    return makers


@pytest.mark.parametrize("world", [2, 3])
def test_strips_match_one_handle(world):
    scene = _stream_scene()
    single = SC.build_simulation(scene, capacity=4096)
    grp = LocalStripGroup(scene, world, capacity=4096, halo_capacity=1024)
    rec_s, rec_g = Rec(), Rec()
    single.add_event_listener(rec_s)
    grp.add_event_listener(rec_g)
    keep = []
    for make in _stream_makers():
        ss = make()
        keep.append(ss)
        single.add_source_sink(ss)
        grp.add_source_sink(make)
    dt = R.Duration(0, 500_000_000)
    for step in range(130):
        single.step(dt)
        grp.step(dt)
        grp.dispatch_events()
        if step % 10 == 9 or step > 120:
            sa, sb = single.read_state(), grp.read_state()
            assert np.array_equal(sa["id"], sb["id"]), step
            for k in ("x", "y", "vx", "vy"):
                assert np.array_equal(sa[k].view(np.uint64), sb[k].view(np.uint64)), (k, step)
            assert np.array_equal(sa["next_waypoint"], sb["next_waypoint"])
    assert sorted(rec_g.added) == sorted(rec_s.added) and len(rec_s.added) > 300
    assert sorted(rec_g.removed) == sorted(rec_s.removed) and len(rec_s.removed) > 50
    assert min(grp.agent_counts()) > 0


def test_zero_dt_with_a_poisson_source_is_refused_and_changes_nothing():
    specs = _ring_specs(12, 7)
    (g, o, host), (ref, _, _) = _mixed_pair(specs), _mixed_pair(specs)
    rec, rec_ref = Rec(), Rec()
    g.add_event_listener(rec)
    ref.add_event_listener(rec_ref)
    dt = R.Duration(0, 500_000_000)
    for step in range(20):
        for sim in (g, ref):
            sim.step_async(dt)
        _oracle_step(o, host, step, dt)
    g.sync()
    ref.sync()
    g._dispatch_events()
    before, steps, graphs, added = g.read_state(), g.stats().steps, g.graph_stats(), len(rec.added)
    assert added > 0
    for call in (lambda: g.step(R.Duration(0, 0)), lambda: g.step_async(R.Duration(0, 0))):
        with pytest.raises(R.CrowdsimError) as e:
            call()
        assert e.value.code == N.RCS_ERR_ARG
    after = g.read_state()
    for key in before:
        assert np.array_equal(before[key], after[key]), key
    assert g.stats().steps == steps == 20 and g.graph_stats() == graphs
    g._dispatch_events()
    assert len(rec.added) == added
    # the host generators were called for the refused steps as well: give both handles the same call counts
    for sid, gen in g._host_gen.items():
        ref._host_gen[sid].calls = gen.calls
    g.step(dt)
    ref.step(dt)
    sa, sb = g.read_state(), ref.read_state()
    for key in sa:
        assert np.array_equal(sa[key], sb[key]), key
    assert [a for a, _ in rec.added] == [a for a, _ in rec_ref.added]


def test_bad_rates_are_refused_at_add():
    g = R.Simulation(R.LocationHash2D(64.0, 64.0, 2.0, (0.0, 0.0), capacity=64))
    hl, lp = R.ConstantVelocityPlan((1.0, 0.0)), R.NoLocalPlan()
    for rate in (0.0, -1.0, float("nan"), float("inf"), -float("inf")):
        with pytest.raises(R.CrowdsimError) as e:
            g.add_source_sink(R.SourceSink((10.0, 10.0), 0.6, R.PoissonCrowd(rate), hl, lp, [(50.0, 10.0)], False, 2.0))
        assert e.value.code == N.RCS_ERR_ARG
    with pytest.raises(R.CrowdsimError):
        g.add_source_sink(R.SourceSink((10.0, 10.0), 0.6, object(), hl, lp, [(50.0, 10.0)], False, 2.0))
    assert g.add_source_sink(R.SourceSink((10.0, 10.0), 0.6, R.PoissonCrowd(1.0), hl, lp, [(50.0, 10.0)], False,
                                          2.0)) == 0
    g.step(R.Duration(0, 100_000_000))


def _set_counts(g, ids, counts):
    ids = np.ascontiguousarray(ids, dtype=np.uint64)
    counts = np.ascontiguousarray(counts, dtype=np.uint64)
    return g._lib.rcs_set_spawn_counts(g._h, len(ids), ids.ctypes.data_as(N.c_u64p), counts.ctypes.data_as(N.c_u64p))


def _direct_step(g):
    N.check(g._h, g._lib.rcs_step(g._h, DT.secs, DT.nanos))
    return g.stats().spawned


def test_set_spawn_counts_refusals_write_nothing_and_counts_are_consumed():
    g = _fast_stream([R.MonotonicCrowd(10.0), PatternCrowd([1]), PatternCrowd([1]), (3.0, 9)])
    g.remove_source_sink(2)
    for ids in ([1, 0], [1, 3], [1, 2], [1, 4], [1, 1 << 40]):  # Monotonic, Poisson, removed, unknown
        assert _set_counts(g, ids, [1, 1]) == N.RCS_ERR_ARG
    assert g._lib.rcs_set_spawn_counts(g._h, 1, None, None) == N.RCS_ERR_ARG
    assert g._lib.rcs_set_spawn_counts(g._h, 0, None, None) == N.RCS_OK
    g.remove_source_sink(3)  # leaves the Monotonic source (spawns every step) and host source 1
    assert _direct_step(g) == 1  # no counts: the host source spawns nothing
    assert _set_counts(g, [1, 1], [1, 0]) == N.RCS_OK  # an id listed twice takes its last count
    assert _direct_step(g) == 1
    assert _set_counts(g, [1], [3]) == N.RCS_OK
    assert _direct_step(g) == 2
    assert _direct_step(g) == 1  # consumed


def test_host_generators_are_called_once_per_step_in_ascending_id():
    log = []
    gens = [PatternCrowd([1, 0], log, tag=k) for k in range(4)]
    g = _fast_stream([gens[0], (2.0, 1), gens[1], gens[2], gens[3]])
    rec = Rec()
    g.add_event_listener(rec)
    tag_of = {0: 0, 2: 1, 3: 2, 4: 3}  # source-sink id -> generator
    for k in range(12):
        if k == 5:
            g.remove_source_sink(3)
            del tag_of[3]
        log.clear()
        rec.added.clear()
        g.step(DT)
        assert [t for t, _ in log] == [tag_of[s] for s in sorted(tag_of)], k
        assert all(d == DT for _, d in log)
        host_rows = sorted(r for r in (_row(p) for _, p in rec.added) if r in tag_of)
        assert host_rows == (sorted(tag_of) if k % 2 == 0 else []), k
