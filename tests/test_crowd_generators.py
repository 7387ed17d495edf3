"""CPU: the keyed PoissonCrowd draw (include/rcs.h) -- a plain Philox4x64-10 against numpy's, the oracle's decisions
against that restatement, the spawn frequency against 1 - exp(-lambda), the two lambda edge cases -- and the oracle's
host-count generator and refusals.  No device needed."""
import math
import os
import sys

import numpy as np
import pytest
from scipy import stats

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import oracle_crowd_generators as G  # noqa: E402
import oracle_ffi as O  # noqa: E402

SEEDS = [0, 1, 7, 0x0123456789ABCDEF, (1 << 63) + 5, (1 << 64) - 1]
KS = [0, 1, 2, 99, 12345, (1 << 32) + 3, (1 << 63) - 1, (1 << 64) - 3]
SIDS = [0, 1, 5, 8191, (1 << 32) - 1]


def test_python_philox_equals_numpy():
    for seed in SEEDS:
        for k in KS:
            for sid in SIDS:
                assert G.python_word0(seed, k, sid) == G.numpy_word0(seed, k, sid), (seed, k, sid)


def test_oracle_philox_equals_numpy():
    L = G.lib()
    for seed in SEEDS:
        for k in KS:
            for sid in SIDS:
                assert L.orc_philox4x64_10_w0(k + 1, sid, seed) == G.numpy_word0(seed, k, sid), (seed, k, sid)


def test_oracle_decisions_equal_the_numpy_pin():
    L = G.lib()
    rng = np.random.default_rng(3)
    durations = [(0, 100_000_000), (0, 1_000), (1, 0), (0, 33_333_333), (2, 500_000_000)]
    rates = [1e-3, 0.1, 1.0, 3.7, 10.0, 250.0]
    checked = spawned = 0
    for secs, nanos in durations:
        dt = secs + nanos / 1e9
        for rate in rates:
            for seed in (0, 42, (1 << 64) - 1):
                for k in [0, 1, 17, 1000] + [int(v) for v in rng.integers(0, 1 << 40, 3)]:
                    for sid in (0, 3, 64, 1000):
                        want = G.poisson_wants(rate, seed, dt, k, sid)
                        assert L.orc_poisson_wants(rate, seed, secs, nanos, k, sid) == int(want)
                        checked += 1
                        spawned += int(want)
    assert checked >= 2500 and 0 < spawned < checked


@pytest.mark.parametrize("lam", [0.01, 0.5, 1.0, 3.0])
def test_spawn_frequency_is_one_minus_exp(lam):
    """Deterministic (fixed seeds): the share of (step, source) draws that spawn lies inside the two-sided 1e-6 binomial
    band around P(Poisson(lambda) >= 1) = 1 - exp(-lambda)."""
    n_src, n_steps, seed = 100, 1000, 20240901
    thr = G.threshold(lam)
    hits = 0
    for sid in range(n_src):
        # counters (k + 1, sid) for k = 0 .. n_steps - 1: one Philox stream per source, word 0 of every block
        bg = np.random.Philox(key=np.array([seed, 0], dtype=np.uint64), counter=np.array([0, sid, 0, 0], dtype=np.uint64))
        w0 = bg.random_raw(4 * n_steps)[::4]
        hits += int(np.count_nonzero((w0 >> np.uint64(11)) >= np.uint64(thr)))
    n = n_src * n_steps
    p = 1.0 - math.exp(-lam)
    lo, hi = stats.binom.ppf(0.5e-6, n, p), stats.binom.isf(0.5e-6, n, p)
    assert lo <= hits <= hi, (hits, lo, hi, n * p)


def test_lambda_edge_cases():
    # lambda < 2^-54: exp(-lambda) rounds to 1, the threshold is 2^53 > every u: never
    assert G.threshold(2.0 ** -55) == 1 << 53
    L = G.lib()
    for k in range(200):
        assert not L.orc_poisson_wants(2.0 ** -55, 1, 1, 0, k, 0)
    # lambda > ~745: exp underflows to 0, the threshold is 0: always
    assert G.threshold(746.0) == 0
    for k in range(200):
        assert L.orc_poisson_wants(746.0, 1, 1, 0, k, 0)
    # in between, exp(-lambda) < 1 makes the threshold < 2^53
    assert G.threshold(2.0 ** -52) < 1 << 53


def _oracle():
    o = G.GenOracle(40.0, 40.0, 1.0, (0.0, 0.0))
    hl, lp = o.hl_constant((10.0, 0.0)), o.lp_none()
    return o, hl, lp


def test_oracle_refuses_bad_rates_and_zero_dt():
    o, hl, lp = _oracle()
    for rate in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(O.OracleError):
            o.add_source_sink_gen((5, 5), 0.5, G.POISSON, rate, 0, hl, lp, [(35, 5)], False, 1.0)
    sid = o.add_source_sink_gen((5, 5), 0.5, G.POISSON, 10.0, 0, hl, lp, [(35, 5)], False, 1.0)
    assert sid == 0  # nothing was added by the refused calls
    with pytest.raises(O.OracleError):
        o.step(0, 0)
    assert o.steps() == 0 and o.agent_count() == 0
    o.step(0, 100_000_000)
    assert o.steps() == 1


def test_oracle_host_counts_spawn_where_count_is_at_least_one():
    o, hl, lp = _oracle()
    ids = [o.add_source_sink_gen((2.0, 2.0 + 3 * i), 0.5, G.HOST, 0.0, 0, hl, lp, [(38, 2.0 + 3 * i)], False, 1.0)
           for i in range(4)]
    rng = np.random.default_rng(9)
    expect_total = 0
    for step in range(30):
        counts = rng.integers(0, 3, len(ids))
        if step % 5 != 4:  # some steps get no counts at all: nothing spawns
            o.set_spawn_counts(ids, counts)
        sp, _, _ = o.poll_events()
        o.step(0, 100_000_000)
        sp, xy, _ = o.poll_events()
        want = [i for i, c in zip(ids, counts) if c >= 1] if step % 5 != 4 else []
        got = sorted(int(round((y - 2.0) / 3)) for y in xy[:, 1])
        assert got == want, (step, got, want)
        expect_total += len(want)
    with pytest.raises(O.OracleError):
        o.set_spawn_counts([99], [1])
    assert expect_total > 20
