"""GPU: `bench.py --dump-outputs` writes the state the timed steps computed.  The frozen-snapshot run (shuffled ids) must
hold one step from the scene, the committed run (lane-ordered ids) the warm-up plus the timed steps from the scene --
both checked against the oracle, within the tolerances of tests/parity.py."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import parity as P
from rmf_crowdsim_b200 import scenes as SC

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("variant", ["shuffled", "lane"])
def test_dump_outputs_hold_the_timed_steps_result(variant, tmp_path):
    steps, warmup = 4, 3  # bench.py runs at least 3 warm-up steps
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c2", "--variant", variant,
                        "--steps", str(steps), "--warmup", str(warmup), "--skip-e2e", "--skip-cpu", "--skip-secondary",
                        "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == steps
    got = {k: np.load(os.path.join(tmp_path, f"{k}.npy")) for k in ("id", "x", "y", "vx", "vy")}
    assert all(a.dtype == np.float64 for a in got.values())

    scene = SC.config_c2(variant)
    o = P.build_oracle(scene)
    for _ in range(1 if variant == "shuffled" else warmup + steps):
        o.step(*scene.dt)
    want = o.read_state()
    assert np.array_equal(got["id"], want["id"].astype(np.float64))
    vmag = np.hypot(want["vx"], want["vy"])
    for k in ("vx", "vy"):
        assert P.rel_err(got[k], want[k], scale=vmag) <= P.REL_TOL, k
    for k in ("x", "y"):
        assert P.rel_err(got[k], want[k]) <= P.REL_TOL, k
    assert not np.array_equal(got["x"], scene.xy[:, 0])  # the dump is a step's result, not the input
