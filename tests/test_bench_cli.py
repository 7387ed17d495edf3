"""CPU: the bench.py contract that can be checked without a GPU -- the reference arm prints one JSON line with the
keys the driver reads, and the product arm refuses to run (no CPU fallback) when there is no CUDA device."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=240):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True,
                          text=True, timeout=timeout)


def _has_cuda_device() -> bool:
    import ctypes as C

    from rmf_crowdsim_b200 import _native as N

    lib = N.load()
    n = C.c_int(0)
    try:
        rt = C.CDLL("libcudart.so")
        return rt.cudaGetDeviceCount(C.byref(n)) == 0 and n.value > 0
    except OSError:
        pass
    # no runtime library to ask: try to create a handle
    from rmf_crowdsim_b200 import LocationHash2D

    try:
        LocationHash2D(8.0, 8.0, 2.0, (0.0, 0.0), capacity=4)
        return True
    except Exception:  # noqa: BLE001
        return False
    finally:
        del lib


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "agent-steps/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("agent-steps/sec") and d["value"] > 0 and d["dtype"] == "f64"
    assert d["steps"] == 1 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_under_a_launcher_only_rank_0_reports():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps",
                        "1", "--warmup", "1"], cwd=ROOT, capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_is_refused_where_it_is_not_implemented(tmp_path):
    for extra in (("--impl", "reference"), ("--workload", "c5"), ("--gpus", "2")):
        r = _run(*extra, "--steps", "1", "--warmup", "1", "--dump-outputs", str(tmp_path / "out"))
        assert r.returncode == 2 and "--dump-outputs" in r.stderr, extra
    assert not (tmp_path / "out").exists()


def test_product_arm_fails_loudly_without_a_cuda_device():
    if _has_cuda_device():
        pytest.skip("a CUDA device is present")
    r = _run("--steps", "1", "--warmup", "1", "--skip-cpu", "--workload", "c2")
    assert r.returncode != 0
    assert "no CPU fallback" in r.stderr
    assert not [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{")]
