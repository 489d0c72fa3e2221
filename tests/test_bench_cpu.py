"""bench.py host-side helpers (no GPU): the JSON contract's static parts, the reference arm's bounded sample, the NUMA
policy switch.  The timed legs themselves need a B200 and are exercised by the driver."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("lins_bench", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_thread_sweep_and_config():
    b = _bench()
    assert b.thread_sweep(128) == [32, 64, 128]
    assert b.thread_sweep(1) == [1]
    cfg = b.bench_config(1000, 1)
    assert "workload" in cfg and "config3" in cfg["workload"] and "model" not in cfg


def test_host_memory_policy_is_harmless():
    b = _bench()
    on = b.host_memory_policy(True)
    off = b.host_memory_policy(False)
    assert isinstance(on, str) and isinstance(off, str)  # one node / refused / interleaved: never raises


def test_dump_outputs_writes_float64_within_the_cap(tmp_path):
    b = _bench()
    defs = importlib.import_module("lins---lidar-inertial-slam_b200.ctypes_defs")
    n = 500
    res = np.zeros(n, dtype=defs.SCAN_RESULT_DTYPE)
    res["scan_id"] = np.arange(n); res["iters"] = 7; res["flags"] = 1; res["pose"] = np.arange(7 * n).reshape(n, 7)
    states, covs = np.random.default_rng(1).standard_normal((n, defs.STATE_DIM)), np.ones((n, defs.COV_SIZE))
    full = b.dump_outputs(str(tmp_path / "full"), states, covs, res)
    assert full == ["cov", "flags", "iters", "pose", "scan_id", "state"]
    got = {k: np.load(tmp_path / "full" / f"{k}.npy") for k in full}
    assert all(a.dtype == np.float64 and len(a) == n for a in got.values())
    assert np.array_equal(got["state"], states) and np.array_equal(got["pose"], res["pose"])
    cap = 300_000  # < n rows: a seeded sample of the units, the same one every time
    for d in ("s1", "s2"):
        b.dump_outputs(str(tmp_path / d), states, covs, res, max_bytes=cap)
    assert sum(os.path.getsize(p) for p in (tmp_path / "s1").iterdir()) <= cap
    ids = np.load(tmp_path / "s1" / "scan_id.npy")
    assert 0 < len(ids) < n and np.all(np.diff(ids) > 0)
    assert np.array_equal(ids, np.load(tmp_path / "s2" / "scan_id.npy"))
    assert np.array_equal(np.load(tmp_path / "s1" / "state.npy"), states[ids.astype(int)])


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ESKF iterations/sec" and d["value"] > 0
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
