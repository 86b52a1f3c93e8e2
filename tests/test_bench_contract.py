"""bench.py contract pieces that can be checked without a GPU: the reference arm prints exactly one JSON line on stdout with
the keys the driver reads, under a plain launch and as a non-zero rank (which must stay silent and exit 0)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env):
    env = dict(os.environ, **extra_env)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--batch", "2048"],
                       capture_output=True, text=True, env=env, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    return p.stdout


def test_reference_arm_prints_one_json_line():
    out = _run({})
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ECDSA-P256 verifies/sec" and d["unit"] == "verifies/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "verifies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_are_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}).strip() == ""


def test_dump_outputs_writes_float32_and_samples_past_the_cap(tmp_path, monkeypatch):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    bits = np.unpackbits(np.arange(256, dtype=np.uint8))
    bench.dump_outputs(str(tmp_path / "full"), {"valid": bits})
    got = np.load(str(tmp_path / "full" / "valid.npy"))
    assert got.dtype == np.float32 and (got == bits).all()
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 4 * 100)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"valid": np.arange(1000)})
    a, b = (np.load(str(tmp_path / d / "valid.npy")) for d in ("a", "b"))
    assert a.dtype == np.float32 and a.size == 100 and (a == b).all() and (np.diff(a) > 0).all()


def test_alg_mac_model_matches_the_window_shapes():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.alg_macs_cached(22, 16) == (11 * (12 + 16) + 3) * 64
    assert bench.alg_macs_cached(16, 12) == (11 * (16 + 22) + 3) * 64
