"""bench.py --impl reference (the reference's CPU implementation of the path = the oracle port on the host cores) needs no
GPU: its JSON line carries the contract's keys, and under torchrun only rank 0 works."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, *args):
    env = dict(os.environ)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny", *args],
                          capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)


def test_reference_arm_line():
    r = _run(None, "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "pods scheduled/sec" and line["unit"] == "pods/s"
    assert line["value"] > 0 and line["steps"] == 2 and line["higher_is_better"] is True and line["gpu_launches"] == 0
    assert line["config"]["workload"].startswith("tiny")
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "pods/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_dump_outputs(tmp_path):
    """--dump-outputs writes the last timed step's result, one float64 .npy per field: the same arrays a direct call of the
    oracle returns on the same seeded workload."""
    import numpy as np
    from oracle.pyoracle import OracleSession
    from volcano_b200.synth import make_snapshot
    r = _run(None, "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    o = OracleSession(make_snapshot("tiny"))
    dec, vis, fe = o.allocate()
    o.close()
    want = {f"decisions_{f}": dec[f] for f in dec.dtype.names}
    want.update({f"visits_{f}": vis[f] for f in vis.dtype.names})
    want["fit_errors"] = fe
    assert sorted(os.listdir(tmp_path)) == sorted(f"{k}.npy" for k in want)
    for k, a in want.items():
        got = np.load(tmp_path / f"{k}.npy")
        assert got.dtype == np.float64 and np.array_equal(got, a), k
    assert len(dec) > 0


def test_reference_arm_other_ranks_do_nothing():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, "--gpus", "2", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0 and not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
