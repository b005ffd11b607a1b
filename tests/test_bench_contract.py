"""bench.py's reference arm (the CPU legs that run without a GPU): one JSON line with the contract's keys; ranks other
than 0 print nothing and exit 0."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.timeout(600)
def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, cwd=ROOT, timeout=580)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[-2000:]
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["unit"] == "rays/s" and j["higher_is_better"] is True
    for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data"):
        assert k in j, k
    assert j["value"] > 0 and j["vs_baseline"] is None and j["data"] == "synthetic"
    assert "workload" in j["config"] and "GF-NeRF global stage" in j["config"]["workload"]
    cb = j["cpu_baseline"]
    # the reference's own kernels where oracle/_ref was built (the build container; it travels to the GPU box), the
    # oracle port otherwise -- and the port beside the reference kernels for continuity
    from oracle import ref_host as rh
    want = "reference" if rh.available("fma") else "port"
    assert cb["kind"] == want, cb
    assert cb["cores"] >= 1 and cb["value"] == j["value"] and "rays/step" in cb["sample"]
    if want == "reference":
        assert "oracle/_ref" in cb["sample"] and cb["port"]["value"] > 0 and "oracle port" in cb["port"]["sample"]
    assert j["e2e"] == {"value": j["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # BASELINE.json configs[0], the reference's own CPU path, beside it
    crp = j["cpu_reference_path"]
    assert crp["value"] > 0 and crp["unit"] == "rays/s" and "configs[0]" in crp["workload"] and crp["cores"] >= 1


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, cwd=ROOT, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_cpu_arm_falls_back_to_the_port_and_says_so(monkeypatch):
    """If the reference's kernels are missing or fail on a box the arm still reports a number: the oracle port, with a
    note -- never an exception that takes the bench line down."""
    sys.path.insert(0, ROOT)
    import bench
    from oracle import ref_host as rh
    monkeypatch.setattr(rh, "available", lambda flavour="off": False)
    monkeypatch.setattr(bench, "time_oracle", lambda *a, **k: (1.0, 2.0, 3, 4.0))
    assert bench.time_cpu_arm(8, 1, 0) == (1.0, 2.0, 3, 4.0, "port",
                                          "oracle/_ref/libgf_ref_host_fma.so is not there (built where /root/reference exists)")
    monkeypatch.setattr(rh, "available", lambda flavour="off": True)

    def boom(*a, **k):
        raise OSError("no such kernel")
    monkeypatch.setattr(bench, "time_reference_native", boom)
    out = bench.time_cpu_arm(8, 1, 0)
    assert out[4] == "port" and "OSError" in out[5]


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    """--dump-outputs: the arrays of the last timed step as float32 / float64 .npy files, 64 MB at most, and the JSON
    line still the only stdout."""
    import numpy as np
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--no-operator-api", "--dump-outputs", str(out)],
                       capture_output=True, text=True, cwd=ROOT, timeout=880)
    assert r.returncode == 0, r.stderr[-2000:]
    assert len([l for l in r.stdout.splitlines() if l.strip()]) == 1 and json.loads(r.stdout)["steps"] == 2
    files = {p.name: np.load(p) for p in out.iterdir()}
    assert {"rgb.npy", "depth.npy", "accumulation.npy", "loss.npy", "mlp_params.npy", "hash_table_sample.npy"} <= set(files)
    assert all(a.dtype in (np.float32, np.float64) for a in files.values())
    assert sum(p.stat().st_size for p in out.iterdir()) <= 64 << 20
    assert files["rgb.npy"].shape == (8192, 3) and np.isfinite(files["rgb.npy"]).all()
    assert np.isfinite(files["loss.npy"]).all() and files["n_samples.npy"][0] > 0
