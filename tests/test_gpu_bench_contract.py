"""bench.py on the GPU: stdout carries exactly ONE JSON line (the NCCL banner and the reference ikd-Tree's printf, which
the CPU baselines trigger, must not reach it) with the contract's keys."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_bench_prints_one_json_line(tmp_path, oracle_mod):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "20", "--warmup", "3", "--cpu-seconds", "1",
                        "--no-frontend", "--no-sweep", "--no-sequence", "--no-sharded", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.strip().splitlines()
    assert len(lines) == 1, r.stdout[:2000]
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "clocks", "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 20 and d["value"] > 1000 and d["gpu_launches"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] > 100
    assert 0 < d["roofline"]["frac"] < 1 and d["roofline"]["bound"] == "hbm"
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["value"] > 1
    # the dumped pose of the last timed step is the oracle's registration of the same seeded workload
    import numpy as np
    import ilsm_b200
    c = ilsm_b200.synth.config1(n_map=100_000)
    x, _, _ = oracle_mod.register_aloam(c["map_corner"], c["map_surf"], c["corner"], c["surf"], np.concatenate([c["q0"], c["t0"]]))
    pose = np.load(tmp_path / "pose.npy")
    assert pose.dtype == np.float64 and pose.shape == (7,)
    assert np.linalg.norm(pose[4:] - x[4:]) < 1e-4 and ilsm_b200.synth.quat_angle(pose[:4], x[:4]) < 1e-4
