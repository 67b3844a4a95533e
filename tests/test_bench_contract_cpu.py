"""bench.py contract pieces that run without a GPU: the reference arm (CPU oracle) alone and under a 2-rank torchrun
launch (rank 0 prints ONE JSON line, the other rank exits 0 without work), and the keys the driver reads."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ["impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"]


def _check_line(out, n_gpus):
    lines = [l for l in out.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1, out
    d = json.loads(lines[0])
    for k in REQUIRED:
        assert k in d, k
    assert d["impl"] == "reference" and d["n_gpus"] == n_gpus and d["unit"] == "registrations/s" and d["value"] > 1
    assert d["metric"].startswith("scan-to-map registrations/sec") and "workload" in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["vs_baseline"] is None and d["higher_is_better"] is True


def test_reference_arm_single_process(oracle_mod, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "1",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    assert len(r.stdout.strip().splitlines()) == 1, r.stdout  # ONE line on stdout: native prints go to stderr
    _check_line(r.stdout, 1)
    # the dumped pose is the registration of the seeded config-1 workload
    import numpy as np
    import ilsm_b200
    c = ilsm_b200.synth.config1(n_map=100_000)
    tree = "nanoflann" if oracle_mod.lib_nanoflann() is not None else "own"
    x, _, _ = oracle_mod.register_aloam(c["map_corner"], c["map_surf"], c["corner"], c["surf"], np.concatenate([c["q0"], c["t0"]]),
                                        tree=tree)
    pose = np.load(tmp_path / "pose.npy")
    assert pose.dtype == np.float64 and np.array_equal(pose, x)


def test_reference_arm_under_torchrun_world2(oracle_mod):
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29611", os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--steps", "3", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    _check_line(r.stdout, 2)
