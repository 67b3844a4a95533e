"""ilsm::IterativeClosestPoint (include/ilsm.hpp): the mirror program compiles and links; without a GPU it stops with
ILSM_ERR_NO_DEVICE, on the GPU its result is byte-identical to ilsm_icp_align_batch on the same pair."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "intensity_based_lidar_slam_for_me-_b200")


def _build(ilsm, tmp_path):
    ilsm.load_library()
    exe = tmp_path / "icp_mirror_test"
    r = subprocess.run(["g++", "-std=c++14", "-O2", "-ffp-contract=off", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "cpp", "icp_mirror_test.cpp"), "-o", str(exe), "-L", PKG, "-lilsm_cuda",
                        "-Wl,-rpath," + PKG], capture_output=True, text=True)
    assert r.returncode == 0 and "warning" not in r.stderr, r.stderr
    return exe


def test_icp_mirror_links(ilsm, tmp_path):
    exe = _build(ilsm, tmp_path)
    import torch
    if not torch.cuda.is_available():
        r = subprocess.run([str(exe)], capture_output=True, text=True)
        assert r.returncode == 100 and "ilsm::Error -3" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
def test_icp_mirror_matches_c_abi(ilsm, tmp_path):
    r = subprocess.run([str(_build(ilsm, tmp_path))], capture_output=True, text=True, timeout=300)
    print(r.stdout, r.stderr)
    assert r.returncode == 0 and "icp mirror checks passed" in r.stdout, r.stdout + r.stderr
