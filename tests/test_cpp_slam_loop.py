"""ilsm::StagedLoamPipeline with loop closure (include/ilsm.hpp): the mirror program compiles and links; without a GPU it
stops with ILSM_ERR_NO_DEVICE (exit status -3); on the GPU its loop events over the closed-loop sequence are byte-identical
to those of a raw ilsm_slam_create_staged handle on the same frames, and it accepts a revisit."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "intensity_based_lidar_slam_for_me-_b200")


def _build(ilsm, tmp_path):
    ilsm.load_library()
    exe = tmp_path / "slam_loop_mirror_test"
    r = subprocess.run(["g++", "-std=c++14", "-O2", "-ffp-contract=off", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "cpp", "slam_loop_mirror_test.cpp"), "-o", str(exe), "-L", PKG, "-lilsm_cuda",
                        "-Wl,-rpath," + PKG], capture_output=True, text=True)
    assert r.returncode == 0 and "warning" not in r.stderr, r.stderr
    return exe


def test_slam_loop_mirror_links(ilsm, tmp_path):
    exe = _build(ilsm, tmp_path)
    import torch
    if not torch.cuda.is_available():
        r = subprocess.run([str(exe), str(tmp_path / "absent.bin")], capture_output=True, text=True)
        assert r.returncode == (-3) & 0xFF and "ilsm::Error -3" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
def test_slam_loop_mirror_matches_c_abi(ilsm, tmp_path):
    import torch
    S = ilsm.synth
    poses = S.closed_loop_poses()[:300]  # the first lap and half of the second
    clouds = S.make_frames_torch(S.Scene(), poses, 0x5EED3000, torch.device("cuda:0"))
    path = tmp_path / "frames.bin"
    with open(path, "wb") as fh:
        fh.write(np.int32(len(poses)).tobytes() + np.int32(clouds.shape[1]).tobytes())
        fh.write(clouds.numpy().tobytes())
    r = subprocess.run([str(_build(ilsm, tmp_path)), str(path)], capture_output=True, text=True, timeout=600)
    print(r.stdout, r.stderr)
    assert r.returncode == 0 and "slam loop mirror checks passed" in r.stdout, r.stdout + r.stderr
