"""ilsm::LoopClosure (include/ilsm.hpp): the mirror program compiles and links; without a GPU it stops with
ILSM_ERR_NO_DEVICE (exit status -3), on the GPU its results are byte-identical to ilsm_loop_add_keyframe on the same
keyframes and it accepts the revisits of synth.loop_keyframes()."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "intensity_based_lidar_slam_for_me-_b200")


def _build(ilsm, tmp_path):
    ilsm.load_library()
    exe = tmp_path / "loop_mirror_test"
    r = subprocess.run(["g++", "-std=c++14", "-O2", "-ffp-contract=off", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "cpp", "loop_mirror_test.cpp"), "-o", str(exe), "-L", PKG, "-lilsm_cuda",
                        "-Wl,-rpath," + PKG], capture_output=True, text=True)
    assert r.returncode == 0 and "warning" not in r.stderr, r.stderr
    return exe


def test_loop_mirror_links(ilsm, tmp_path):
    exe = _build(ilsm, tmp_path)
    import torch
    if not torch.cuda.is_available():
        r = subprocess.run([str(exe), str(tmp_path / "absent.bin")], capture_output=True, text=True)
        assert r.returncode == (-3) & 0xFF and "ilsm::Error -3" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
def test_loop_mirror_matches_c_abi(ilsm, tmp_path):
    path = tmp_path / "keyframes.bin"
    kfs = ilsm.synth.loop_keyframes()
    with open(path, "wb") as fh:
        fh.write(np.int32(len(kfs)).tobytes())
        for kf in kfs:
            fh.write(np.int32(len(kf["src"])).tobytes() + np.asarray(kf["q"], np.float64).tobytes() +
                     np.asarray(kf["t"], np.float64).tobytes() + np.ascontiguousarray(kf["src"], np.float32).tobytes())
    r = subprocess.run([str(_build(ilsm, tmp_path)), str(path)], capture_output=True, text=True, timeout=300)
    print(r.stdout, r.stderr)
    assert r.returncode == 0 and "loop mirror checks passed" in r.stdout, r.stdout + r.stderr
