"""ilsm::Stage (csrc/ilsm_stage.hpp), the host-thread hand-off of the pipelined and three-stage loops, built on its own
with g++ and ThreadSanitizer: results in FIFO order, the in-flight count, shutdown, and errors carried across threads."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "intensity_based_lidar_slam_for_me-_b200", "csrc")


def test_stage_under_thread_sanitizer(tmp_path):
    exe = tmp_path / "stage_test"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-Wall", "-Wextra", "-pthread", "-fsanitize=thread", "-I", CSRC,
                        os.path.join(ROOT, "tests", "cpp", "stage_test.cpp"), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and "warning" not in r.stderr, r.stderr
    env = dict(os.environ, TSAN_OPTIONS="halt_on_error=1 exitcode=66")
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and "ThreadSanitizer" not in r.stderr and "stage checks passed" in r.stdout, r.stdout + r.stderr
