"""Loop closure of the full loop (ilsm_slam_enable_loop / ilsm_slam_loop_results) without a GPU: struct layouts against gcc,
the defaults, argument errors before any CUDA call, ILSM_ERR_NO_DEVICE, the keyframe rule's Python restatement against
the library's own rule (csrc/ilsm_keyframe.hpp) at, just below and just above both thresholds, and Stage::ready()."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "intensity_based_lidar_slam_for_me-_b200", "csrc")
INVALID_ARG, NO_DEVICE = -1, -3


def test_abi_struct_layouts_match_gcc(ilsm, tmp_path):
    from ilsm_b200 import binding as b
    fields = {"ilsm_slam_loop_opts": [f[0] for f in b.SlamLoopOpts._fields_],
              "ilsm_slam_loop_event": [f[0] for f in b.SlamLoopEvent._fields_]}
    body = "".join(f'printf("%zu\\n", sizeof({s}));' + "".join(f'printf("%zu\\n", offsetof({s}, {f}));' for f in fs)
                   for s, fs in fields.items())
    src = tmp_path / "s.c"
    src.write_text(f'#include <stddef.h>\n#include <stdio.h>\n#include "ilsm.h"\nint main(void){{{body} return 0;}}\n')
    exe = tmp_path / "s"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = list(map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()))
    want = []
    for cls, fs in ((b.SlamLoopOpts, fields["ilsm_slam_loop_opts"]), (b.SlamLoopEvent, fields["ilsm_slam_loop_event"])):
        want += [C.sizeof(cls)] + [getattr(cls, f).offset for f in fs]
    assert got == want
    assert (C.sizeof(b.SlamLoopOpts), C.sizeof(b.SlamLoopEvent)) == (112, 264)


def test_defaults(ilsm):
    o = ilsm.SlamLoopOpts()
    assert (o.keyframe_dist, o.keyframe_angle_rad, o.max_pending) == (1.0, 0.2, 8)
    assert bytes(o.loop) == bytes(ilsm.LoopOpts())
    o = ilsm.SlamLoopOpts(max_pending=2, loop=dict(exclude_recent=20, icp=dict(max_iterations=7)))
    assert (o.max_pending, o.loop.exclude_recent, o.loop.icp.max_iterations, o.loop.tree_period) == (2, 20, 7, 50)


def test_argument_errors_come_before_any_cuda_call(ilsm):
    from ilsm_b200 import binding as b
    lib = b.load_library()
    fake = C.cast(C.create_string_buffer(64), C.c_void_p)  # a handle that is never dereferenced on these paths
    assert lib.ilsm_slam_enable_loop(None, None) == INVALID_ARG and b"null handle" in lib.ilsm_last_error()
    nan, inf = float("nan"), float("inf")
    for bad in (dict(keyframe_dist=-0.1), dict(keyframe_dist=nan), dict(keyframe_dist=inf), dict(keyframe_angle_rad=-1e-9),
                dict(keyframe_angle_rad=nan), dict(keyframe_angle_rad=inf), dict(max_pending=0), dict(max_pending=-3)):
        assert lib.ilsm_slam_enable_loop(fake, C.byref(b.SlamLoopOpts(**bad))) == INVALID_ARG, bad
        assert b"slam_enable_loop" in lib.ilsm_last_error()
    for bad in (dict(exclude_recent=0), dict(tree_period=0), dict(num_candidates=17), dict(submap_half=8), dict(leaf=0.0),
                dict(cell=inf), dict(sc_dist_threshold=nan), dict(fitness_threshold=nan), dict(icp=dict(max_iterations=-1))):
        assert lib.ilsm_slam_enable_loop(fake, C.byref(b.SlamLoopOpts(loop=bad))) == INVALID_ARG, bad
    ev, n = (b.SlamLoopEvent * 4)(), C.c_int32(7)
    assert lib.ilsm_slam_loop_results(None, 0, ev, 4, C.byref(n)) == INVALID_ARG
    assert lib.ilsm_slam_loop_results(fake, 0, ev, 4, None) == INVALID_ARG
    assert lib.ilsm_slam_loop_results(fake, 0, None, 4, C.byref(n)) == INVALID_ARG
    assert lib.ilsm_slam_loop_results(fake, 1, ev, -1, C.byref(n)) == INVALID_ARG and b"capacity" in lib.ilsm_last_error()
    lib.ilsm_slam_loop_opts_default(None)


def test_enable_without_a_device_returns_no_device(ilsm):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from ilsm_b200 import binding as b
    lib = b.load_library()
    fake = C.cast(C.create_string_buffer(64), C.c_void_p)
    assert lib.ilsm_slam_enable_loop(fake, None) == NO_DEVICE
    assert lib.ilsm_slam_enable_loop(fake, C.byref(b.SlamLoopOpts(keyframe_dist=0.0, keyframe_angle_rad=0.0))) == NO_DEVICE


def _rz(a):
    return np.array([0.0, 0.0, math.sin(a / 2), math.cos(a / 2)])


def _rule_cases(S):
    """(q_kf, t_kf, q, t, dist, angle) at, just below and just above both thresholds, and with both thresholds 0."""
    rng = np.random.default_rng(11)
    cases = []
    for _ in range(40):
        qk = S.quat_from_rotvec(rng.normal(0, 0.5, 3))
        tk = rng.normal(0, 20, 3)
        step = rng.normal(0, 1, 3)
        dq = S.quat_from_rotvec(rng.normal(0, 0.2, 3))
        q, t = S.quat_mul(qk, dq), tk + step
        dx = [float(t[i]) - float(tk[i]) for i in range(3)]
        d = math.sqrt(dx[0] * dx[0] + dx[1] * dx[1] + dx[2] * dx[2])
        # the angle the rule computes: find it as the smallest threshold that does not select by rotation
        lo, hi = 0.0, 4.0
        for _ in range(200):  # bisection on the restatement: the exact double where the decision flips
            mid = 0.5 * (lo + hi)
            if S.keyframe_due(qk, tk, q, t, math.inf, mid):
                lo = mid
            else:
                hi = mid
        a = lo
        for dist in (d, math.nextafter(d, 0.0), math.nextafter(d, math.inf)):
            cases.append((qk, tk, q, t, dist, math.inf))
        for ang in (a, math.nextafter(a, 0.0), math.nextafter(a, math.inf)):
            cases.append((qk, tk, q, t, math.inf, ang))
        cases.append((qk, tk, q, t, 0.0, 0.0))
        cases.append((qk, tk, qk, tk, 0.0, 0.0))  # the same pose again
    # hand-made: 1 m straight ahead and a 0.2 rad turn about z
    z = np.zeros(3)
    one = 1.0
    cases += [(_rz(0.0), z, _rz(0.0), np.array([one, 0, 0]), 1.0, 0.2), (_rz(0.0), z, _rz(0.0), np.array([math.nextafter(one, 0), 0, 0]), 1.0, 0.2),
              (_rz(0.0), z, _rz(0.3), z, 1.0, 0.2), (_rz(0.0), z, _rz(0.1), z, 1.0, 0.2), (_rz(0.0), z, -_rz(0.1), z, 1.0, 0.2)]
    return cases


def test_keyframe_rule_restatement_matches_the_library_rule(ilsm, tmp_path):
    S = ilsm.synth
    exe = tmp_path / "keyframe_rule_test"
    r = subprocess.run(["g++", "-std=c++17", "-O3", "-ffp-contract=off", "-Wall", "-Wextra", "-I", CSRC,
                        os.path.join(ROOT, "tests", "cpp", "keyframe_rule_test.cpp"),
                        "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and "warning" not in r.stderr, r.stderr
    cases = _rule_cases(S)
    lines = [" ".join(float(v).hex() for v in [*qk, *tk, *q, *t, dist, ang]) for qk, tk, q, t, dist, ang in cases]
    out = subprocess.run([str(exe)], input="\n".join(lines) + "\n", capture_output=True, text=True, check=True).stdout.split()
    want = [S.keyframe_due(*c) for c in cases]
    assert [o == "1" for o in out] == want
    # at a threshold: selected; just below it (of the computed value): selected; just above: not -- for both thresholds
    for i in range(40):
        block = want[8 * i: 8 * i + 8]
        assert block[:6] == [True, True, False, True, True, False], i
        assert block[6:] == [True, True], i  # thresholds 0 select every pose, even the same one again
    assert want[-5:] == [True, False, True, False, False]


def test_select_keyframes_on_a_hand_made_sequence(ilsm):
    S = ilsm.synth
    z = np.zeros(3)
    poses = [(_rz(0.0), z), (_rz(0.0), np.array([0.5, 0, 0])), (_rz(0.0), np.array([1.0, 0, 0])), (_rz(0.0), np.array([1.9, 0, 0])),
             (_rz(0.15), np.array([1.9, 0, 0])), (_rz(0.25), np.array([1.9, 0, 0])), (_rz(0.25), np.array([1.9, 0, 0]))]
    assert S.select_keyframes(poses, 1.0, 0.2) == [0, 2, 5]
    assert S.select_keyframes(poses, 0.0, 0.0) == list(range(7))
    assert S.select_keyframes(poses, 100.0, 100.0) == [0]
    assert S.select_keyframes([], 1.0, 0.2) == []


def test_closed_loop_sequence(ilsm):
    S = ilsm.synth
    poses = S.closed_loop_poses()
    n = len(poses) // 2
    steps = [np.linalg.norm(poses[k + 1][1] - poses[k][1]) for k in range(len(poses) - 1)]
    turns = [S.quat_angle(poses[k + 1][0], poses[k][0]) for k in range(len(poses) - 1)]
    assert 0.24 < min(steps) and max(steps) < 0.26 and np.rad2deg(max(turns)) < 2.0
    # the second lap passes ~0.1 m outside the first, heading turned by 3 degrees
    for k in range(0, n, 17):
        assert abs(np.linalg.norm(poses[n + k][1] - poses[k][1]) - 0.1) < 1e-9
        assert abs(np.rad2deg(S.quat_angle(poses[n + k][0], poses[k][0])) - 3.0) < 1e-6


def test_stage_ready_under_thread_sanitizer(tmp_path):
    exe = tmp_path / "stage_ready_test"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-Wall", "-Wextra", "-pthread", "-fsanitize=thread", "-I", CSRC,
                        os.path.join(ROOT, "tests", "cpp", "stage_ready_test.cpp"), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and "warning" not in r.stderr, r.stderr
    env = dict(os.environ, TSAN_OPTIONS="halt_on_error=1 exitcode=66")
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and "ThreadSanitizer" not in r.stderr and "stage ready checks passed" in r.stdout, r.stdout + r.stderr
