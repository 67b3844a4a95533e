"""K7 loop closure per keyframe (ilsm_loop) without a GPU: struct layouts against gcc, the defaults, argument errors before
any CUDA call, ILSM_ERR_NO_DEVICE from ilsm_loop_create, and the yaw convention of the ICP guess on the CPU oracle."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID_ARG, NO_DEVICE = -1, -3


def test_abi_struct_layouts_match_gcc(ilsm, tmp_path):
    from ilsm_b200 import binding as b
    fields = {"ilsm_loop_opts": [f[0] for f in b.LoopOpts._fields_], "ilsm_loop_result": [f[0] for f in b.LoopResult._fields_]}
    body = "".join(f'printf("%zu\\n", sizeof({s}));' + "".join(f'printf("%zu\\n", offsetof({s}, {f}));' for f in fs)
                   for s, fs in fields.items())
    src = tmp_path / "s.c"
    src.write_text(f'#include <stddef.h>\n#include <stdio.h>\n#include "ilsm.h"\nint main(void){{{body} return 0;}}\n')
    exe = tmp_path / "s"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = list(map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()))
    want = []
    for cls, fs in ((b.LoopOpts, fields["ilsm_loop_opts"]), (b.LoopResult, fields["ilsm_loop_result"])):
        want += [C.sizeof(cls)] + [getattr(cls, f).offset for f in fs]
    assert got == want
    assert (C.sizeof(b.LoopOpts), C.sizeof(b.LoopResult)) == (88, 200)


def test_defaults(ilsm):
    o = ilsm.LoopOpts()
    assert (o.exclude_recent, o.tree_period, o.num_candidates, o.submap_half) == (50, 50, 10, 2)
    assert (o.sc_dist_threshold, o.fitness_threshold) == (0.13, 0.3)
    assert (o.leaf, o.cell) == (np.float32(0.4), 1.0)
    assert (o.icp.max_correspondence_distance, o.icp.max_iterations, o.icp.transformation_epsilon,
            o.icp.euclidean_fitness_epsilon) == (2.0, 50, 1e-8, 1e-6)
    assert o.icp.transformation_rotation_epsilon == 0 and o.icp.fitness_max_range == np.finfo(np.float64).max
    assert ilsm.LoopOpts(submap_half=3, icp=dict(max_iterations=7)).icp.max_iterations == 7


def test_bad_options_and_null_handles_are_rejected_before_any_cuda_call(ilsm):
    from ilsm_b200 import binding as b
    lib = b.load_library()
    fake = C.create_string_buffer(64)  # a context that is never dereferenced on these paths
    h = C.c_void_p()
    assert lib.ilsm_loop_create(None, None, C.byref(h)) == INVALID_ARG
    assert lib.ilsm_loop_create(C.cast(fake, C.c_void_p), None, None) == INVALID_ARG
    for bad in (dict(exclude_recent=0), dict(tree_period=0), dict(num_candidates=0), dict(num_candidates=17), dict(submap_half=-1),
                dict(submap_half=8), dict(leaf=0.0), dict(cell=-1.0), dict(leaf=float("inf")), dict(sc_dist_threshold=float("nan")),
                dict(fitness_threshold=float("nan")), dict(icp=dict(max_iterations=-1))):
        assert lib.ilsm_loop_create(C.cast(fake, C.c_void_p), C.byref(b.LoopOpts(**bad)), C.byref(h)) == INVALID_ARG, bad
        assert b"loop_create" in lib.ilsm_last_error()
    # the keyframe entry points: every check comes before the handle is used
    pts = np.zeros((8, 4), np.float32)
    q, t = np.array([0.0, 0.0, 0.0, 1.0]), np.zeros(3)
    r = b.LoopResult()
    loop = C.cast(fake, C.c_void_p)
    for fn in (lib.ilsm_loop_add_keyframe, lib.ilsm_loop_add_keyframe_dev):
        call = lambda lp=loop, p=pts.ctypes.data, n=8, s=16, qq=q, tt=t, res=C.byref(r): fn(lp, p, n, s, qq.ctypes.data, tt.ctypes.data, res)
        assert call(lp=None) == INVALID_ARG
        assert call(p=None) == INVALID_ARG and b"null argument" in lib.ilsm_last_error()
        assert call(res=None) == INVALID_ARG
        assert call(n=-1) == INVALID_ARG and call(s=12) == INVALID_ARG and call(s=18) == INVALID_ARG
        assert call(n=1 << 24) == INVALID_ARG
        for badq in ([0, 0, 0, 1.00001], [0, 0, 0, 0.9999], [0, 0, 0, np.nan], [0.6, 0, 0, 0.6]):
            assert call(qq=np.array(badq, np.float64)) == INVALID_ARG and b"not unit" in lib.ilsm_last_error()
        assert call(tt=np.array([0, np.inf, 0.0])) == INVALID_ARG
    assert lib.ilsm_loop_size(None) == 0
    lib.ilsm_loop_destroy(None)


def test_create_without_a_device_returns_no_device(ilsm):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from ilsm_b200 import binding as b
    lib = b.load_library()
    fake = C.create_string_buffer(64)
    h = C.c_void_p()
    assert lib.ilsm_loop_create(C.cast(fake, C.c_void_p), None, C.byref(h)) == NO_DEVICE
    assert h.value is None


def test_yaw_convention_on_the_oracle(ilsm, oracle_mod):
    """Keyframe 4 re-observed 0.1 m away with its yaw turned: the aligning shift s of distanceBtnScanContext(revisit,
    keyframe) gives the revisit's heading as q_4 * Rz(-deg2rad(6 s)); Rz(+deg2rad(6 s)) is off by twice the turn."""
    S = ilsm.synth
    kfs = S.loop_keyframes(laps=1)
    base = oracle_mod.sc_make(kfs[4]["src"])
    for yaw, shift, wrong in ((30.0, 55, 60.0), (-30.0, 5, 60.0), (90.0, 45, 180.0)):
        rv = S.revisit_keyframe(kfs[4], yaw)
        d, s = oracle_mod.sc_distance(oracle_mod.sc_make(rv["src"]), base)
        assert s == shift and d < 0.13
        yd = float(np.float32(s * 6.0 * math.pi / 180.0))
        err = [math.degrees(S.quat_angle(S.quat_mul(kfs[4]["q"], [0, 0, math.sin(sg * yd / 2), math.cos(sg * yd / 2)]), rv["q"]))
               for sg in (-1.0, 1.0)]
        assert err[0] < 1e-3 and abs(err[1] - wrong) < 1e-3, (yaw, err)  # the float yaw is within 1e-5 degrees
