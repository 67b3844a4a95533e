"""Host paths of the C ABI: the stand-alone evaluation at a host pose equals the one at the same pose on the device, the
launches each entry point makes per call, and the stride rule every entry point applies."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

INVALID_ARG = -1


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def launches(ilsm, fn):
    before = ilsm.launch_count()
    fn()
    return ilsm.launch_count() - before


@pytest.fixture(scope="module")
def maps(ctx, cfg_small):
    c = cfg_small
    return ctx.new_map().set_input_cloud(c["map_corner"]), ctx.new_map().set_input_cloud(c["map_surf"])


@pytest.mark.parametrize("tiles", [1, 0], ids=["small", "bulk"])
@pytest.mark.parametrize("h", [0.0, 0.1])
def test_eval_normal_eq_host_pose_equals_device_pose(ctx, cfg_small, maps, tiles, h):
    """Both regimes of the evaluation: the small kernel, and the bulk kernel at >= 148 x 352 factors."""
    import torch
    c = cfg_small
    mc, ms = maps
    k = tiles or 1 + (148 * 352) // (len(c["corner"]) + len(c["surf"]))
    corner, surf = np.tile(c["corner"], (k, 1)), np.tile(c["surf"], (k, 1))
    assert (tiles == 0) == (len(corner) + len(surf) >= 148 * 352)
    ctx.associate(mc, ms, corner, surf, c["q0"], c["t0"])
    cost, H, g = ctx.eval_normal_eq(c["q0"], c["t0"], h)
    pose = torch.from_numpy(np.concatenate([c["q0"], c["t0"]]).astype(np.float64)).cuda()
    out = torch.zeros(32, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.eval_normal_eq_dev(pose.data_ptr(), out.data_ptr(), h)
    ctx.sync()
    o = out.cpu().numpy()
    iu = np.triu_indices(6)
    assert cost == o[0]
    assert np.array_equal(H[iu], o[1:22]) and np.array_equal(H, H.T)
    assert np.array_equal(g, o[22:28])


def test_launches_per_call(ilsm, ctx, cfg_small, maps):
    """A pose from the host goes up with a copy, not a kernel: associate, odometry, eval_normal_eq and solve make one
    launch fewer than a 1-thread pose kernel would cost; every other entry point keeps its count."""
    import torch
    c = cfg_small
    mc, ms = maps
    corner, surf = c["corner"], c["surf"]
    # association + factor export
    assert launches(ilsm, lambda: ctx.associate(mc, ms, corner, surf, c["q0"], c["t0"])) == 2
    assert launches(ilsm, lambda: ctx.eval_normal_eq(c["q0"], c["t0"], 0.1)) == 1
    assert launches(ilsm, lambda: ctx.solve(c["q0"], c["t0"])) == 1
    pose = torch.from_numpy(np.concatenate([c["q0"], c["t0"]]).astype(np.float64)).cuda()
    out = torch.zeros(32, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    assert launches(ilsm, lambda: ctx.eval_normal_eq_dev(pose.data_ptr(), out.data_ptr())) == 1
    assert launches(ilsm, lambda: (ctx.solve_dev(pose.data_ptr()), ctx.sync())) == 2  # pose seed + solve
    assert launches(ilsm, lambda: (ctx.solve_dev(0), ctx.sync())) == 1
    # 2 passes x (association + solve)
    assert launches(ilsm, lambda: ctx.register(mc, ms, corner, surf, c["q0"], c["t0"])) == 4
    # odometry: 2 passes x (association + solve); with factors, one association and the export
    assert launches(ilsm, lambda: ctx.odometry(mc, ms, corner, surf, c["q0"], c["t0"])) == 4
    assert launches(ilsm, lambda: ctx.odometry(mc, ms, corner, surf, c["q0"], c["t0"], factors_only=True)) == 2
    # point-to-point factors + solve
    assert launches(ilsm, lambda: ctx.align_points(surf[:200, :3], surf[:200, :3])) == 2
    # VoxelGrid: one block; the tiled path at 20000 points (pack/bbox, init, keys, 2 tile sorts, 1 global stage, head
    # count, scan, centroids)
    assert launches(ilsm, lambda: ctx.voxelgrid(surf, 0.4)) == 1
    big = np.tile(surf, (20000 // len(surf) + 1, 1))[:20000]
    assert launches(ilsm, lambda: ctx.voxelgrid(big, 0.4)) == 9
    # frame registration: 10 front-end kernels, the less-sharp gather, one VoxelGrid launch for both stacks, 2 x 2
    assert launches(ilsm, lambda: ctx.register_frame(mc, ms, c["cloud"], c["q0"], c["t0"])) == 16


@pytest.mark.parametrize("stride", [8, 14, 16])
def test_stride_rule(ilsm, ctx, stride):
    """Every entry point rejects a stride below 12 bytes or off a 4-byte boundary with ILSM_ERR_INVALID_ARG; 16 passes
    the check."""
    lib = ilsm.load_library()
    m = ctx.new_map()
    pts = np.zeros(64, np.float32)
    pts[:12] = np.arange(12, dtype=np.float32)
    q, t = np.array([0.0, 0, 0, 1]), np.zeros(3)
    q2, t2 = q.copy(), t.copy()
    n_out = C.c_int(0)
    out = np.zeros((64, 4), np.float32)
    idx, d2 = np.zeros(64, np.int32), np.zeros(64, np.float32)
    ge, mo, cm = ilsm.GroundExtractor(ctx), ilsm.MapOptimization(ctx), ilsm.CubeMap(ctx, 0.4, 0.8)
    calls = {
        "voxelgrid": lambda: lib.ilsm_voxelgrid(ctx._h, _ptr(pts), 2, stride, 0.4, _ptr(out), C.byref(n_out)),
        "align_points": lambda: lib.ilsm_align_points(ctx._h, _ptr(pts), _ptr(pts), 2, stride, _ptr(q2), _ptr(t2), 2, 0.1, None),
        "map_build": lambda: lib.ilsm_map_build(m._h, _ptr(pts), 2, stride, 0.0),
        "map_insert": lambda: lib.ilsm_map_insert(m._h, _ptr(pts), 2, stride, 0, 0.0),
        "knn": lambda: lib.ilsm_knn(m._h, _ptr(pts), 2, stride, 1, 0.0, _ptr(idx), _ptr(d2)),
        "ground_extract": lambda: lib.ilsm_ground_extract(ge._h, _ptr(pts), 2, stride, None, _ptr(out), 64, C.byref(n_out),
                                                          None, None),
        "cubemap_insert_world": lambda: lib.ilsm_cubemap_insert_world(cm._h, _ptr(pts), 2, _ptr(pts), 2, stride, _ptr(t)),
        "mapopt_frame(frame)": lambda: lib.ilsm_mapopt_frame(mo._h, _ptr(pts), 2, stride, _ptr(pts), 2, 16, _ptr(q), _ptr(t),
                                                             _ptr(q2), _ptr(t2), None, None),
        "mapopt_frame(plane)": lambda: lib.ilsm_mapopt_frame(mo._h, _ptr(pts), 2, 16, _ptr(pts), 2, stride, _ptr(q), _ptr(t),
                                                             _ptr(q2), _ptr(t2), None, None),
    }
    # entry points whose work on two points is well defined; the others run at stride 16 throughout the suite
    at16 = ("voxelgrid", "align_points", "map_build", "map_insert", "knn")
    try:
        for name, call in calls.items():
            if stride == 16:
                if name in at16:
                    assert call() == 0, (name, lib.ilsm_last_error())
            else:
                rc = call()
                assert rc == INVALID_ARG, (name, rc)
                assert b"stride" in lib.ilsm_last_error(), (name, lib.ilsm_last_error())
    finally:
        ctx.sync()
        ge.close(), mo.close(), cm.close(), m.close()
